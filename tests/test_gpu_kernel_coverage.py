"""Every compiled instantiation of the env-step kernels, and every launch regime, against the C oracle.

`launch_cfg` and `launch_step` (marllb_b200/csrc/mlb_api.cu) pick among 40 `event_kernel<POLICY, R, RNG>`, 8
`feature_kernel<R, SMALL>` and 8 `pair_kernel<R, CLS>` instantiations, and run the pair kernels side by side (small
launches) or one after the other (more than 8192 (env, agent) pairs).  `launched()` restates those rules in Python and
the CPU test below checks that the case list reaches every instantiation and regime, naming any that it does not.  The
GPU tests step each case and replay it on oracle/flow_oracle.c:

  every step: n_flow_on exact, observations within OBS_RTOL / OBS_ATOL, rewards within REWARD_RTOL, done exact;
  at the end: reservoir slot values / timestamps / counts, Algorithm R draw cursors, drop counters and arrival cursors
  bit-exact, and no sticky error.

The near-cutoff test builds arrivals whose decay-weighted p90 lands exactly on a cumulative weight, which sends the
decision to the float64 tier (`weighted_index_exact`, and the `n_old = 255` hand-off from `pair_kernel`), and proves
from the oracle's own reservoirs that it got there.  With decay 0.9 those ties are decided by the last bit of the
float64 weights: it failed while tier 3 used CUDA's pow, which can be 2 ulp off the host's.
"""
import collections
import zlib

import numpy as np
import pytest

import flow_oracle as fo
from conftest import OBS_ATOL, OBS_RTOL, REWARD_RTOL

DT = 0.25
SEED_BASE = 5
POLICIES = ("sed", "lsq", "alias", "sed2", "lsq2")
RNGS = ("replay", "philox")
WP_MARGIN = 5e-5            # MLB_WP_MARGIN, mlb_features.cuh: relative distance below which float32 is not trusted

Case = collections.namedtuple("Case", "id E A Sa K policy rng fc path steps action metric field Q")


def case(E, A, Sa, K, policy, rng, fc=1, path="step", steps=60, action="i32", metric="jain", field=10, Q=160):
    parts = [f"E{E}", f"A{A}", f"Sa{Sa}", f"K{K}", policy, rng]
    parts += [f"fc{fc}"] if fc != 1 else []
    parts += [path] if path != "step" else []
    parts += [action] if action != "i32" else []
    parts += [metric] if metric != "jain" else []
    parts += [f"field{field}"] if field != 10 else []
    parts += [f"Q{Q}"] if Q != 160 else []
    return Case("-".join(parts), E, A, Sa, K, policy, rng, fc, path, steps, action, metric, field, Q)


# ---------------------------------------------------------------- selection rules (marllb_b200/csrc/mlb_api.cu)
def lanes_r(Sa):                       # lanes_r, mlb_api.cu:308
    return 1 if Sa <= 32 else 2 if Sa <= 64 else 4 if Sa <= 128 else 8


def envs_per_block(A):                 # feature kernel epb, launch_cfg, mlb_api.cu:360
    return 4 if A == 1 else 2 if A == 2 else 1


def pair_launches(c):
    """(env, agent) pairs of every launch_step call one step of `c` makes: mlb_step runs host-buffer steps of
    >= 8 * 1024 envs in 8 chunks rounded to whole feature blocks (mlb_api.cu:942-956), anything else in one launch."""
    out = []
    if "step" in c.path.split("+"):
        out.append(c.E * c.A)
    if "host" in c.path.split("+"):
        if c.E >= 8 * 1024:
            epb = envs_per_block(c.A)
            per = ((c.E + 7) // 8 + epb - 1) // epb * epb
            out += [(min(e0 + per, c.E) - e0) * c.A for e0 in range(0, c.E, per)]
        else:
            out.append(c.E * c.A)
    return out


def launched(c):
    """The kernel instantiations and regimes one case runs."""
    R = lanes_r(c.Sa)
    small = 32 * c.A * envs_per_block(c.A) <= 128                  # ft_threads <= 128, mlb_api.cu:361,368
    KP = (c.K + 31) & ~31                                          # mlb_api.cu:535
    use_pair = KP == 128 and c.fc == 1                             # mlb_api.cu:371
    got = {("event", c.policy, R, c.rng), ("feature", R, small), ("feature_cache", c.fc, small)}
    if use_pair:
        for pairs in pair_launches(c):
            wpe = 4 if pairs <= 8192 else 1                        # launch_step, mlb_api.cu:903-906
            got.add(("pair", R, wpe))
            if c.K < 128:
                got.add(("pair K<128", wpe))
    return got


REQUIRED = ({("event", p, R, g) for p in POLICIES for R in (1, 2, 4, 8) for g in RNGS}
            | {("feature", R, s) for R in (1, 2, 4, 8) for s in (True, False)}
            | {("pair", R, w) for R in (1, 2, 4, 8) for w in (4, 1)}
            | {("pair K<128", w) for w in (4, 1)}
            | {("feature_cache", f, s) for f in (0, 1, 2) for s in (True, False)})


# ---------------------------------------------------------------- the cases
# Small launches (host-loaded arrivals, every env replayed).  Sa covers every lane boundary; each R = lanes_r(Sa)
# takes all 5 policies x 2 RNG modes.
SMALL_CASES = [
    # R = 1 (Sa <= 32); the other R = 1 combinations are the reward-metric cases below
    case(3, 32, 1, 128, "sed", "replay", steps=40),                     # 32 warps of one lane each, not SMALL
    case(4, 3, 31, 31, "sed", "philox"),
    case(4, 1, 32, 1, "lsq", "replay", action="u8"),
    case(4, 1, 1, 32, "alias", "replay"),
    # R = 2 (33..64 servers)
    case(4, 4, 33, 33, "sed", "replay"),
    case(2, 5, 63, 96, "sed", "philox"),                                # first not-SMALL agent count
    case(4, 2, 64, 97, "lsq", "replay"),                                # pair kernels with K < 128 reservoirs
    case(2, 17, 33, 128, "lsq", "philox", steps=120),
    case(4, 1, 63, 112, "alias", "replay", fc=0),
    case(4, 3, 64, 128, "alias", "philox", action="f32"),               # continuous weights, A > 1
    case(4, 1, 33, 127, "sed2", "replay", action="u8"),
    case(4, 2, 63, 128, "sed2", "philox", fc=2),
    case(2, 7, 64, 112, "lsq2", "replay", fc=0),
    case(2, 8, 33, 128, "lsq2", "philox", fc=2),
    # R = 4 (65..128 servers)
    case(4, 1, 65, 128, "sed", "replay", field=4, steps=120),
    case(4, 2, 127, 112, "sed", "philox", steps=120),
    case(2, 3, 128, 97, "lsq", "replay"),
    case(2, 5, 65, 127, "lsq", "philox", steps=120),
    case(4, 1, 127, 128, "alias", "replay"),
    case(2, 4, 128, 33, "alias", "philox"),
    case(4, 2, 65, 128, "sed2", "replay", action="u8", field=0),
    case(4, 1, 127, 96, "sed2", "philox"),
    case(4, 2, 128, 128, "lsq2", "replay", action="f32"),
    case(2, 3, 65, 128, "lsq2", "philox", field=8),
    # R = 8 (129..256 servers)
    case(2, 32, 256, 128, "sed", "philox", steps=100),                  # the largest config: 224 KB feature block
    case(4, 1, 129, 128, "sed", "replay", steps=120),
    case(2, 2, 255, 112, "lsq", "replay", steps=120),
    case(2, 5, 129, 97, "lsq", "philox"),
    case(4, 1, 256, 128, "alias", "replay", Q=8),                       # drops on the widest event kernel
    case(2, 3, 129, 128, "alias", "philox"),
    case(4, 1, 255, 33, "sed2", "replay", field=2),
    case(2, 2, 256, 128, "sed2", "philox", action="u8"),
    case(2, 4, 129, 127, "lsq2", "replay"),
    case(4, 1, 255, 31, "lsq2", "philox", Q=3),
]
# Every reward metric with A > 1 and S = 35 (not a multiple of 32), spread over the R = 1 policy / RNG pairs.
SMALL_CASES += [case(2, 5, 7, 128, POLICIES[i % 5], RNGS[(i // 5) % 2], metric=m, steps=100)
                for i, m in enumerate(fo.METRICS)]

# Large launches (device-generated arrivals, sampled envs replayed): more than 8192 (env, agent) pairs, so the pair
# kernels run one after the other.  "step+host": the device step first, then 8-chunk host-buffer steps on the same
# episode, whose chunks are small enough to run the pair kernels side by side.
LARGE_CASES = [
    case(8192, 2, 48, 128, "sed2", "replay", path="step+host", action="u8"),
    case(8300, 1, 100, 112, "alias", "replay", path="step+host"),
    case(1700, 5, 200, 97, "lsq", "philox", steps=100),
    case(1200, 7, 20, 128, "sed", "replay", steps=80, action="u8"),
]

CUTOFF_CASES = [case(4, 1, 16, 128, "alias", "replay", fc=fc, steps=14) for fc in (1, 2, 0)]

ALL_CASES = SMALL_CASES + LARGE_CASES + CUTOFF_CASES


def _entry(e):
    kind, *rest = e
    names = {"event": "event_kernel<{}, R={}, {}>", "feature": "feature_kernel<R={}, SMALL={}>",
             "pair": "pair_kernel<R={}, .> wpe={}", "pair K<128": "pair kernels with K < 128, wpe={}",
             "feature_cache": "feature_cache={} with SMALL={}"}
    return names[kind].format(*rest)


def test_case_list_reaches_every_instantiation():
    """CPU: the case list below launches every event / feature / pair kernel instantiation, both pair regimes (also
    with K < 128) and every feature_cache mode on both feature kernel sizes."""
    got = set().union(*(launched(c) for c in ALL_CASES))
    assert len(REQUIRED) == 40 + 8 + 8 + 2 + 6
    assert got <= REQUIRED, sorted(map(_entry, got - REQUIRED))
    missing = sorted(map(_entry, REQUIRED - got))
    assert not missing, "not launched by any case: " + "; ".join(missing)


# ---------------------------------------------------------------- shared helpers
def _speeds(S):
    return np.where(np.arange(S) % 2 == 0, 1.0, 2.0).astype(np.float32)


def _rate(Sa):
    return max(4.0, 2.0 * Sa)                     # flows per second per agent: ~Sa / 2 per step


def _mean_work(Sa, speeds_agent, rate, rho=0.9):
    return rho * float(speeds_agent.sum()) / rate


def _synth(rng, c):
    """Host arrivals of every (env, agent): Poisson times, exponential work at load 0.9, pre-drawn buckets / u."""
    speeds = _speeds(c.A * c.Sa)
    rate, horizon = _rate(c.Sa), c.steps * DT + 0.5
    out = []
    for _ in range(c.E):
        per_env = []
        for a in range(c.A):
            n = int(rate * horizon * 1.3) + 10
            t = np.cumsum(rng.exponential(1.0 / rate, n))
            t = t[t < horizon].astype(np.float32)
            mw = _mean_work(c.Sa, speeds[a * c.Sa:(a + 1) * c.Sa], rate)
            per_env.append({"time": t, "work": rng.exponential(mw, len(t)).astype(np.float32),
                            "bucket": rng.randint(0, c.Sa, len(t)).astype(np.int32),
                            "u": rng.random_sample(len(t)).astype(np.float32)})
        out.append(per_env)
    return out


def _make_env(c):
    from marllb_b200 import VecLoadBalanceEnv
    env = VecLoadBalanceEnv(c.E, num_servers=c.Sa, num_agents=c.A, policy=c.policy, reservoir_capacity=c.K,
                            queue_capacity=c.Q, max_steps=c.steps, feature_cache=c.fc, rng_mode=c.rng,
                            seed_base=SEED_BASE, reward_metric=c.metric, reward_field=c.field,
                            action_type="continuous" if c.action == "f32" else "discrete",
                            action_dtype="uint8" if c.action == "u8" else "int32")
    env.set_speeds(_speeds(c.A * c.Sa))
    return env


def _oracle(c, streams, env_id, speeds=None):
    return fo.FlowEnv(c.A, c.Sa, _speeds(c.A * c.Sa) if speeds is None else speeds, streams, reservoir_k=c.K,
                      queue_cap=c.Q, policy=c.policy, action_type="continuous" if c.action == "f32" else "discrete",
                      reward_metric=c.metric, reward_field=c.field, max_steps=c.steps, seed_base=SEED_BASE,
                      rng_mode=c.rng, env_id=env_id)


def _oracle_actions(c, act):
    return np.ascontiguousarray(act, np.float32 if c.action == "f32" else np.int32)


def _reward_rtol(c):
    # the default field (obs column 10, a decay-weighted p90: one stored sample) and n_flow_on are bit-equal, so the
    # float64 reward is computed from identical inputs; the other fields carry the float32 tolerance of the features
    return REWARD_RTOL if c.field in (0, 10) else 10 * OBS_RTOL


def _compare_step(c, k, obs, rew, done, o_ref, r_ref, d_ref):
    tag = f"{c.id} step {k}"
    assert np.array_equal(obs[..., 0], o_ref[..., 0]), f"{tag}: n_flow_on"
    np.testing.assert_allclose(obs, o_ref, rtol=OBS_RTOL, atol=OBS_ATOL, err_msg=f"{tag}: observations")
    np.testing.assert_allclose(rew, r_ref, rtol=_reward_rtol(c), atol=1e-12, err_msg=f"{tag}: rewards")
    assert np.array_equal(done.astype(bool), d_ref.astype(bool)), f"{tag}: done"


def _draw_cursor(word, K, n):
    """Words Algorithm R consumed in a reservoir that has seen n samples: numpy's legacy randint(0, c + 1) -- masked
    rejection over 32-bit words -- for every c in [K, n) (reservoir.py:76; res_draw_slot in mlb_step_kernel.cuh)."""
    cur = 0
    for cnt in range(K, n):
        mask = (1 << cnt.bit_length()) - 1
        while word(cur) & mask > cnt:
            cur += 1
        cur += 1
    return cur


class _MTWords:
    """Raw MT19937 words of RandomState(seed), the stream every reservoir of one server replays."""

    def __init__(self, seed):
        self.seed, self.words = seed, fo.mt_fill(seed, 1024)

    def __call__(self, i):
        if i >= len(self.words):
            self.words = fo.mt_fill(self.seed, 2 * i)
        return int(self.words[i])


def _check_final_state(c, env, ora, ids, streams, total_steps):
    env.check_status()
    get = {f: env.get_state(f, ids) for f in ("res_values", "res_ts", "res_count", "res_cursor", "dropped",
                                              "n_flow_on", "arr_cursor")}
    t_end = np.float32(total_steps) * np.float32(DT)
    mt = {}
    for i, e in enumerate(ids):
        d = ora[i].dump()
        tag = f"{c.id} env {e}"
        assert np.array_equal(get["res_values"][i], d["res_values"]), f"{tag}: reservoir slot values"
        assert np.array_equal(get["res_ts"][i], d["res_ts"]), f"{tag}: reservoir slot timestamps"
        cnt = get["res_count"][i].T.astype(np.int64)                  # (S, 2)
        assert np.array_equal(cnt, d["res_count"]), f"{tag}: reservoir counts"
        assert np.array_equal(get["dropped"][i].astype(np.int64), d["dropped"]), f"{tag}: drops"
        assert np.array_equal(get["n_flow_on"][i], d["n_flow_on"]), f"{tag}: n_flow_on"
        # arrivals consumed: every flow with time < t1 of the last step (mlb_step_kernel.cuh, flow_oracle.c:619)
        want = [int(np.searchsorted(streams[i][a]["time"], t_end, side="left")) for a in range(c.A)]
        assert get["arr_cursor"][i].tolist() == want, f"{tag}: arrival cursors"
        # draw cursors of a spread of servers (and the fullest one): both metrics of server j draw from its stream
        S = c.A * c.Sa
        cur = get["res_cursor"][i].T.astype(np.int64)                 # (S, 2)
        js = set(np.linspace(0, S - 1, min(S, 24)).astype(int).tolist()) | {int(cnt.max(axis=1).argmax())}
        for j in sorted(js):
            if c.rng == "replay":
                word = mt.setdefault(j, _MTWords(SEED_BASE + j))
            else:
                word = lambda w, j=j, e=e: fo.philox_word(w, j, e, SEED_BASE)   # noqa: E731
            for m in range(2):
                assert cur[j, m] == _draw_cursor(word, c.K, int(cnt[j, m])), f"{tag}: draw cursor of ({j}, {m})"
    return get


# ---------------------------------------------------------------- small launches
@pytest.mark.gpu
@pytest.mark.parametrize("c", SMALL_CASES, ids=lambda c: c.id)
def test_small_launch_matches_oracle(c):
    rng = np.random.RandomState(zlib.crc32(c.id.encode()))
    streams = _synth(rng, c)
    env = _make_env(c)
    env.load_arrivals([s for per_env in streams for s in per_env])
    env.reset()
    ora = [_oracle(c, streams[e], e) for e in range(c.E)]
    S = c.A * c.Sa
    for k in range(c.steps):
        if c.action == "f32":
            act = (rng.random_sample((c.E, S)) * 3.0 - 0.5).astype(np.float32)     # clipped at min_weight 0.1
        else:
            act = rng.randint(0, 3, (c.E, S)).astype(np.uint8 if c.action == "u8" else np.int32)
        obs, rew, done = env.step(act)
        o_ref, r_ref, d_ref, _ = fo.step_batch(ora, _oracle_actions(c, act))
        _compare_step(c, k, obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy(), o_ref, r_ref, d_ref)
    get = _check_final_state(c, env, ora, list(range(c.E)), streams, c.steps)
    assert int(get["res_count"].max()) > c.K, "the episode must reach Algorithm R's replacement regime"
    if c.Q < 160:
        assert int(get["dropped"].sum()) > 0, "a small queue must drop flows"
    env.close()


# ---------------------------------------------------------------- large launches
def _sample_envs(c):
    """First and last env and both sides of every host-pipeline chunk boundary (or of the middle)."""
    E = c.E
    cand = {0, 1, E // 2 - 1, E // 2, E - 2, E - 1}
    if "host" in c.path and E >= 8 * 1024:
        epb = envs_per_block(c.A)
        per = ((E + 7) // 8 + epb - 1) // epb * epb
        for b in range(per, E, per):
            cand |= {b - 1, b}
    return sorted(cand)


@pytest.mark.gpu
@pytest.mark.parametrize("c", LARGE_CASES, ids=lambda c: c.id)
def test_large_launch_matches_oracle(c):
    import torch
    env = _make_env(c)
    S = c.A * c.Sa
    speeds = _speeds(S)
    rate = _rate(c.Sa)
    env.gen_poisson(rate, _mean_work(c.Sa, speeds[:c.Sa], rate), c.steps * DT + 0.5, seed=77)
    env.reset()
    ids = _sample_envs(c)
    idx = torch.as_tensor(ids, device="cuda")
    streams = [[env.get_arrivals(e, a) for a in range(c.A)] for e in ids]
    ora = [_oracle(c, streams[i], e) for i, e in enumerate(ids)]
    n_dev = c.steps if c.path == "step" else c.steps // 2
    gen = torch.Generator(device="cuda").manual_seed(31)
    adt = torch.uint8 if c.action == "u8" else torch.int32
    for k in range(c.steps):
        act = torch.randint(0, 3, (c.E, S), generator=gen, device="cuda", dtype=adt)
        if k < n_dev:
            obs, rew, done = env.step(act)
            o, r, d = (x.index_select(0, idx).cpu().numpy() for x in (obs, rew, done))
        else:
            o_h, r_h, d_h = env.step_host(act.cpu().numpy())
            o, r, d = o_h[ids].copy(), r_h[ids].copy(), d_h[ids].copy()
        o_ref, r_ref, d_ref, _ = fo.step_batch(ora, _oracle_actions(c, act.index_select(0, idx).cpu().numpy()))
        _compare_step(c, k, o, r, d, o_ref, r_ref, d_ref)
    get = _check_final_state(c, env, ora, ids, streams, c.steps)
    assert int(get["res_count"].max()) > c.K, "the episode must reach Algorithm R's replacement regime"
    env.close()
    del env
    torch.cuda.empty_cache()


# ---------------------------------------------------------------- the float64 tier of the weighted percentile
def _cutoff_streams(c):
    """Arrivals that put the 0.9 * W cutoff of the decay-weighted p90 exactly on a cumulative weight.

    Speeds are 1, every time is a multiple of 1/1024 s (exact in float32), the alias policy with u = 0 sends each flow
    to its bucket, and every server j runs one cycle starting at step s:
      * step s: a leader flow (finishing at F = t1_s + delta) and 10m - 1 zero-work flows queued behind it, so all
        10m finish at F;  the flow-duration reservoir takes 10m samples at t1_s;
      * step s + 1: the 10m flows retire together: the FCT reservoir takes 10m samples of equal weight (a resort);
        until s + 4 (flow durations) and s + 5 (FCTs) nothing is added, and the reference re-decides these ties
        every step with weights decay^(now - t) whose last bits change;
      * step s + 4: m flows arrive (a leader finishing at F + 1 and m - 1 zero-work ones), each with a larger duration
        than any earlier sample: the flow-duration reservoir takes m samples with weight 1 against 10m of weight
        0.9^1, so W = 10m and the m new ones weigh exactly 0.1 W (an incremental update of 1-3 slots);
      * step s + 5: they retire at F + 1 with larger FCTs than the first 10m: the same tie in the FCT reservoir.
    m and delta vary over servers, so float32 and float64 rounding disagree on some of these ties."""
    out = []
    for e in range(c.E):
        t, w, b = [], [], []
        for j in range(c.Sa):
            g = e * c.Sa + j
            m = 1 + g % 3
            ts = (1 + g % 6) * DT                              # t1 of step s
            F = ts + (20 + (g * 37) % 180) / 1024.0
            a0 = ts - 200 / 1024.0
            t += [a0 + i / 1024.0 for i in range(10 * m)]
            w += [F - a0] + [0.0] * (10 * m - 1)
            ap = ts + 0.75 + 1 / 1024.0
            t += [ap + i / 1024.0 for i in range(m)]
            w += [F + 1.0 - ap] + [0.0] * (m - 1)
            b += [j] * (11 * m)
        order = np.argsort(np.asarray(t), kind="stable")
        out.append([{"time": np.asarray(t, np.float32)[order], "work": np.asarray(w, np.float32)[order],
                     "bucket": np.asarray(b, np.int32)[order], "u": np.zeros(len(t), np.float32)}])
    return out


def _cutoff_distance(d, K, now, decay=0.9):
    """Per reservoir (S, 2): min_k |cumsum_k - 0.9 W| / W over the cumulative decay weights in value order, in
    float64 (reservoir.py:181-196); inf for an empty reservoir."""
    vals, ts = d["res_values"].astype(np.float64), d["res_ts"].astype(np.float64)
    n = np.minimum(d["res_count"], K)
    valid = np.arange(K) < n[..., None]
    order = np.lexsort((np.broadcast_to(np.arange(K), vals.shape), np.where(valid, vals, np.inf)), axis=-1)
    wgt = np.where(valid, decay ** (now - ts), 0.0)
    cum = np.cumsum(np.take_along_axis(wgt, order, axis=-1), axis=-1)
    W = cum[..., -1:]
    with np.errstate(invalid="ignore", divide="ignore"):
        dist = np.where(valid, np.abs(cum - 0.9 * W), np.inf).min(axis=-1) / W[..., 0]
    return np.where(n > 0, dist, np.inf)


@pytest.mark.gpu
@pytest.mark.parametrize("c", CUTOFF_CASES, ids=lambda c: c.id)
def test_near_cutoff_weighted_percentile_matches_oracle(c):
    """feature_cache = 1: the pair kernels meet the ties on 1-3-slot updates and hand them to feature_kernel's float64
    tier; the 10m-sample updates are re-sorted and take feature_kernel's own fallback.  feature_cache = 2 re-sorts
    every touched reservoir, feature_cache = 0 every reservoir.  In all three the reference re-decides untouched ties
    every step from rescaled weights, so the decision hangs on their last bits (tier 3 must round them as the host's
    pow does), and with feature_cache 1 / 2 the kernel must re-evaluate a reservoir left on a tie."""
    streams = _cutoff_streams(c)
    env, host = _make_env(c), _make_env(c)          # host: the same episode through step_host(obs="changed")
    for x in (env, host):
        x.set_speeds(np.ones(c.Sa, np.float32))
        x.load_arrivals([s for per_env in streams for s in per_env])
        x.reset()
    ones = np.ones(c.Sa, np.float32)
    ora = [_oracle(c, streams[e], e, speeds=ones) for e in range(c.E)]
    rng = np.random.RandomState(8)
    prev = np.zeros((c.E, c.Sa, 2), np.int64)
    hits = {"incremental": 0, "resort": 0, "untouched": 0}
    for k in range(c.steps):
        act = rng.randint(0, 3, (c.E, c.Sa)).astype(np.int32)
        obs, rew, done = env.step(act)
        o_host, _, _ = host.step_host(act, obs="changed")
        assert np.array_equal(o_host, obs.cpu().numpy()), f"{c.id} step {k}: step_host(obs='changed')"
        o_ref, r_ref, d_ref, _ = fo.step_batch(ora, act)
        now = float(np.float32(k + 1) * np.float32(DT))
        for e in range(c.E):
            d = ora[e].dump()
            near = _cutoff_distance(d, c.K, now) < WP_MARGIN
            cnt, old = d["res_count"], prev[e]
            # below K every add fills a new slot, so the count delta is the number of written slots
            assert int(cnt.max()) <= c.K, "the precondition counts written slots as count deltas: stay below K"
            touched = cnt > old
            if c.fc == 1:
                inc = touched & (old > 0) & (cnt - old <= 3)      # pair_kernel's share: 1-3 written slots, n_old > 0
                hits["incremental"] += int((near & inc).sum())
                hits["resort"] += int((near & touched & ~inc).sum())
            else:
                hits["resort"] += int((near & (touched if c.fc == 2 else True)).sum())
            hits["untouched"] += int((near & ~touched).sum())
            prev[e] = cnt
        _compare_step(c, k, obs.cpu().numpy(), rew.cpu().numpy(), done.cpu().numpy(), o_ref, r_ref, d_ref)
    assert hits["resort"] > 0, "no re-sorted reservoir came within MLB_WP_MARGIN of the cutoff"
    assert hits["untouched"] > 0, "no reservoir was left on a tie without new samples"
    if c.fc == 1:
        assert hits["incremental"] > 0, "no incrementally updated reservoir came within MLB_WP_MARGIN of the cutoff"
    _check_final_state(c, env, ora, list(range(c.E)), streams, c.steps)
    env.close()
    host.close()
