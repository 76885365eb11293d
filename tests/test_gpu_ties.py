"""GPU: reservoirs full of EQUAL values (regression for the tie handling of the incremental rank updates).

Durations are float32 differences of float32 timestamps, i.e. quantised, so equal values inside one reservoir are not
exotic: late in an episode (time ~ 500 s, ulp 3e-5 s) a 128-slot reservoir holds a tied pair with probability ~0.4 and
triple ties do occur at bench scale (131072 envs x thousands of steps).  The cached ranks may hold tied values in any
order (the bitonic re-sort does not order ties); an incremental update that assumed "ties are ranked by slot index"
produced duplicate ranks -- and with them garbage decay-weighted features until the next re-sort -- when a third equal
value met a tied pair in the other order.  tools/determinism_probe.py found it as a run-to-run difference at the bench
size (7 envs of 131072 within 2148 steps).  Here arrival times and work sit on a 1/32 s grid, so EVERY duration is a
multiple of 1/32 s and every reservoir is mostly ties; the observations must equal the C oracle's (which sorts from
scratch every step, like the reference: reservoir.py:105-196) over a long episode, through every statistics path:
the pair kernels at K = 128, the pair kernels at K = 112 (a 128-slot stride with full reservoirs below 128 slots, whose
replacements take the general incremental update) and full re-sorts (feature_cache=False).
"""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import flow_oracle as fo  # noqa: E402

pytestmark = pytest.mark.gpu
OBS_RTOL, OBS_ATOL = 1e-5, 1e-6


def _grid_streams(rng, E, Sa, rate, horizon):
    """Arrival times on a 1/32 s grid (non-decreasing), work in {1/32 .. 6/32}: every duration is a multiple of 1/32."""
    out = []
    for _ in range(E):
        n = int(rate * horizon)
        t = np.sort(rng.randint(0, int(horizon * 32), n)).astype(np.float32) / 32.0
        w = rng.randint(1, 7, n).astype(np.float32) / 32.0
        out.append([{"time": t, "work": w, "bucket": rng.randint(0, Sa, n).astype(np.int32),
                     "u": rng.random_sample(n).astype(np.float32)}])
    return out


@pytest.mark.parametrize("mode", ["pair", "pair_k112", "resort"])
def test_tied_values_through_every_statistics_path(mode):
    from marllb_b200 import VecLoadBalanceEnv
    E, Sa, steps, rate, K = 6, 8, 900, 48.0, 112 if mode == "pair_k112" else 128
    rng = np.random.RandomState(4242)
    speeds = np.where(np.arange(Sa) % 2 == 0, 1.0, 2.0).astype(np.float32)
    streams = _grid_streams(rng, E, Sa, rate, steps * 0.25 + 0.5)
    env = VecLoadBalanceEnv(E, num_servers=Sa, reservoir_capacity=K, max_steps=steps, feature_cache=(mode != "resort"))
    env.set_speeds(speeds)
    env.load_arrivals([s for es in streams for s in es])
    env.reset()
    ora = [fo.FlowEnv(1, Sa, speeds, streams[e], reservoir_k=K, policy="sed", max_steps=steps) for e in range(E)]
    worst = 0.0
    for k in range(steps):
        act = rng.randint(0, 3, (E, Sa)).astype(np.int32)
        obs, rew, _ = env.step(act)
        obs, rew = obs.cpu().numpy(), rew.cpu().numpy()
        o_ref, r_ref, _, _ = fo.step_batch(ora, act)
        assert np.array_equal(obs[..., 0], o_ref[..., 0]), k
        err = np.abs(obs - o_ref) / (OBS_ATOL + OBS_RTOL * np.abs(o_ref))
        worst = max(worst, float(err.max()))
        assert err.max() <= 1.0, (mode, k, np.argwhere(err > 1.0)[:4].tolist(), float(err.max()))
        np.testing.assert_allclose(rew, r_ref, rtol=1e-9, atol=1e-12)
    env.check_status()
    vals = env.get_state("res_values")
    # the point of the test: the reservoirs really are full of ties
    full = vals[0, 0, 0, :K]
    assert len(np.unique(full)) < K // 2
    for e in range(E):
        assert np.array_equal(vals[e], ora[e].dump()["res_values"])
    env.close()


def test_two_runs_of_the_same_episode_are_bit_identical():
    """No cross-env communication, fixed random streams: two runs must agree bit for bit (observations and reservoirs).
    A difference means a race or a read of memory nothing wrote -- which is how the tie bug above first showed."""
    import torch
    from marllb_b200 import VecLoadBalanceEnv
    E, S, steps = 8192, 16, 400
    outs = []
    for _ in range(2):
        env = VecLoadBalanceEnv(E, num_servers=S, max_steps=steps + 1)
        env.set_speeds(np.where(np.arange(S) % 2 == 0, 1.0, 2.0).astype(np.float32))
        env.gen_poisson(64.0, 0.8 * 1.5 * S / 64.0, steps * 0.25 + 1.0, seed=77)
        env.reset()
        g = torch.Generator(device="cuda").manual_seed(5)
        acc = torch.zeros((E,), dtype=torch.float64, device="cuda")
        for k in range(steps):
            obs, rew, _ = env.step(torch.randint(0, 3, (E, S), device="cuda", dtype=torch.uint8, generator=g))
            acc += obs.view(E, -1).sum(1, dtype=torch.float64) * (1 + k % 7) + rew
        outs.append((acc.cpu().numpy(), obs.cpu().numpy().copy(), env.get_state("res_values", envs=[0, 1, E - 1])))
        env.check_status()
        env.close()
    assert np.array_equal(outs[0][0], outs[1][0])
    assert np.array_equal(outs[0][1], outs[1][1]) and np.array_equal(outs[0][2], outs[1][2])
