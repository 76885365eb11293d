"""GPU: the offline training driver (SURVEY 8f f1) end to end on a tiny budget -- trace files are
parsed and replayed, episodes are stored, the agent updates, checkpoints and training_stats.json
appear with the reference's keys (training_pipeline.py:263-292)."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _write_trace(path, rate, horizon, seed):
    rng = np.random.RandomState(seed)
    t = np.cumsum(rng.exponential(1.0 / rate, int(rate * horizon)))
    with open(path, "w") as f:
        f.write("time\tquery\n")
        for x in t[t < horizon]:
            f.write(f"{x:.6f}\t/dummy.php/?n={int(rng.exponential(60000)) + 1}\n")      # data/trace/poisson_for_loop format


@pytest.mark.parametrize("agent", ["qmix", "sac-gru"])
def test_training_pipeline_runs_and_writes_reference_artifacts(tmp_path, agent):
    from marllb_b200.training_pipeline import TrainingPipeline
    tdir = tmp_path / "trace" / "poisson_for_loop"
    tdir.mkdir(parents=True)
    _write_trace(tdir / "rate_100.csv", 100.0, 50.0, 1)
    _write_trace(tdir / "rate_200.csv", 200.0, 50.0, 2)
    ck = tmp_path / "ck"
    cfg = {"batch_size": 8 if agent == "qmix" else 64, "seed": 3}
    pipe = TrainingPipeline(agent, num_servers=8, num_agents=2, trace_dir=str(tmp_path / "trace"),
                            checkpoint_dir=str(ck), config=cfg, num_envs=8, verbose=False)
    assert len(pipe.traces) == 2 and len(pipe.traces[0]["time"]) > 1000
    out = pipe.train(num_episodes=16, save_interval=8, eval_interval=8)
    assert out["total_episodes"] == 16
    stats = json.load(open(ck / "training_stats.json"))
    assert set(stats) == {"episode_rewards", "episode_lengths", "losses", "best_reward", "total_episodes", "total_time"}
    assert len(stats["episode_rewards"]) == 16 and all(np.isfinite(stats["episode_rewards"]))
    assert len(stats["losses"]) >= 1 and all(np.isfinite(stats["losses"]))
    assert os.path.exists(ck / f"{agent}_best.pth") and os.path.exists(ck / f"{agent}_ep16.pth")
    # Jain rewards in (0, 1] per step, 200 steps (x A agents for QMIX like sum(rewards))
    per_step = np.array(stats["episode_rewards"]) / (200 * (2 if agent == "qmix" else 1))
    assert (per_step > 0).all() and (per_step <= 1.0 + 1e-9).all()


def test_sac_training_beats_the_random_policy(tmp_path):
    """Evidence that the driver trains (VERDICT r1 missing #5; the reference claims a rising reward curve,
    problem-04-sac-gru/README.md:461-464).  8 servers, four fast (speed 2) and four slow (speed 1): weights
    proportional to speed even out the flow durations (Jain 0.92), equal weights give 0.86, the random policy --
    SAC's raw action range, uniform per step -- 0.82.  After 6 rounds x 100 updates (a few seconds) the greedy policy
    must be clearly above both the random policy and its own untrained self.  Everything is seeded; the kernels are
    deterministic."""
    import random
    import torch
    from marllb_b200.training_pipeline import MAX_EPISODE_STEPS, TrainingPipeline
    speeds = [2.0, 2.0, 2.0, 2.0, 1.0, 1.0, 1.0, 1.0]
    cfg = dict(server_speeds=speeds, rates=[24.0], seed=1, updates_per_round=100, batch_size=256)
    torch.manual_seed(0); np.random.seed(0); random.seed(0)
    tp = TrainingPipeline('sac-gru', num_servers=8, num_agents=1, trace_dir=str(tmp_path / 'no_traces'), checkpoint_dir=str(tmp_path),
                          config=cfg, num_envs=16, verbose=False)
    E = tp.num_envs

    def random_policy():
        tp._load_round()
        g = torch.Generator(device="cuda"); g.manual_seed(0)
        tot = 0.0
        for _ in range(MAX_EPISODE_STEPS):
            _, r, _ = tp.env.step(torch.rand((E, 8), generator=g, device="cuda") * 2 - 1)   # clipped to [0.1, 10] by the env
            tot += float(r.mean())
        return tot / MAX_EPISODE_STEPS

    greedy = lambda: float(tp._run_round(0, explore=False, learn=False)[0].mean()) / MAX_EPISODE_STEPS
    rnd = float(np.mean([random_policy() for _ in range(2)]))
    before = greedy()
    evals = []
    for r in range(6):
        rets, loss = tp._run_round(r * E)
        assert loss is not None and np.isfinite(loss)
        evals.append(greedy())
    after = float(np.mean(evals[-3:]))
    assert 0.7 < rnd < 0.9, rnd
    assert after > rnd + 0.03, (rnd, before, evals)
    assert after > before + 0.05, (rnd, before, evals)
