"""Quick device-side timing of the env step at the bench's c5 slice, without per-kernel profiling events:
    python tools/quick_ms.py [--envs N] [--burnin B] [--steps K]
MARLLB_B200_LIB=marllb_b200/_variants/NAME.so times a variant built by tools/build_variant.sh.  Prints ms per step."""
import argparse
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from marllb_b200 import VecLoadBalanceEnv  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--servers", type=int, default=64)
    ap.add_argument("--burnin", type=int, default=256)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--graph", action="store_true", help="replay the step from a CUDA graph")
    a = ap.parse_args()
    E, S = a.envs, a.servers
    total = a.burnin + a.steps + 16
    env = VecLoadBalanceEnv(E, num_servers=S, max_steps=total + 1)
    env.set_speeds(np.where(np.arange(S) % 2 == 0, 1.0, 2.0).astype(np.float32))
    rate = 128.0 * S / 64          # bench c5: 128 flows/s/agent at 64 servers, rho = 0.8
    env.gen_poisson(rate, 0.8 * 1.5 * S / rate, total * 0.25 + 1.0, seed=1234)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(0)
    acts = [torch.randint(0, 3, (E, S), device="cuda", dtype=torch.uint8, generator=g) for _ in range(8)]
    for k in range(a.burnin):
        env.step(acts[k % 8])
    if a.graph:
        env.capture()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(a.steps):
        if a.graph:
            env.graph_action.copy_(acts[k % 8])
            env.step_graph()
        else:
            env.step(acts[k % 8])
    e1.record()
    torch.cuda.synchronize()
    env.check_status()
    tag = os.environ.get("MARLLB_B200_LIB", "in-tree library")
    print(f"[{tag}] {e0.elapsed_time(e1) / a.steps:.3f} ms per step, checksum {float(env.obs.sum(dtype=torch.float64)):.6e}")


if __name__ == "__main__":
    main()
