"""Ring-fed updates/s of the tensor-core mode at more than 32 actions, beside the 6-action walker shape: walker (A = 6,
F = 50), DMC dog (A = 38, F = 50) and CMU humanoid (A = 56, F = 100), all at B = 256, H = 1024.  One agent and one
GPU-resident replay ring per shape; the shapes are timed in alternation (block 1 of every shape, then block 2, ...) so
that a drift of the shared machine touches all three alike.  Per shape: updates/s as the median and range of the
blocks, and the policy head's GPU time inside the captured update (CUDA event-record nodes around its launch, median
of 20 replays).  The card's name and power limit are printed with the numbers.

    python tools/bench_action_dims.py [--steps-per-block 200] [--blocks 5]
"""
import argparse
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402

SHAPES = (("walker", 6, 50), ("dog", 38, 50), ("cmu_humanoid", 56, 100))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (s.strip() for s in q.stdout.strip().split(",")) if q.returncode == 0 else (torch.cuda.get_device_name(), "unknown")
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--hidden-dim", type=int, default=1024)
    ap.add_argument("--episodes", type=int, default=64)
    ap.add_argument("--steps-per-block", type=int, default=200)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_action_dims.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, power = card()
    B = args.batch
    cfg = SimpleNamespace(hidden_dim=args.hidden_dim, mode="bf16")
    runs = []
    for i, (tag, A, Fd) in enumerate(SHAPES):
        torch.manual_seed(i)
        agent = bench.new_agent(cfg, A, Fd, seed=i)
        it = bench.ring_iter(f"/bench_action_dims/{tag}", A, args.episodes, B, dev, seed=1 + i)
        runs.append(dict(tag=tag, A=A, F=Fd, agent=agent, it=it, step=0, ms=[]))
    for r in runs:                                  # eager warm-up, capture, replays
        for _ in range(args.warmup):
            r["agent"].update(r["it"], r["step"])
            r["step"] += 2
    torch.cuda.synchronize()
    for _ in range(args.blocks):
        for r in runs:
            def step(r=r):
                r["agent"].update(r["it"], r["step"])
                r["step"] += 2
            r["ms"] += bench.timed_blocks(step, [args.steps_per_block], 1, dev)
    out = dict(card=name, power_limit=power, batch=B, hidden_dim=args.hidden_dim, steps_per_block=args.steps_per_block,
               shapes={})
    print(f"{name}, power limit {power}; B = {B}, H = {args.hidden_dim}, ring-fed, CUDA graph, "
          f"{args.blocks} alternating blocks of {args.steps_per_block} updates")
    for r in runs:
        _, st = bench.block_stats(r["ms"], [args.steps_per_block] * args.blocks, 1)
        head = bench.in_graph_run_time(r["agent"], r["it"], "drq_policy_head_fwd_bf16")
        rec = dict(A=r["A"], F=r["F"], updates_per_s_median=st["value_median"], updates_per_s_worst=st["value_worst"],
                   updates_per_s_best=st["value_best"], ms_per_update_median=st["ms_per_step_median"],
                   policy_head_us_in_graph=None if head is None else head[0])
        out["shapes"][r["tag"]] = rec
        head_s = "not measured (no external CUDA events)" if head is None else f"{head[0]:.2f} us"
        print(f"{r['tag']:>13} A = {r['A']:3d} F = {r['F']:3d}: {st['value_median']:7.1f} updates/s "
              f"(blocks {st['value_worst']:.1f} .. {st['value_best']:.1f}), policy head in the update {head_s}")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
