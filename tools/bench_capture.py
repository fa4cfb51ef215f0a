"""The reference's update body through autograd, eager and captured in a CUDA graph, at the walker shape (B = 256,
A = 6, F = 50, H = 1024, device-resident batch), against the fused update().

Arms, timed in alternating blocks in one process so that a drift of the shared machine touches all alike:
  bf16_plain    DrQV2Agent(mode="bf16", differentiable="bf16", pixels="float"): the body run eagerly on a plain agent,
                whose step() takes its Adam scalars from the host through the scalar ring (the path of
                profiles/autograd_b256.txt and profiles/pixel_grad_b256.txt)
  bf16_eager    the same agent built with capturable=True, run eagerly (step(): scalars derived on the device)
  bf16_graph    the capturable agent's body captured once and replayed (INTEGRATION.md, "Capturing the update body";
                the stddev is a 0-d tensor written before each replay)
  fp32_*        the same three with mode="fp32", differentiable=True (the fp32 CUDA-core kernels)
  update_bf16   the default tensor-core agent's fused, captured update()
ms per update from CUDA events at block boundaries.  A separate torch.profiler pass counts the device activities
(kernels, copies, memsets) per update and sums their durations.  The card's name and power limit are read in the
same process and printed with the numbers.

    python tools/bench_capture.py [--blocks 5] [--steps-per-block 50] [--out FILE]
"""
import argparse
import json
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bench  # noqa: E402
from bench_autograd import SCHED, card  # noqa: E402


def reference_body(agent, batch, stddev):
    """drqv2.py:230-262 with update_critic (177-204) and update_actor (206-228) inlined, use_tb off; `stddev` is
    utils.schedule(...) of the step (a float eagerly, a 0-d CUDA tensor the caller rewrites inside a graph)"""
    from drqv2_b200 import utils
    obs, action, reward, discount, next_obs = batch
    obs = agent.aug(obs.float())
    next_obs = agent.aug(next_obs.float())
    obs = agent.encoder(obs)
    with torch.no_grad():
        next_obs = agent.encoder(next_obs)
    with torch.no_grad():
        dist = agent.actor(next_obs, stddev)
        next_action = dist.sample(clip=agent.stddev_clip)
        target_Q1, target_Q2 = agent.critic_target(next_obs, next_action)
        target_V = torch.min(target_Q1, target_Q2)
        target_Q = reward + (discount * target_V)
    Q1, Q2 = agent.critic(obs, action)
    critic_loss = F.mse_loss(Q1, target_Q) + F.mse_loss(Q2, target_Q)
    agent.encoder_opt.zero_grad(set_to_none=True)
    agent.critic_opt.zero_grad(set_to_none=True)
    critic_loss.backward()
    agent.critic_opt.step()
    agent.encoder_opt.step()
    obs = obs.detach()
    dist = agent.actor(obs, stddev)
    action = dist.sample(clip=agent.stddev_clip)
    log_prob = dist.log_prob(action).sum(-1, keepdim=True)   # noqa: F841  (the reference computes it for its metrics)
    Q1, Q2 = agent.critic(obs, action)
    actor_loss = -torch.min(Q1, Q2).mean()
    agent.actor_opt.zero_grad(set_to_none=True)
    actor_loss.backward()
    agent.actor_opt.step()
    utils.soft_update_params(agent.critic, agent.critic_target, agent.critic_target_tau)


def device_activity(fn, n):
    """(device activities per call, sum of their durations per call in ms) over n calls, from torch.profiler"""
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
    evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return len(evs) / n, sum(e.time_range.elapsed_us() for e in evs) / n / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps-per-block", type=int, default=50)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--profile-steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_capture.py measures on a CUDA device; none is available")
    from drqv2_b200 import DrQV2Agent, utils
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, power = card()
    B, A, Fd, H, cin = args.batch, 6, 50, 1024, 9
    g = torch.Generator().manual_seed(0)
    batch = (torch.randint(0, 256, (B, cin, 84, 84), dtype=torch.uint8, generator=g).to(dev),
             (torch.rand(B, A, generator=g) * 2 - 1).to(dev), torch.rand(B, 1, generator=g).to(dev),
             torch.full((B, 1), 0.99 ** 3).to(dev),
             torch.randint(0, 256, (B, cin, 84, 84), dtype=torch.uint8, generator=g).to(dev))

    def agent(mode, differentiable=False, capturable=False):
        torch.manual_seed(1)
        return DrQV2Agent((cin, 84, 84), (A,), "cuda", 1e-4, Fd, H, 0.01, 2000, 2, SCHED, 0.3, False,
                          use_cuda_graph=True, seed=1, mode=mode, differentiable=differentiable,
                          pixels="float" if differentiable else "u8", capturable=capturable)

    class Forever:
        def __iter__(self):
            return self

        def __next__(self):
            return batch

    runs = []
    for tag, mode, diff in (("bf16", "bf16", "bf16"), ("fp32", "fp32", True)):
        runs.append(dict(tag=f"{tag}_plain", agent=agent(mode, diff)))
        runs.append(dict(tag=f"{tag}_eager", agent=agent(mode, diff, capturable=True)))
        runs.append(dict(tag=f"{tag}_graph", agent=agent(mode, diff, capturable=True)))
    runs.append(dict(tag="update_bf16", agent=agent("bf16")))
    for r in runs:
        r.update(step=0, ms=[])
        ag = r["agent"]
        if r["tag"].endswith(("_plain", "_eager")):
            def step(r=r, ag=ag):
                reference_body(ag, batch, utils.schedule(SCHED, r["step"]))
                r["step"] += 2
            for _ in range(args.warmup):
                step()
        elif r["tag"].endswith("_graph"):
            std = torch.tensor(utils.schedule(SCHED, 0), device=dev)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):           # warm-up on a side stream, then capture
                for _ in range(args.warmup):
                    reference_body(ag, batch, std)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                reference_body(ag, batch, std)
            r["graph"] = graph

            def step(r=r, std=std, graph=graph):
                std.fill_(utils.schedule(SCHED, r["step"]))
                graph.replay()
                r["step"] += 2
            step()
        else:
            it = Forever()

            def step(r=r, ag=ag, it=it):
                ag.update(it, r["step"])
                r["step"] += 2
            for _ in range(args.warmup):
                step()
        r["fn"] = step
    torch.cuda.synchronize()
    for _ in range(args.blocks):
        for r in runs:
            r["ms"] += bench.timed_blocks(r["fn"], [args.steps_per_block], 1, dev)
    for r in runs:                                  # a separate pass: tracing slows the host
        r["launches"], r["kernel_ms"] = device_activity(r["fn"], args.profile_steps)
    for r in runs:
        if r["tag"].endswith("_graph"):
            steps = r["agent"].encoder_opt.state_dict()["step"]
            assert steps == args.warmup + r["step"] // 2, (r["tag"], steps)   # every replay stepped

    out = dict(card=name, power_limit=power, batch=B, action_dim=A, feature_dim=Fd, hidden_dim=H,
               steps_per_block=args.steps_per_block, blocks=args.blocks, arms={})
    lines = [f"{name}, power limit {power}; B = {B}, A = {A}, F = {Fd}, H = {H}, cin = {cin}, pixels='float' for the "
             f"reference body, device-resident batch; {args.blocks} alternating blocks of {args.steps_per_block} updates",
             f"{'arm':>12}  ms/update (blocks min .. max)  updates/s | device activities per update, sum of their "
             f"durations (torch.profiler, {args.profile_steps} updates, separate pass)"]
    for r in runs:
        _, st = bench.block_stats(r["ms"], [args.steps_per_block] * args.blocks, 1)
        out["arms"][r["tag"]] = dict(ms_per_update_median=st["ms_per_step_median"], ms_per_update_min=st["ms_per_step_min"],
                                     ms_per_update_max=st["ms_per_step_max"], updates_per_s_median=st["value_median"],
                                     device_activities_per_update=r["launches"], device_ms_per_update=r["kernel_ms"])
        lines.append(f"{r['tag']:>12}: {st['ms_per_step_median']:7.3f} ({st['ms_per_step_min']:.3f} .. "
                     f"{st['ms_per_step_max']:.3f}) {st['value_median']:7.1f} | {r['launches']:6.1f}, "
                     f"{r['kernel_ms']:7.3f} ms")
    for kind in ("bf16", "fp32"):
        pl, e, c = (out["arms"][f"{kind}_{x}"]["ms_per_update_median"] for x in ("plain", "eager", "graph"))
        out[f"{kind}_plain_over_graph"] = pl / c
        out[f"{kind}_eager_over_graph"] = e / c
        lines.append(f"{kind}: plain eager / captured {pl / c:.2f}x, capturable eager / captured {e / c:.2f}x; "
                     f"captured / fused update() {c / out['arms']['update_bf16']['ms_per_update_median']:.2f}x")
    text = "\n".join(lines) + "\n" + json.dumps(out) + "\n"
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
