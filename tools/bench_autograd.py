"""Cost of training through autograd (DrQV2Agent(differentiable=True) driven by the reference's own update body,
drqv2.py:230-262) against the fused update() at the walker shape (B = 256, A = 6, F = 50, H = 1024).

Arms, timed in alternating blocks so that a drift of the shared machine touches all alike:
  autograd     fp32 agent, differentiable=True: aug -> encoder -> update_critic -> update_actor -> soft update as the
               reference writes them (torch losses, loss.backward(), opt.step()), every draw from torch's generator
  autograd_bf16  tensor-core agent, differentiable="bf16": the same body on the tcgen05 kernels
  update_fp32  fp32 agent, update() (CUDA graph) - the same kernels, fused and captured
  update_bf16  the default tensor-core agent, update() (CUDA graph)
All arms take the same device-resident batch.  ms per update from CUDA events at block boundaries; the card's name and
power limit are read in the same process and printed with the numbers.

    python tools/bench_autograd.py [--blocks 5] [--steps-per-block 50]
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402

SCHED = "linear(1.0,0.1,100000)"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (s.strip() for s in q.stdout.strip().split(",")) if q.returncode == 0 else (torch.cuda.get_device_name(), "unknown")
    return name, power


def reference_update(agent, batch, step):
    """drqv2.py:230-262 with update_critic (177-204) and update_actor (206-228) inlined, use_tb off"""
    from drqv2_b200 import utils
    obs, action, reward, discount, next_obs = batch
    obs = agent.aug(obs.float())
    next_obs = agent.aug(next_obs.float())
    obs = agent.encoder(obs)
    with torch.no_grad():
        next_obs = agent.encoder(next_obs)
    with torch.no_grad():
        stddev = utils.schedule(agent.stddev_schedule, step)
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--action-dim", type=int, default=6)
    ap.add_argument("--feature-dim", type=int, default=50)
    ap.add_argument("--hidden-dim", type=int, default=1024)
    ap.add_argument("--steps-per-block", type=int, default=50)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_autograd.py measures on a CUDA device; none is available")
    from drqv2_b200 import DrQV2Agent
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, power = card()
    B, A, Fd, H = args.batch, args.action_dim, args.feature_dim, args.hidden_dim
    g = torch.Generator().manual_seed(0)
    batch = (torch.randint(0, 256, (B, 9, 84, 84), dtype=torch.uint8, generator=g).to(dev),
             (torch.rand(B, A, generator=g) * 2 - 1).to(dev), torch.rand(B, 1, generator=g).to(dev),
             torch.full((B, 1), 0.99 ** 3).to(dev),
             torch.randint(0, 256, (B, 9, 84, 84), dtype=torch.uint8, generator=g).to(dev))

    def agent(mode, differentiable=False):
        torch.manual_seed(1)
        return DrQV2Agent((9, 84, 84), (A,), "cuda", 1e-4, Fd, H, 0.01, 2000, 2, SCHED, 0.3, False, use_cuda_graph=True,
                          seed=1, mode=mode, differentiable=differentiable)

    class Forever:
        def __iter__(self):
            return self

        def __next__(self):
            return batch

    runs = [dict(tag="autograd", agent=agent("fp32", True)), dict(tag="autograd_bf16", agent=agent("bf16", "bf16")),
            dict(tag="update_fp32", agent=agent("fp32")),
            dict(tag="update_bf16", agent=agent("bf16"))]
    for r in runs:
        r.update(step=0, ms=[], it=Forever())

        def step(r=r):
            if r["tag"].startswith("autograd"):
                reference_update(r["agent"], batch, r["step"])
            else:
                r["agent"].update(r["it"], r["step"])
            r["step"] += 2
        r["fn"] = step
        for _ in range(args.warmup):               # eager warm-up, capture, replays / allocator warm-up
            step()
    torch.cuda.synchronize()
    for _ in range(args.blocks):
        for r in runs:
            r["ms"] += bench.timed_blocks(r["fn"], [args.steps_per_block], 1, dev)
    out = dict(card=name, power_limit=power, batch=B, action_dim=A, feature_dim=Fd, hidden_dim=H,
               steps_per_block=args.steps_per_block, blocks=args.blocks, arms={})
    print(f"{name}, power limit {power}; B = {B}, A = {A}, F = {Fd}, H = {H}, device-resident batch, "
          f"{args.blocks} alternating blocks of {args.steps_per_block} updates")
    for r in runs:
        _, st = bench.block_stats(r["ms"], [args.steps_per_block] * args.blocks, 1)
        out["arms"][r["tag"]] = dict(ms_per_update_median=st["ms_per_step_median"], ms_per_update_min=st["ms_per_step_min"],
                                     ms_per_update_max=st["ms_per_step_max"], updates_per_s_median=st["value_median"])
        print(f"{r['tag']:>12}: {st['ms_per_step_median']:7.3f} ms/update (blocks {st['ms_per_step_min']:.3f} .. "
              f"{st['ms_per_step_max']:.3f}), {st['value_median']:7.1f} updates/s")
    for arm in ("autograd", "autograd_bf16"):
        ag = out["arms"][arm]["ms_per_update_median"]
        for tag in ("update_fp32", "update_bf16"):
            out[f"{arm}_over_{tag}"] = ag / out["arms"][tag]["ms_per_update_median"]
            print(f"{arm} path / {tag}: {out[f'{arm}_over_{tag}']:.2f}x")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
