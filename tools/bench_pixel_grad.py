"""Cost of real-valued pixels and of gradients w.r.t. them at the walker shape (B = 256, A = 6, F = 50, H = 1024).

  (a) the reference's update body through autograd (tools/bench_autograd.py reference_update) on an agent built with
      pixels="float" against one with pixels="u8", in both differentiable modes, in alternating blocks
  (b) one saliency call, torch.autograd.grad(min(Q1, Q2).sum(), obs) through agent.encoder and agent.critic
  (c) each new kernel alone (drq_conv1_dgrad_{f32,bf16}, drq_random_shift_bwd_f32, the *_from_f32 conv1 kernels)
ms from CUDA events; the card's name and power limit are read in the same process and printed with the numbers.

    python tools/bench_pixel_grad.py [--blocks 5] [--steps-per-block 30] [--out FILE]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bench  # noqa: E402
from bench_autograd import SCHED, card, reference_update  # noqa: E402


def event_ms(fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps-per-block", type=int, default=30)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--kernel-reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pixel_grad.py measures on a CUDA device; none is available")
    from drqv2_b200 import DrQV2Agent, _lib
    from drqv2_b200._lib import call
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, power = card()
    B, A, Fd, H, cin = args.batch, 6, 50, 1024, 9
    g = torch.Generator().manual_seed(0)
    batch = (torch.randint(0, 256, (B, cin, 84, 84), dtype=torch.uint8, generator=g).to(dev),
             (torch.rand(B, A, generator=g) * 2 - 1).to(dev), torch.rand(B, 1, generator=g).to(dev),
             torch.full((B, 1), 0.99 ** 3).to(dev),
             torch.randint(0, 256, (B, cin, 84, 84), dtype=torch.uint8, generator=g).to(dev))

    def agent(differentiable, pixels):
        torch.manual_seed(1)
        return DrQV2Agent((cin, 84, 84), (A,), "cuda", 1e-4, Fd, H, 0.01, 2000, 2, SCHED, 0.3, False,
                          use_cuda_graph=True, seed=1, mode="bf16" if differentiable == "bf16" else "fp32",
                          differentiable=differentiable, pixels=pixels)

    lines = [f"{name}, power limit {power}; B = {B}, A = {A}, F = {Fd}, H = {H}, cin = {cin}, device-resident batch"]
    out = dict(card=name, power_limit=power, batch=B, arms={}, saliency_ms={}, kernel_ms={})
    # (a)
    runs = []
    for diff in (True, "bf16"):
        for pixels in ("u8", "float"):
            runs.append(dict(tag=f"{'fp32' if diff is True else 'bf16'}_{pixels}", agent=agent(diff, pixels), step=0, ms=[]))
    for r in runs:
        def step(r=r):
            reference_update(r["agent"], batch, r["step"])
            r["step"] += 2
        r["fn"] = step
        for _ in range(args.warmup):
            step()
    torch.cuda.synchronize()
    for _ in range(args.blocks):
        for r in runs:
            r["ms"] += bench.timed_blocks(r["fn"], [args.steps_per_block], 1, dev)
    lines.append(f"(a) reference update body through autograd, {args.blocks} alternating blocks of "
                 f"{args.steps_per_block} updates")
    for r in runs:
        _, st = bench.block_stats(r["ms"], [args.steps_per_block] * args.blocks, 1)
        out["arms"][r["tag"]] = dict(ms_per_update_median=st["ms_per_step_median"], ms_min=st["ms_per_step_min"],
                                     ms_max=st["ms_per_step_max"], updates_per_s_median=st["value_median"])
        lines.append(f"  {r['tag']:>10}: {st['ms_per_step_median']:7.3f} ms/update (blocks {st['ms_per_step_min']:.3f} .. "
                     f"{st['ms_per_step_max']:.3f}), {st['value_median']:7.1f} updates/s")
    # (b)
    lines.append("(b) saliency: torch.autograd.grad(min(Q1, Q2).sum(), obs), obs fp32 non-integral, ms per call")
    for r in runs:
        if not r["tag"].endswith("float"):
            continue
        ag = r["agent"]
        obs = (torch.rand(B, cin, 84, 84, generator=g) * 255).to(dev).requires_grad_(True)

        def sal(ag=ag, obs=obs):
            q = torch.min(*ag.critic(ag.encoder(obs), batch[1])).sum()
            torch.autograd.grad(q, obs)
        ms = event_ms(sal, 20)
        out["saliency_ms"][r["tag"]] = ms
        lines.append(f"  {r['tag']:>10}: {ms:7.3f} ms")
    # (c)
    s = torch.cuda.current_stream().cuda_stream
    L = _lib.lib()
    x = (torch.rand(B, cin, 84, 84, generator=g) * 255).to(dev)
    dx = torch.empty_like(x)
    w = (0.1 * torch.randn(32, cin, 3, 3, generator=g)).to(dev)
    b = torch.randn(32, generator=g).to(dev)
    dplanes = torch.randn(B, 32, 1696, generator=g).to(dev)
    planes = torch.empty(B, 32, 1696, device=dev)
    part = torch.empty(L.drq_conv_wgrad_ws_floats(cin), device=dev)
    dw, db = torch.empty(32, cin, 3, 3, device=dev), torch.empty(32, device=dev)
    wb = torch.randn(int(L.drq_wb_elems(B)), generator=g).to(dev).bfloat16()
    wbo = torch.empty_like(wb)
    packed = torch.empty(L.drq_conv1_w_packed_elems(), dtype=torch.bfloat16, device=dev)
    call("drq_pack_conv1_w_bf16", w.data_ptr(), b.data_ptr(), packed.data_ptr(), cin, s)
    part16 = torch.empty(L.drq_conv1_wgrad_bf16_ws_floats(), device=dev)
    shift = torch.randint(0, 9, (B, 2), generator=g, dtype=torch.int32).to(dev)
    u8 = batch[0]
    kernels = {
        "drq_conv1_dgrad_f32": lambda: call("drq_conv1_dgrad_f32", dplanes.data_ptr(), w.data_ptr(), dx.data_ptr(), B, cin, s),
        "drq_conv1_dgrad_bf16": lambda: call("drq_conv1_dgrad_bf16", wb.data_ptr(), packed.data_ptr(), dx.data_ptr(), B, cin, s),
        "drq_random_shift_bwd_f32": lambda: call("drq_random_shift_bwd_f32", x.data_ptr(), shift.data_ptr(), dx.data_ptr(),
                                                 B, cin, 84, 84, 4, s),
        "drq_conv1_fwd_f32_from_f32": lambda: call("drq_conv1_fwd_f32_from_f32", x.data_ptr(), w.data_ptr(), b.data_ptr(),
                                                   planes.data_ptr(), B, cin, s),
        "drq_conv1_fwd_f32 (u8, for comparison)": lambda: call("drq_conv1_fwd_f32", u8.data_ptr(), None, w.data_ptr(),
                                                               b.data_ptr(), planes.data_ptr(), B, cin, 4, s),
        "drq_conv1_wgrad_f32_from_f32": lambda: call("drq_conv1_wgrad_f32_from_f32", x.data_ptr(), dplanes.data_ptr(),
                                                     part.data_ptr(), dw.data_ptr(), db.data_ptr(), B, cin, s),
        "drq_conv1_fwd_bf16_from_f32": lambda: call("drq_conv1_fwd_bf16_from_f32", x.data_ptr(), packed.data_ptr(),
                                                    wbo.data_ptr(), B, cin, s),
        "drq_conv1_fwd_bf16 (u8, for comparison)": lambda: call("drq_conv1_fwd_bf16", u8.data_ptr(), None, packed.data_ptr(),
                                                                wbo.data_ptr(), B, cin, 4, s),
        "drq_conv1_wgrad_bf16_from_f32": lambda: call("drq_conv1_wgrad_bf16_from_f32", x.data_ptr(), wb.data_ptr(),
                                                      part16.data_ptr(), dw.data_ptr(), db.data_ptr(), B, cin, s),
    }
    lines.append(f"(c) kernels alone at N = {B}, cin = {cin}: ms per launch (CUDA events over {args.kernel_reps} launches)")
    for k, fn in kernels.items():
        ms = event_ms(fn, args.kernel_reps)
        out["kernel_ms"][k] = ms
        lines.append(f"  {k:>40}: {ms:8.4f} ms")
    text = "\n".join(lines) + "\n" + json.dumps(out) + "\n"
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
