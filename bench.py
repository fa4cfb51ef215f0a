#!/usr/bin/env python
"""Benchmark of the DrQ-v2 agent update (BASELINE.json metric: updates/sec at batch 256).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one DrQV2Agent.update (critic + actor + soft target update) on a fresh
batch of the walker_walk shape (B=256, 9x84x84 uint8 stacks, A=6, F=50, H=1024, n-step 3).

ours      : `value` = updates/s with the replay ring resident in HBM (sample + n-step
            gather + update captured in one CUDA graph, timed with CUDA events; the K timed steps are
            split into --blocks blocks, `value` is the median block, min / max are reported beside it);
            --dump-outputs DIR writes the parameters and metrics of the last timed step (seeded inputs:
            the same arguments give the same inputs, so two builds can be compared output for output);
            `e2e` = the same update through the public API fed from HOST batches
            (pinned memory -> H2D inside the timed region, metrics read back D2H).
            Before anything is timed, one update at this configuration is checked against the oracle
            (`parity_checked`).  Every launch of one update is then timed alone (L2 flushed before each) for the
            roofline record; the unmodified reference runs on the same GPU (`gpu_reference`: eager, TF32 on/off,
            and captured in a CUDA graph with Adam(capturable=True)) and on the host cores (`cpu_baseline`).
            Sub-records `ensemble_8_per_gpu` (BASELINE configs[3]) and `dp_humanoid_b4096` (configs[4]) carry
            the two multi-GPU configurations with their own one-GPU points.
reference : the reference's own update on the host cores (unmodified sources from baseline/_ref, else the
            oracle port), --steps timed updates (default 40).
Multi-GPU : one process per GPU (torchrun); the headline is independent agents (ensemble members) with no
            collective, value = sum over ranks / max-over-ranks time, scaling "weak".
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SCHED = "linear(1.0,0.1,100000)"
E_F, E_B = 84_561_984, 160_409_664     # encoder fwd / bwd FLOP per sample (SURVEY §8d)
CONV_MACS = {39: 14_017_536, 37: 12_616_704, 35: 11_289_600}
CONV1_MACS_PER_CIN = 41 * 41 * 32 * 9   # x cin


def update_flops(B, A, F, H):
    T = 2 * 39200 * F
    Q = 2 * ((F + A) * H + H * H + H)
    P = 2 * (F * H + H * H + H * A)
    return B * (2 * E_F + E_B + 8 * T + (2 * P + 6 * Q) + (6 * Q + 2 * P))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def fill_ring(loader_dir, A, episodes, rows, device, seed=1):
    """SURVEY §8d synthetic replay: E episodes x rows steps of uniform u8 frames, action~U(-1,1),
    reward~U(0,1), discount 1; row 0 is the reset dummy.  Written straight into the ring."""
    from drqv2_b200 import replay_buffer as rb
    cap = episodes * rows
    ring = rb.GpuRing(cap, 3, 3, A, device)
    g = torch.Generator(device=device).manual_seed(seed)
    ring.frames.copy_(torch.randint(0, 256, ring.frames.shape, dtype=torch.uint8, device=device, generator=g))
    ring.action.copy_(torch.rand(cap, A, device=device, generator=g) * 2 - 1)
    ring.reward.copy_(torch.rand(cap, device=device, generator=g))
    ring.discount.fill_(1.0)
    starts = torch.arange(episodes, device=device) * rows
    ring.action[starts] = 0
    ring.reward[starts] = 0
    ring.episodes = [(int(e * rows), rows) for e in range(episodes)]
    ring.head = 0
    ring._upload_table()
    rb._RINGS[str(loader_dir)] = dict(ring=ring, capacity=cap, storage=None)
    return ring


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d["bf16_tflops"], d.get("bf16_tflops_sustained", d["bf16_tflops"]), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


def new_agent(args, A, Fd, seed, mode=None, dp=False, lr=1e-4):
    from drqv2_b200 import DrQV2Agent
    return DrQV2Agent((9, 84, 84), (A,), "cuda", lr, Fd, args.hidden_dim, 0.01, 2000, 2, SCHED, 0.3, False,
                      use_cuda_graph=True, seed=seed, mode=mode or args.mode, data_parallel=dp)


def ring_iter(key, A, episodes, B, dev, seed):
    from drqv2_b200 import make_replay_loader
    fill_ring(key, A, episodes, 501, dev, seed=seed)
    return iter(make_replay_loader(key, episodes * 501, B, 0, False, 3, 0.99))


def block_sizes(steps, blocks):
    """`steps` updates split into at most `blocks` back-to-back blocks of near-equal size (none empty)."""
    n = max(1, min(blocks, steps))
    return [steps // n + (i < steps % n) for i in range(n)]


def timed_blocks(step_fn, sizes, world, dev):
    """Blocks of exactly sizes[i] updates, enqueued back to back after one barrier + synchronize and timed with CUDA
    events on the launching stream at every block boundary: nothing pauses between blocks, so only the first carries
    the pipeline fill, however the steps are split.  Per block the max over ranks.  Returns the ms of every block."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(sizes) + 1)]
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    ev[0].record()
    for e, steps in zip(ev[1:], sizes):
        for _ in range(steps):
            step_fn()
        e.record()
    torch.cuda.synchronize()
    out = [a.elapsed_time(b) for a, b in zip(ev, ev[1:])]
    if world > 1:
        t = torch.tensor(out, device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        out = t.tolist()
    return out


def block_stats(ms_blocks, sizes, units):
    per = sorted(m / n for m, n in zip(ms_blocks, sizes))
    med = statistics.median(per)
    return med, {"blocks": len(per), "steps_per_block": sizes, "ms_per_step_median": med, "ms_per_step_min": per[0],
                 "ms_per_step_max": per[-1], "value_median": units * 1e3 / med, "value_best": units * 1e3 / per[0],
                 "value_worst": units * 1e3 / per[-1]}


# ----------------------------------------------------------------------------- parity at the benched configuration
def parity_check(args):
    """One update at the benched shape (B, A, F, H, mode) from identical parameters and injected draws against the
    oracle (bf16 mode: its bf16-faithful variant), through the same CUDA-graph path the timed loop replays.
    Tolerances are the ones tests/test_gpu_bench_config.py states."""
    from oracle import drq_oracle as O
    B, A, Fd, H = args.batch, args.action_dim, args.feature_dim, args.hidden_dim
    torch.set_num_threads(os.cpu_count())
    params = O.synthetic_params(9, A, Fd, H, seed=4)
    agent = new_agent(args, A, Fd, seed=5)
    agent.use_tb = True
    for net in ("encoder", "actor", "critic", "critic_target"):
        getattr(agent, net).load_state_dict(params[net])
    agent.refresh()
    bf = args.mode == "bf16"
    oracle = O.OracleAgent(params, 1e-4, 0.01, SCHED, 0.3, dtype=torch.float64, operands="bf16" if bf else "exact")
    worst, rec = 0.0, {}
    keys = ("batch_reward", "critic_target_q", "critic_q1", "critic_q2", "critic_loss")
    for s in range(3):                      # eager warm-up, capture + first replay, replay
        b = O.synthetic_batch(B, A, seed=10 + s)
        agent.inject_draws(b["shift_obs"], b["shift_next"], b["eps_critic"], b["eps_actor"])
        m = agent.update(iter([(b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"])]), 2 * s)
        mo = oracle.update(b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"], 2 * s, b["shift_obs"],
                           b["shift_next"], b["eps_critic"], b["eps_actor"])
        tol = (2e-3 if bf else 1e-4) if s == 0 else 2e-2     # after an Adam step: its sign-like noise (SURVEY §8c)
        for k in keys:
            err = abs(m[k] - mo[k]) / (abs(mo[k]) + 1e-12)
            rec[f"update{s}.{k}"] = err
            worst = max(worst, err / tol)
    lr = 1e-4
    dmax = max((p.detach().cpu().double() - oracle.p[net][name]).abs().max().item()
               for net in ("encoder", "critic", "actor", "critic_target") for name, p in getattr(agent, net).named_parameters())
    ok = worst <= 1.0 and dmax <= 2.5 * lr * 3
    graphed = any(isinstance(v, torch.cuda.CUDAGraph) for v in agent._graphs.values())
    return {"parity_checked": bool(ok and graphed),
            "parity": {"oracle": "oracle/drq_oracle.py OracleAgent(float64, operands=%s)" % ("bf16" if bf else "exact"),
                       "updates_compared": 3, "max_rel_err_first_update": max(rec[f"update0.{k}"] for k in keys),
                       "max_rel_err_later_updates": max(v for k, v in rec.items() if not k.startswith("update0")),
                       "max_abs_param_diff_over_lr": dmax / lr, "cuda_graph_path": graphed}}


# ----------------------------------------------------------------------------- every launch of one update, timed alone
def profile_update_launches(agent, it, B, reps=5):
    """Runs eager single-stream updates with every C-ABI call bracketed by CUDA events on its launch stream and a
    write of a 256 MB buffer (> the 126 MB L2) in front of it: per launch the cold-cache duration, plus the
    algorithmic FLOP / bytes the call's own arguments imply.  Median over `reps` updates."""
    import drqv2_b200._bf16 as BF
    import drqv2_b200.drqv2 as D
    import drqv2_b200.replay_buffer as R
    from drqv2_b200 import _lib
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    orig = _lib.call
    records, cur = [], []

    def work_of(name, a):
        if name == "drq_conv1_fwd_bf16":
            return "conv", f"conv1_fwd(N={a[4]})", 2 * CONV1_MACS_PER_CIN * a[5] * a[4], 0
        if name == "drq_conv1_wgrad_bf16":
            return "conv", f"conv1_wgrad(N={a[6]})", 2 * CONV1_MACS_PER_CIN * a[7] * a[6], 0
        if name == "drq_conv1_fwd_bf16_ring":        # 9 stacked channels (3 frames x RGB), rows straight from the ring
            return "conv", f"conv1_fwd(N={a[5]},from ring)", 2 * CONV1_MACS_PER_CIN * 9 * a[5], 0
        if name == "drq_conv1_wgrad_bf16_ring":
            return "conv", f"conv1_wgrad(N={a[7]},from ring)", 2 * CONV1_MACS_PER_CIN * 9 * a[7], 0
        if name == "drq_conv3x3_fwd_bf16":
            return "conv", f"conv3x3_fwd(hout={a[5]},N={a[4]}{',TB' if a[6] == 2 else ''})", 2 * CONV_MACS[a[5]] * a[4], 0
        if name == "drq_conv3x3_dgrad_bf16":
            return "conv", f"conv3x3_dgrad(hout={a[6]},N={a[5]})", 2 * CONV_MACS[a[6]] * a[5], 0
        if name == "drq_conv3x3_wgrad_bf16":
            return "conv", f"conv3x3_wgrad(hout={a[7]},N={a[6]})", 2 * CONV_MACS[a[7]] * a[6], 0
        if name == "drq_gemm_bf16":
            M, N, K, batch = a[11], a[12], a[13], a[16]
            return "gemm", f"gemm(mode={a[4]},M={M},N={N},K={K},batch={batch},splitk={a[19]},bn={a[20]},epi={a[14]})", 2 * M * N * K * batch, 0
        if name.startswith("drq_conv") and name.endswith("_f32") or name == "drq_gemm_f32":
            return "fp32", name, 0, 0
        if name == "drq_adam_pack_step":
            plan, n = a[9], a[10]
            by = sum((12 if plan[i].ema else 28) * plan[i].n + (2 * plan[i].n if plan[i].kind else 0) for i in range(n))
            return "hbm", f"adam_pack(segs={n})", 0, by
        if name in ("drq_adam_step", "drq_adam_ema_step"):
            return "hbm", name, 0, 28 * a[4] + (12 * a[8] if name == "drq_adam_ema_step" else 0)
        if name == "drq_ring_gather_nstep":
            return "hbm", "ring_gather", 0, 2 * 2 * a[10] * a[5] * a[6] * 84 * 84
        return "latency", name, 0, 0

    def timed_call(name, *a):
        s = torch.cuda.current_stream()
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        orig(name, *a)
        e1.record(s)
        cur.append((name, a, e0, e1))

    was_graph, was_overlap = agent.use_cuda_graph, agent.overlap_encoder_backward
    agent.use_cuda_graph, agent.overlap_encoder_backward = False, False      # one stream: every launch alone
    step = 10_000
    try:
        agent.update(it, step)
        D.call = R.call = BF.call = timed_call
        for r in range(reps):
            cur.clear()
            step += 2
            agent.update(it, step)
            torch.cuda.synchronize()
            records.append([(n, a, e0.elapsed_time(e1)) for n, a, e0, e1 in cur])
        # second pass, in sequence: nothing is flushed, and a run of consecutive launches of the same entry point (the three
        # conv3x3 forwards behind conv1) shares ONE bracket - every launch finds the cache state it has in the real update
        # (its input was just written by the launch in front of it) and the bracket's cost is paid once per run
        runs, state = [], {"name": None, "e0": None, "e1": None, "n": 0}

        def seq_call(name, *a):
            s_ = torch.cuda.current_stream()
            if name != state["name"]:
                if state["name"] is not None:
                    runs.append((state["name"], state["n"], state["e0"], state["e1"]))
                state.update(name=name, n=0, e0=torch.cuda.Event(enable_timing=True))
                state["e0"].record(s_)
            orig(name, *a)
            state["n"] += 1
            state["e1"] = torch.cuda.Event(enable_timing=True)
            state["e1"].record(s_)

        D.call = R.call = BF.call = seq_call
        seq_records = []
        for r in range(reps):
            runs.clear()
            state.update(name=None, n=0)
            step += 2
            agent.update(it, step)
            if state["name"] is not None:
                runs.append((state["name"], state["n"], state["e0"], state["e1"]))
            torch.cuda.synchronize()
            seq_records.append([(n, k, e0.elapsed_time(e1) * 1e3) for n, k, e0, e1 in runs])
        profile_update_launches.sequence_runs = [
            {"entry": seq_records[0][i][0], "launches": seq_records[0][i][1],
             "us": statistics.median(rec[i][2] for rec in seq_records)} for i in range(len(seq_records[0]))]
    finally:
        D.call = R.call = BF.call = orig
        agent.use_cuda_graph, agent.overlap_encoder_backward = was_graph, was_overlap
    # what the bracket itself costs: a one-thread kernel timed in exactly the same way (flush, event, launch, event)
    scratch = torch.zeros(1, dtype=torch.int64, device="cuda")
    floor = []
    for _ in range(9):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig("drq_counter_advance", scratch.data_ptr(), torch.cuda.current_stream().cuda_stream)
        e1.record()
        torch.cuda.synchronize()
        floor.append(e0.elapsed_time(e1) * 1e3)
    profile_update_launches.event_floor_us = statistics.median(floor)
    launches = []
    for i, (name, a, _) in enumerate(records[0]):
        ms = statistics.median(rec[i][2] for rec in records)
        cls, label, flop, by = work_of(name, a)
        launches.append({"i": i, "kernel": label, "class": cls, "us": ms * 1e3, "flop": flop, "bytes": by})
    del flush
    return launches


def roofline_record(launches, value, world, flops_update, mode):
    hbm, tf_burst, tf_sust, src = peaks()
    traffic_file = os.path.join(ROOT, "profiles", "r2c_dram_traffic.json")
    traffic = json.load(open(traffic_file)) if os.path.exists(traffic_file) else {}

    def cls(c):
        sel = [l for l in launches if l["class"] == c]
        us = sum(l["us"] for l in sel)
        return sel, us

    roof = {"peak_source": src, "timing": "every launch of one eager single-stream update timed alone with CUDA events on "
            "its launch stream, a 256 MB buffer written in front of each (cold L2); median of 5 updates",
            "event_bracket_floor_us": getattr(profile_update_launches, "event_floor_us", None),
            "event_bracket_floor_note": "a one-thread kernel timed in the same bracket: every `us` below includes about this much "
                                        "launch / event overhead that ncu's gpu__time_duration (profiles/) does not"}
    tensor = [l for l in launches if l["class"] in ("conv", "gemm") and l["flop"]]
    if tensor:
        # the dominant kernel = the kernel (entry point) with the largest share of the update's time; its achieved rate is
        # its algorithmic FLOP over its summed cold-cache launch time.  The slowest single launch is reported beside it.
        def kernel_of(label):          # one family per kernel function: gemm_tc_kernel<MODE, BN, EPI> instantiations are different kernels
            name = label.split("(")[0]
            if name != "gemm":
                return name
            kv = dict(p.split("=") for p in label[label.index("(") + 1:-1].split(","))
            return f"gemm<mode={kv['mode']},bn={kv['bn']},epi={kv['epi']}>"
        fam = {}
        for l in tensor:
            f = fam.setdefault(kernel_of(l["kernel"]), {"us": 0.0, "flop": 0, "launches": []})
            f["us"] += l["us"]; f["flop"] += l["flop"]; f["launches"].append(l["kernel"])
        name, dom = max(fam.items(), key=lambda kv: kv[1]["us"])
        ach = dom["flop"] / (dom["us"] * 1e-6) / 1e12
        tr = (traffic.get("kernels", {}).get(name) or {})
        floor = roof["event_bracket_floor_us"] or 0.0
        net_us = dom["us"] - floor * len(dom["launches"])
        roof.update({"bound": "tensor", "kernel": name, "kernel_launches": dom["launches"], "achieved": ach, "peak": tf_burst,
                     "unit": "TFLOP/s", "frac": ach / tf_burst, "kernel_us": dom["us"] / len(dom["launches"]),
                     "frac_net_of_event_bracket": (dom["flop"] / (net_us * 1e-6) / 1e12 / tf_burst) if net_us > 0 else None,
                     "traffic": tr.get("dram_bytes"), "traffic_launch": tr.get("launch"), "traffic_source": traffic.get("source")})
        # the same kernel's launches timed in sequence (profile_update_launches, second pass): the headline achieved / frac
        entry = {"conv3x3_fwd": "drq_conv3x3_fwd_bf16", "conv3x3_dgrad": "drq_conv3x3_dgrad_bf16",
                 "conv3x3_wgrad": "drq_conv3x3_wgrad_bf16"}.get(name)
        seq = [r for r in getattr(profile_update_launches, "sequence_runs", []) if r["entry"] == entry]
        if seq and sum(r["launches"] for r in seq) == len(dom["launches"]):
            us_seq = sum(r["us"] for r in seq)
            ach_seq = dom["flop"] / (us_seq * 1e-6) / 1e12
            roof["cold_isolated"] = {"achieved": ach, "frac": ach / tf_burst, "kernel_us": roof["kernel_us"],
                                     "frac_net_of_event_bracket": roof.pop("frac_net_of_event_bracket"),
                                     "note": "every launch alone behind an L2 flush, one event bracket each (the per-launch list below)"}
            roof.update({"achieved": ach_seq, "frac": ach_seq / tf_burst, "kernel_us": us_seq / len(dom["launches"]),
                         "measured": "%d run(s) of consecutive launches of this kernel, as they follow each other in the update "
                                     "(eager, one stream, nothing flushed: each launch reads what the launch in front of it just "
                                     "wrote), one CUDA-event bracket per run (%d bracket(s) of ~%.1f us included), median of 5 updates"
                                     % (len(seq), len(seq), floor)})
        slow = max(tensor, key=lambda l: l["us"])
        sach = slow["flop"] / (slow["us"] * 1e-6) / 1e12
        roof["slowest_launch"] = {"kernel": slow["kernel"], "us": slow["us"], "achieved": sach, "frac": sach / tf_burst,
                                  "traffic": (traffic.get("kernels", {}).get(slow["kernel"].split("(")[0]) or {}).get("dram_bytes")}
        for c in ("conv", "gemm"):
            sel, us = cls(c)
            fl = sum(l["flop"] for l in sel)
            if us:
                roof[f"{c}_class"] = {"launches": len(sel), "us": us, "flop": fl, "achieved": fl / (us * 1e-6) / 1e12,
                                      "frac": fl / (us * 1e-6) / 1e12 / tf_burst, "unit": "TFLOP/s"}
    else:
        roof.update({"bound": "tensor", "kernel": "fp32 CUDA-core path (parity mode)", "achieved": None, "peak": tf_burst,
                     "unit": "TFLOP/s", "frac": None, "traffic": None})
    sel, us = cls("hbm")
    roof["hbm_kernels"] = [{"kernel": l["kernel"], "us": l["us"], "bytes": l["bytes"], "achieved_gbs": l["bytes"] / (l["us"] * 1e-6) / 1e9,
                            "frac": l["bytes"] / (l["us"] * 1e-6) / 1e9 / hbm, "peak_gbs": hbm} for l in sel]
    _, us_lat = cls("latency")
    roof["latency_class"] = {"launches": len(cls("latency")[0]), "us": us_lat}
    roof["serial_sum_us"] = sum(l["us"] for l in launches)
    roof["whole_update"] = {"flop": flops_update, "achieved_per_gpu": flops_update * value / world / 1e12,
                            "frac_of_burst": flops_update * value / world / 1e12 / tf_burst,
                            "frac_of_sustained": flops_update * value / world / 1e12 / tf_sust}
    roof["launches"] = [{k: (round(v, 2) if k == "us" else v) for k, v in l.items() if k != "i"} for l in launches]
    return roof


def in_graph_run_time(agent, it, entry, step0=20_000, reps=20):
    """GPU time of the launches of C-ABI entry point `entry` INSIDE the captured update graph: the update is captured once
    more with two external CUDA events (event-record nodes: torch.cuda.Event(external=True)) around the run of consecutive
    `entry` launches, replayed `reps` times, and the events' distance read after every replay.  Returns (median us of the
    run, launches in the run) or None when this torch build has no external events."""
    import drqv2_b200._bf16 as BF
    import drqv2_b200.drqv2 as D
    import drqv2_b200.replay_buffer as R
    from drqv2_b200 import _lib
    orig = _lib.call
    ev = {"e0": None, "e1": None, "n": 0}

    def marked_call(name, *a):
        cap = torch.cuda.is_current_stream_capturing()
        if cap and name == entry and ev["e0"] is None:
            ev["e0"] = torch.cuda.Event(enable_timing=True, external=True)
            ev["e0"].record(torch.cuda.current_stream())
        r = orig(name, *a)
        if cap and name == entry:
            ev["n"] += 1
        return r

    # the closing event goes behind the LAST launch of the run: wrap so that the first different call after the run records it
    def marked_call2(name, *a):
        cap = torch.cuda.is_current_stream_capturing()
        if cap and name != entry and ev["e0"] is not None and ev["e1"] is None and not name.startswith(("drq_set_", "drq_debug_")):
            ev["e1"] = torch.cuda.Event(enable_timing=True, external=True)
            ev["e1"].record(torch.cuda.current_stream())
        return marked_call(name, *a)

    saved = dict(agent._graphs)
    try:
        agent._graphs.clear()
        D.call = R.call = BF.call = marked_call2
        step = step0
        for _ in range(2):                       # eager warm-up, then the capture
            agent.update(it, step); step += 2
        if ev["e0"] is None or ev["e1"] is None:
            return None
        D.call = R.call = BF.call = orig
        ts = []
        for _ in range(reps):
            agent.update(it, step); step += 2
            torch.cuda.synchronize()
            ts.append(ev["e0"].elapsed_time(ev["e1"]) * 1e3)
        return statistics.median(ts), ev["n"]
    except (TypeError, RuntimeError):
        return None
    finally:
        D.call = R.call = BF.call = orig
        agent._graphs.clear()
        agent._graphs.update(saved)


# ----------------------------------------------------------------------------- the reference on the same GPU
def gpu_reference(args, steps=30):
    """The unmodified reference agent (baseline/_ref) on cuda: eager with cudnn.benchmark as train.py:25 sets it,
    TF32 on (its default) and off, and the same update captured in a CUDA graph with Adam(capturable=True)."""
    ref = _load_reference()
    if ref is None:
        return {"unavailable": "baseline/_ref not present"}
    B, A, Fd, H = args.batch, args.action_dim, args.feature_dim, args.hidden_dim
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(1)
    batch = tuple(t.to(dev) for t in (
        torch.randint(0, 256, (B, 9, 84, 84), dtype=torch.uint8, generator=g), torch.rand(B, A, generator=g) * 2 - 1,
        torch.rand(B, 1, generator=g), torch.full((B, 1), 0.970299065),
        torch.randint(0, 256, (B, 9, 84, 84), dtype=torch.uint8, generator=g)))

    def it():
        while True:
            yield batch

    saved = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    out = {}

    def time_updates(fn, n):
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    def count_launches(fn):
        try:
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn()
                torch.cuda.synchronize()
            return sum(e.count for e in prof.key_averages() if e.device_type == torch.autograd.DeviceType.CUDA)
        except Exception as e:                       # CUPTI may be unavailable on the box
            return f"unavailable: {type(e).__name__}"

    try:
        torch.backends.cudnn.benchmark = True
        for tag, tf32 in (("eager_tf32_on", True), ("eager_tf32_off", False)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.manual_seed(0)
            agent = ref.DrQV2Agent((9, 84, 84), (A,), "cuda", 1e-4, Fd, H, 0.01, 2000, 2, SCHED, 0.3, False)
            ri, st = it(), [0]

            def one():
                agent.update(ri, st[0])
                st[0] += 2
            ms = time_updates(one, steps)
            out[tag] = {"updates_per_s": 1e3 / ms, "ms_per_update": ms, "launches_per_update": count_launches(one)}
        # graph-captured: the reference's own update() with capturable Adam (its ops, no host sync at use_tb=False)
        try:
            torch.backends.cudnn.allow_tf32 = True
            torch.manual_seed(0)
            agent = ref.DrQV2Agent((9, 84, 84), (A,), "cuda", 1e-4, Fd, H, 0.01, 2000, 2, SCHED, 0.3, False)
            for net in ("encoder", "actor", "critic"):
                setattr(agent, f"{net}_opt", torch.optim.Adam(getattr(agent, net).parameters(), lr=1e-4, capturable=True))
            ri = it()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for i in range(4):
                    agent.update(ri, 2 * i)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                agent.update(ri, 8)
            ms = time_updates(graph.replay, steps)
            out["cuda_graph_capturable_adam_tf32_on"] = {"updates_per_s": 1e3 / ms, "ms_per_update": ms,
                                                         "launches_per_update": count_launches(graph.replay)}
            del graph
        except Exception as e:
            out["cuda_graph_capturable_adam_tf32_on"] = {"unavailable": f"{type(e).__name__}: {str(e)[:200]}"}
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
    out["note"] = "unmodified reference sources (baseline/_ref) on the same GPU, device-resident pre-collated batch, use_tb=False"
    return out


# ----------------------------------------------------------------------------- sub-records: the multi-GPU configurations
def sub_ensemble(args, rank, world, dev, K=8):
    """BASELINE configs[3]: K = 8 independent walker-shape agents per GPU (64 on 8 GPUs), no collective.  The
    one-GPU point (rank 0 alone, the other ranks idle) is measured in the same run."""
    from drqv2_b200 import AgentEnsemble
    A, Fd, B = 6, 50, 256
    ens = AgentEnsemble(K, (9, 84, 84), (A,), "cuda", 1e-4, Fd, args.hidden_dim, 0.01, 2000, 2, SCHED, 0.3, False,
                        seeds=[10_000 * rank + k for k in range(K)], use_cuda_graph=True, mode=args.mode)
    its = [ring_iter(f"/bench/ens{rank}_{k}", A, 8, B, dev, seed=77 + 100 * rank + k) for k in range(K)]
    step = [0]

    def one():
        ens.update(its, step[0])
        step[0] += 2
    for _ in range(4):
        one()
    steps = max(10, min(args.steps, 100))
    solo_ms = None
    if world > 1:                                    # one-GPU point: rank 0 runs while the others wait
        if rank == 0:
            solo_ms = statistics.median(m / steps for m in timed_blocks(one, [steps] * 3, 1, dev))
        torch.distributed.barrier()
    med, stats = block_stats(timed_blocks(one, [steps] * 3, world, dev), [steps] * 3, world * K)
    if solo_ms is None:
        solo_ms = med
    del ens, its
    return {"config": f"{world * K} independent agents (walker_walk shape, B=256), {K} per GPU on {world} GPU(s), no collective",
            "value": stats["value_median"], "unit": "updates/s (sum over agents)", "ms_per_step": med,
            "one_gpu_value": K * 1e3 / solo_ms, "efficiency_vs_one_gpu": stats["value_median"] / (world * K * 1e3 / solo_ms),
            "per_gpu": stats["value_median"] / world, "repeat": stats}


def sub_dp(args, rank, world, dev):
    """BASELINE configs[4]: humanoid shape (A=21, F=100), global batch 4096 sharded over the GPUs, NCCL gradient
    all-reduce inside the graph; the one-GPU B=4096 point is measured by rank 0 in the same run."""
    from drqv2_b200 import dist as D
    A, Fd, Bg = 21, 100, 4096
    steps = max(10, min(args.steps, 50))
    rec = {"config": f"humanoid_run shape (A=21, F=100, H={args.hidden_dim}), global batch {Bg} over {world} GPU(s)"}
    one_gpu = None
    if rank == 0:                                    # strong-scaling yardstick: the whole batch on one GPU
        agent = new_agent(args, A, Fd, seed=0)
        it = ring_iter("/bench/dp_one", A, 16, Bg, dev, seed=5)
        st = [0]

        def solo():
            agent.update(it, st[0])
            st[0] += 2
        for _ in range(3):
            solo()
        one_gpu = statistics.median(m / steps for m in timed_blocks(solo, [steps] * 3, 1, dev))
        del agent, it
        torch.cuda.empty_cache()
    rec["one_gpu_b4096"] = None if one_gpu is None else {"ms_per_step": one_gpu, "value": 1e3 / one_gpu}
    if world == 1:
        rec.update({"value": 1e3 / one_gpu, "unit": "global-batch updates/s", "ms_per_step": one_gpu})
        return rec
    torch.distributed.barrier()
    Bs = Bg // world
    torch.manual_seed(0)
    agent = new_agent(args, A, Fd, seed=0, dp=True)
    it = ring_iter(f"/bench/dp{rank}", A, 16, Bs, dev, seed=5 + rank)
    st = [0]

    def one():
        agent.update(it, st[0])
        st[0] += 2
    for _ in range(4):
        one()
    med, stats = block_stats(timed_blocks(one, [steps] * 3, world, dev), [steps] * 3, 1)
    a = agent._arena
    identical = D.replicas_identical([a.params, a.target, a.exp_avg, a.exp_avg_sq])
    # the same shard update without communication, and the collectives alone (eager, same tensors)
    torch.manual_seed(0)
    solo_agent = new_agent(args, A, Fd, seed=0)
    it2 = ring_iter(f"/bench/dp_nocomm{rank}", A, 16, Bs, dev, seed=5 + rank)

    def nocomm():
        solo_agent.update(it2, st[0])
        st[0] += 2
    for _ in range(4):
        nocomm()
    nc = statistics.median(m / steps for m in timed_blocks(nocomm, [steps] * 3, world, dev))
    ranges = {"critic": a._grads_full[a.seg["critic"][0]:a.seg["critic"][0] + a.seg["critic"][2]],
              "actor+metrics": a._grads_full[a.seg["actor"][0]:a.total + 8],
              "encoder": a._grads_full[a.seg["encoder"][0]:a.seg["encoder"][0] + a.seg["encoder"][2]]}
    ar = {}
    for name, t in ranges.items():
        t = t.clone()
        for _ in range(5):
            D.average_(t)
        ms = statistics.median(timed_blocks(lambda: D.average_(t), [20] * 3, world, dev)) / 20
        ar[name] = {"mbytes": t.numel() * 4 / 1e6, "us": ms * 1e3}
    rec.update({"value": 1e3 / med, "unit": "global-batch updates/s", "ms_per_step": med, "repeat": stats,
                "shard_batch": Bs, "ms_per_step_same_shard_no_communication": nc, "ratio_vs_no_communication": med / nc,
                "strong_scaling_efficiency_vs_one_gpu_b4096": None if one_gpu is None else (one_gpu / med) / world,
                "allreduce_alone": ar, "allreduce_us_per_step": sum(v["us"] for v in ar.values()),
                "dp_replicas_identical": bool(identical)})
    agent._graphs.clear()
    del agent, solo_agent
    return rec


def sub_act(args):
    """BASELINE configs[2]: act() = encoder + actor, quadruped shape (A=12), through the public API (host numpy in,
    host numpy out, as drqv2.py:164-175): latency at batch 1 (what train.py calls every environment step) and
    throughput at batch 1024 (the vectorised rollout / batched eval of drqv2_b200.loop)."""
    agent = new_agent(args, 12, 50, seed=0)
    rng = np.random.default_rng(0)
    rec = {"config": "quadruped_walk shape (A=12, F=50), exploration sample, host numpy -> host numpy"}
    for n, reps in ((1, 300), (1024, 20)):
        obs = rng.integers(0, 256, (n, 9, 84, 84) if n > 1 else (9, 84, 84), dtype=np.uint8)
        for _ in range(5):
            agent.act(obs, 5000, False)
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(reps):
            a = agent.act(obs, 5000, False)
        dt = (time.perf_counter() - t) / reps
        assert np.all(np.abs(a) <= 1.0)
        rec[f"batch_{n}"] = {"ms_per_call": dt * 1e3, "observations_per_s": n / dt}
    ref = _load_reference()
    if ref is not None:                              # the unmodified reference's act on the same GPU, batch 1
        torch.manual_seed(0)
        ragent = ref.DrQV2Agent((9, 84, 84), (12,), "cuda", 1e-4, 50, args.hidden_dim, 0.01, 2000, 2, SCHED, 0.3, False)
        obs = rng.integers(0, 256, (9, 84, 84), dtype=np.uint8)
        with torch.no_grad():
            for _ in range(10):
                ragent.act(obs, 5000, False)
            torch.cuda.synchronize()
            t = time.perf_counter()
            for _ in range(100):
                ragent.act(obs, 5000, False)
        rec["reference_on_gpu_batch_1_ms_per_call"] = (time.perf_counter() - t) / 100 * 1e3
    return rec


# ----------------------------------------------------------------------------- outputs of the timed path
DUMP_BYTES = 60 << 20     # array data; with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, agent, B):
    """Writes what the last timed update computed, as a caller of DrQV2Agent.update receives it: every parameter of
    the four networks (`<net>.<name>.npy`) and the 8 metrics (`metrics.npy`, in METRIC_KEYS order), float32.  Arrays
    stay whole while everything fits DUMP_BYTES; past that the largest are cut to a fixed seeded sample of their
    flattened elements (the same positions for the same size on every run), smallest arrays first."""
    from drqv2_b200.drqv2 import METRIC_KEYS
    m = agent.read_metrics(agent.workspace(B))
    arrays = {"metrics": np.array([m[k] for k in METRIC_KEYS], dtype=np.float32)}
    for net in ("encoder", "actor", "critic", "critic_target"):
        for name, p in getattr(agent, net).named_parameters():
            arrays[f"{net}.{name}"] = p.detach().float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    left, n = DUMP_BYTES // 4, len(arrays)
    for name, a in sorted(arrays.items(), key=lambda kv: kv[1].size):
        keep = left // n
        if a.size > keep:
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
        left, n = left - a.size, n - 1


# ----------------------------------------------------------------------------- main arm
def run_ours(args, rank, world):
    from drqv2_b200 import _lib
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    dp = args.parallel == "dp" and world > 1
    A, Fd, H = args.action_dim, args.feature_dim, args.hidden_dim
    B = args.batch // world if dp else args.batch  # dp: --batch is the global batch, sharded over the ranks
    if dp and args.batch % world:
        raise SystemExit(f"--batch {args.batch} does not split over {world} ranks")
    parity = parity_check(args) if (rank == 0 and not args.no_parity) else {}
    torch.manual_seed(0 if dp else rank)          # ensemble member = independent seed; dp = one agent
    np.random.seed(7 + rank)
    agent = new_agent(args, A, Fd, seed=0 if dp else rank, dp=dp)
    key = f"/bench/ring{rank}"
    it = ring_iter(key, A, args.episodes, B, dev, seed=1 + rank)
    K = 1 if dp else max(1, args.agents_per_gpu)
    # further ensemble members of this GPU: own parameters, optimiser state, ring, RNG stream, graph and CUDA stream
    members, member_its = [agent], [it]
    for k in range(1, K):
        torch.manual_seed(1000 * k + rank)
        members.append(new_agent(args, A, Fd, seed=1000 * k + rank))
        member_its.append(ring_iter(f"{key}_m{k}", A, args.episodes, B, dev, seed=1 + rank + 1000 * k))
    member_streams = [torch.cuda.Stream(device=dev) for _ in range(K)]

    def update_all(iters, step):
        """one update of every member of this GPU; returns member 0's metrics"""
        if K == 1:
            return agent.update(iters[0], step)
        cur = torch.cuda.current_stream()
        pending = []
        for ag, mit, st in zip(members, iters, member_streams):
            st.wait_stream(cur)
            with torch.cuda.stream(st):
                pending.append(ag.update_async(mit, step))
        m = dict()
        for ag, ws_, st in zip(members, pending, member_streams):
            if ag.use_tb:
                with torch.cuda.stream(st):
                    mk = ag.read_metrics(ws_)
                m = m or mk
            cur.wait_stream(st)
        return m

    # count kernel launches of one update (eager pass == what the graph replays): every C-ABI call of the
    # update goes through _lib.call; entry points that launch two kernels are listed below
    n_calls = [0]
    orig_call = _lib.call
    two_kernel_calls = ("drq_conv3x3_wgrad_bf16", "drq_conv1_wgrad_bf16", "drq_conv3x3_wgrad_f32", "drq_conv1_wgrad_f32")

    def counting_call(name, *a):
        # drq_ln_tanh_bwd launches its parameter-gradient kernel only when dgamma (argument 8) is given
        # the bf16 wgrad entry points skip their reduce kernel when dw (argument 4) is NULL (reduced by one launch later)
        two = ((name in two_kernel_calls and (not name.endswith("_bf16") or a[4])) or (name == "drq_ln_tanh_bwd" and a[8])
               or (name == "drq_conv1_wgrad_bf16_ring" and a[5]))
        if not name.startswith(("drq_set_", "drq_debug_")):          # host-side switches launch nothing
            n_calls[0] += 2 if two else 1
        return orig_call(name, *a)

    import drqv2_b200._bf16 as BF
    import drqv2_b200.drqv2 as D
    import drqv2_b200.replay_buffer as R
    step = [0]
    agent.update(it, step[0]); step[0] += 2             # eager warm-up
    D.call = R.call = BF.call = counting_call
    agent.use_cuda_graph = False
    agent.update(it, step[0]); step[0] += 2             # eager, counted
    agent.use_cuda_graph = True
    launches_per_update = n_calls[0]
    D.call = R.call = BF.call = orig_call

    def one_device_step():
        update_all(member_its, step[0])
        step[0] += 2
    W = max(args.warmup, 3)
    for _ in range(W):
        one_device_step()
    sampler = ClockSampler(dev.index)
    if rank == 0:                     # one nvidia-smi poller per job: NVML queries perturb the GPUs they touch, and in
        sampler.start()               # data-parallel mode a stall on any rank stalls every rank twice per update
    units = 1 if dp else world * K    # dp: global-batch updates/s; ensemble: sum over agents
    sizes = block_sizes(args.steps, args.blocks)
    ms_per_step, repeat = block_stats(timed_blocks(one_device_step, sizes, world, dev), sizes, units)
    value = units * 1e3 / ms_per_step
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, agent, B)

    # ---- e2e: public API fed from host batches (pinned), metrics read back.  prefetch: the agent pulls the next
    # host batch one update ahead and overlaps its H2D copy with the running update (a DrQV2Agent option)
    for ag in members:
        ag.use_tb = True
        ag.prefetch = True
    g = torch.Generator().manual_seed(100 + rank)
    nhost = 4
    host_batches = []
    for _ in range(nhost):
        host_batches.append(tuple(t.pin_memory() for t in (
            torch.randint(0, 256, (B, 9, 84, 84), dtype=torch.uint8, generator=g),
            torch.rand(B, A, generator=g) * 2 - 1, torch.rand(B, 1, generator=g),
            torch.full((B, 1), 0.970299065), torch.randint(0, 256, (B, 9, 84, 84), dtype=torch.uint8, generator=g))))

    def host_iter():
        i = 0
        while True:
            yield host_batches[i % nhost]
            i += 1

    hits = [host_iter() for _ in range(K)]
    last = [None]

    def one_host_step():
        last[0] = update_all(hits, step[0])
        step[0] += 2
    for _ in range(4):
        one_host_step()
    e2e_ms, e2e_repeat = block_stats(timed_blocks(one_host_step, sizes, world, dev), sizes, units)
    clocks = sampler.stop()
    e2e_value = units * 1e3 / e2e_ms
    h2d = K * (sum(t.numel() * t.element_size() for t in host_batches[0]) + 4 * 32)
    d2h = K * 8 * 4
    assert np.isfinite(last[0]["critic_loss"])
    for ag in members:
        ag.use_tb = False
        ag.prefetch = False

    extra = {}
    if rank == 0:
        launches = profile_update_launches(agent, it, B) if not args.no_kernels else []
        roof = roofline_record(launches, value, world, update_flops(B, A, Fd, H) * (world if dp else 1), args.mode) if launches else None
        if roof and roof.get("kernel") == "conv3x3_fwd" and not dp and K == 1:
            # the dominant kernel's launches where the metric is measured: inside the captured graph the timed region replays
            got = in_graph_run_time(agent, it, "drq_conv3x3_fwd_bf16")
            if got and got[1] == len(roof["kernel_launches"]):
                us_run, n_run = got
                fl = sum(l["flop"] for l in launches if l["kernel"].startswith("conv3x3_fwd"))
                ach = fl / (us_run * 1e-6) / 1e12
                roof["eager_in_sequence"] = {"achieved": roof["achieved"], "frac": roof["frac"], "kernel_us": roof["kernel_us"],
                                             "measured": roof.get("measured")}
                roof.update({"achieved": ach, "frac": ach / roof["peak"], "kernel_us": us_run / n_run,
                             "measured": "the %d consecutive launches of this kernel INSIDE the captured update graph (the graph the "
                                         "timed region replays): two CUDA event-record nodes around the run, their distance read after "
                                         "each of 20 replays, median; the run follows conv1 as in every update, nothing is flushed" % n_run})
    for ag in members[1:]:
        ag._graphs.clear()
    del members[1:], member_its[1:]
    torch.cuda.empty_cache()
    if not args.no_subrecords and not dp and K == 1 and args.mode == "bf16":
        extra["ensemble_8_per_gpu"] = sub_ensemble(args, rank, world, dev)
        torch.cuda.empty_cache()
        extra["dp_humanoid_b4096"] = sub_dp(args, rank, world, dev)
        torch.cuda.empty_cache()
    out = None
    if rank == 0:
        if not args.no_subrecords and args.mode == "bf16" and world == 1:   # a one-GPU path: measured in the N=1 run
            extra["act_quadruped"] = sub_act(args)
        gref = gpu_reference(args) if not args.no_gpu_reference else None
        cpu = cpu_baseline(args, steps=5)
        out = {"metric": "DrQ-v2 updates/sec at batch 256", "value": value, "unit": "updates/s", "n_gpus": world,
               "steps": args.steps, "warmup": W, "ms_per_step": ms_per_step,
               "higher_is_better": True, "scaling": "strong" if dp else "weak", "vs_baseline": None,
               "dtype": "bf16" if args.mode == "bf16" else "f32",
               "data": "synthetic",
               "config": {"workload": f"configs[1]: walker_walk-shape agent.update, B={B}, 9x84x84 u8 stacks, A={A}, "
                                      f"F={Fd}, H={H}, n-step 3, GPU-resident replay ring ({args.episodes} episodes x 501 "
                                      f"rows), CUDA-graphed, {'bf16 tensor-core mode (fp32 master weights, fp32 accumulation)' if args.mode == 'bf16' else 'fp32 parity mode'}" + (f"; global batch {args.batch} data-parallel over {world} GPUs (NCCL gradient all-reduce in the graph)" if dp else (f"; {world * K} independent agents (ensemble), {K} per GPU on their own streams, no collective" if world * K > 1 else "")),
                          "l2": "inputs larger than L2: each step gathers a fresh 32.5 MB batch from a "
                                f"{args.episodes * 501 * 21168 / 1e6:.0f} MB ring and streams ~700 MB of activations",
                          "timed_blocks": f"{args.steps} steps in {len(sizes)} blocks; value / ms_per_step = the median block",
                          "mode": args.mode, "agents_per_gpu": K},
               "repeat": repeat,
               "e2e": {"value": e2e_value, "unit": "updates/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                       "repeat": e2e_repeat},
               "gpu_launches": launches_per_update * args.steps * K, "launches_per_update": launches_per_update,
               "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "gpu_reference": gref}
        out.update(parity)
        out.update(extra)
    return out


def _load_reference():
    """The unmodified reference modules from baseline/_ref (baseline/install_ref.py), or None."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref, "drqv2.py")):
        return None
    import types
    for name in ("hydra", "omegaconf"):                     # imported by the reference, unused on this path
        sys.modules.setdefault(name, types.ModuleType(name))
    if not hasattr(sys.modules["omegaconf"], "OmegaConf"):
        sys.modules["omegaconf"].OmegaConf = object
    import importlib.util
    mods = {}
    for name in ("utils", "drqv2"):
        spec = importlib.util.spec_from_file_location(f"_ref_{name}", os.path.join(ref, f"{name}.py"))
        m = importlib.util.module_from_spec(spec)
        if name == "drqv2":
            saved = sys.modules.get("utils")
            sys.modules["utils"] = mods["utils"]            # the reference's `import utils`
            try:
                spec.loader.exec_module(m)
            finally:
                if saved is None:
                    sys.modules.pop("utils", None)
                else:
                    sys.modules["utils"] = saved
        else:
            spec.loader.exec_module(m)
        mods[name] = m
    return mods["drqv2"]


def cpu_baseline(args, steps=5, warm=1):
    """The reference's own agent.update (unmodified sources in baseline/_ref, device 'cpu', all host
    threads) on a bounded sample: `steps` updates of the same B=256 workload from pre-collated tensors.
    Falls back to the oracle port of the same path when the reference sources are not present."""
    torch.set_num_threads(os.cpu_count())
    B, A, Fd, H = args.batch, args.action_dim, args.feature_dim, args.hidden_dim
    ref = _load_reference()
    if ref is not None:
        torch.manual_seed(0)
        agent = ref.DrQV2Agent((9, 84, 84), (A,), "cpu", 1e-4, Fd, H, 0.01, 2000, 2, SCHED, 0.3, False)
        g = torch.Generator().manual_seed(1)
        batch = (torch.randint(0, 256, (B, 9, 84, 84), dtype=torch.uint8, generator=g),
                 torch.rand(B, A, generator=g) * 2 - 1, torch.rand(B, 1, generator=g),
                 torch.full((B, 1), 0.970299065), torch.randint(0, 256, (B, 9, 84, 84), dtype=torch.uint8, generator=g))

        def it():
            while True:
                yield batch
        ri = it()
        for i in range(warm):
            agent.update(ri, 2 * i)
        t = time.perf_counter()
        for i in range(steps):
            agent.update(ri, 2 * (i + warm))
        dt = (time.perf_counter() - t) / steps
        return {"value": 1.0 / dt, "unit": "updates/s", "cores": torch.get_num_threads(), "kind": "reference",
                "sample": f"{steps} updates (after {warm} warm-up) of the reference's DrQV2Agent.update on CPU, B={B}, "
                          "pre-collated synthetic tensors"}
    from oracle import drq_oracle as O
    params = O.synthetic_params(9, A, Fd, H, seed=0)
    agent = O.OracleAgent(params, 1e-4, 0.01, SCHED, 0.3, dtype=torch.float32, aug="grid")
    b = O.synthetic_batch(B, A, seed=1)
    a = (b["obs"], b["action"], b["reward"], b["discount"], b["next_obs"])
    k = (b["shift_obs"], b["shift_next"], b["eps_critic"], b["eps_actor"])
    for i in range(warm):
        agent.update(*a, 2 * i, *k)
    t = time.perf_counter()
    for i in range(steps):
        agent.update(*a, 2 * (i + warm), *k)
    dt = (time.perf_counter() - t) / steps
    return {"value": 1.0 / dt, "unit": "updates/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{steps} updates (after {warm} warm-up) of the same B={B} workload, pre-collated tensors, "
                      "float grid_sample aug as the reference ships it"}


def run_reference(args, rank, world):
    if rank != 0:
        return None
    steps = args.steps
    warm = max(1, min(args.warmup, 3))
    cpu = cpu_baseline(args, steps=steps, warm=warm)
    B, A, Fd, H = args.batch, args.action_dim, args.feature_dim, args.hidden_dim
    return {"impl": "reference", "metric": "DrQ-v2 updates/sec at batch 256", "value": cpu["value"],
            "unit": "updates/s", "n_gpus": world, "steps": steps, "warmup": warm,
            "ms_per_step": 1e3 / cpu["value"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"configs[0]: reference's CPU update path ({cpu['kind']}, torch CPU), B={B}, A={A}, "
                                   f"F={Fd}, H={H}"},
            "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed updates (default 1000; --impl reference: 40, its CPU update takes ~0.25 s)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--blocks", type=int, default=5,
                    help="the --steps timed updates are split into this many blocks; value = median block")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--action-dim", type=int, default=6)
    ap.add_argument("--feature-dim", type=int, default=50)
    ap.add_argument("--hidden-dim", type=int, default=1024)
    ap.add_argument("--episodes", type=int, default=64)
    ap.add_argument("--mode", default="bf16", choices=["fp32", "bf16"])
    ap.add_argument("--agents-per-gpu", type=int, default=1,
                    help="ensemble members per GPU (BASELINE configs[3] uses 8): independent agents replayed on their own "
                         "streams; value = updates/s summed over all members of all GPUs")
    ap.add_argument("--parallel", default="ensemble", choices=["ensemble", "dp"],
                    help="N > 1: independent agents per GPU (weak scaling, no collective) or one agent with the "
                         "global --batch sharded over the GPUs and NCCL gradient all-reduce (strong scaling)")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of the first updates")
    ap.add_argument("--no-kernels", action="store_true", help="skip the per-launch roofline timings")
    ap.add_argument("--no-subrecords", action="store_true", help="skip ensemble_8_per_gpu / dp_humanoid_b4096")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip the reference-on-GPU baseline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the parameters and metrics the last timed update computed "
                         "(rank 0, ensemble member 0) as DIR/<name>.npy, float32, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 40 if args.impl == "reference" else 1000
    if args.steps < 1 or args.blocks < 1:
        ap.error("--steps and --blocks must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        out = run_reference(args, rank, world)
        if out is not None:
            print(json.dumps(out), flush=True)
        return
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"              # rank 0's stdout carries exactly one JSON line
        if int(os.environ.get("DRQV2_B200_DP_RESERVE_SMS", "0")) > 0:   # opt-in: cap NCCL to the SMs the persistent kernels leave
            os.environ.setdefault("NCCL_MAX_CTAS", os.environ["DRQV2_B200_DP_RESERVE_SMS"])
        local = int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(local)
        kw = {}
        if os.environ.get("DRQV2_B200_NCCL_HIPRIO", "0") != "0":
            # the collectives captured into the update graph then run at the highest stream priority: their CTAs are
            # placed before the persistent conv kernels' when both are waiting for SMs
            opts = torch.distributed.ProcessGroupNCCL.Options()
            opts.is_high_priority_stream = True
            kw["pg_options"] = opts
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local), **kw)
    out = run_ours(args, rank, world)
    if out is not None:
        print(json.dumps(out), flush=True)
    if world > 1:
        # graphs holding captured NCCL kernels were dropped with the agent (run_ours returned); a teardown
        # that still blocks must not hold the job: force-exit after a grace period
        import gc
        gc.collect()
        torch.cuda.synchronize()
        threading.Timer(20.0, lambda: os._exit(0)).start()
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
        os._exit(0)


if __name__ == "__main__":
    main()
