#!/usr/bin/env python
"""bench.py -- masked-coalition Wav2Vec2 forwards/sec on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C2] [--impl reference] [--dump-outputs DIR]

A "step" = one pass of the hot path over one batch of synthetic input: every coalition of the workload
(C2: 2048 coalitions of one 5 s clip, 100 segments) through mask -> Wav2Vec2 -> per-character CTC
log-probabilities.  N > 1 (torchrun, one rank per GPU): coalitions are independent, so every rank
evaluates its own full set (weak scaling, no data-path collective) and the ranks exchange only the
single all-gather of the per-coalition output rows.  Rank 0 prints ONE JSON line.

`--impl reference` times the reference's own CPU implementation of the path (the `transformers`
fp32 forward the reference calls, shap_calculation.py:42, behind a restated callback) on the host
cores with a bounded sample per step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "masked_coalition_forwards_per_sec"
UNIT = "coalition-forwards/s"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], source="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


def ncu_traffic(workload):
    """DRAM bytes per launch of the dominant kernel.  NOT measured in this run: read from the committed summary of an
    `ncu --set full` capture of the same command (profiles/), and labelled as such in the line; None if absent."""
    for name in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if workload == "C2" and os.path.exists(p):
            d = json.load(open(p))
            return d["mean_traffic_bytes_per_launch"], {
                "dram_bytes_per_launch": d["mean_traffic_bytes_per_launch"],
                "algorithmic_bytes_per_launch": d["mean_algorithmic_bytes_per_launch"],
                "source": f"committed ncu file profiles/{name} (not captured in this run)"}
    return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def build_problem(workload_name):
    from shap_transformer_asr_b200 import MODELS, WORKLOADS, sample_coalitions, synthetic_clip
    wl = WORKLOADS[workload_name]
    cfg = MODELS[wl.model]
    clip = synthetic_clip(wl.num_samples)
    Z, kw, info = sample_coalitions(wl.num_segments, wl.num_coalitions, seed=0)
    return wl, cfg, clip, Z, kw


def make_hf_model(cfg):
    from shap_transformer_asr_b200.modelzoo import build_random_init_model   # random-init weights of the named arch
    return build_random_init_model(cfg, seed=0)


def clip_targets(model, clip):
    """Per-character (frame, token) targets of the unmasked clip, from the fp32 forward of `model` on the host.  Random-init
    logits are nearly flat (on C2 about one frame in ten has its top-2 margin inside the bf16 error of the device path), so
    targets taken from the build under test would differ between builds; these do not.  -> (logits, frames, tokens)"""
    from shap_transformer_asr_b200 import char_targets
    with torch.no_grad():
        lg = model(torch.from_numpy(clip)[None]).logits[0].numpy()
    frames, tokens = char_targets(lg)
    return lg, frames, tokens


DUMP_LIMIT = 60 << 20          # data bytes of a --dump-outputs file: with its header, under 64 MB


def dump_outputs(path, name, a):
    """Write `a` as <path>/<name>.npy in float32; above DUMP_LIMIT bytes, a fixed seeded sample of its rows."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.nbytes > DUMP_LIMIT:
        rows = DUMP_LIMIT // a[:1].nbytes
        a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], rows, replace=False))]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, name + ".npy"), a)


def cpu_reference_rate(model, cfg, clip, Z, bounds, frames, tokens, n_rows, batch=32, threads=None):
    """forwards/s of the reference's CPU path: transformers fp32 forward on masked waveforms -> log_softmax -> gather."""
    from oracle import callback as CB
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    f = torch.as_tensor(frames, dtype=torch.long)
    t = torch.as_tensor(tokens, dtype=torch.long)

    def run(rows):
        X = torch.from_numpy(CB.materialize(clip, rows, bounds))
        with torch.no_grad():
            lg = model(X, attention_mask=torch.ones_like(X)).logits        # shap_calculation.py:39-42
            return torch.log_softmax(lg, -1)[:, f, t]

    run(Z[:min(batch, 4)])                                                  # warm-up excluded
    t0 = time.perf_counter()
    done = 0
    outs = []
    while done < n_rows:
        outs.append(run(Z[done:min(done + batch, n_rows)]))
        done += min(batch, n_rows - done)
    dt = time.perf_counter() - t0
    cpu_reference_rate.last_outputs = torch.cat(outs).numpy()               # kept for the parity check of the bench line
    return done / dt, done, dt, threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl, cfg, clip, Z, kw = build_problem(args.workload)
    from oracle import callback as CB
    model = make_hf_model(cfg)
    bounds = CB.segment_bounds(wl.num_samples, wl.num_segments)
    _, frames, tokens = clip_targets(model, clip)
    threads = os.cpu_count() or 1
    # bounded sample per step: calibrate on 8 rows so that warmup+steps finish within a few minutes
    r0, _, dt0, _ = cpu_reference_rate(model, cfg, clip, Z, bounds, frames, tokens, 8, batch=8, threads=threads)
    budget = 150.0 / max(1, args.steps + args.warmup)
    n_rows = int(max(8, min(wl.num_coalitions, (r0 * budget) // 8 * 8)))
    times = []
    for i in range(args.warmup + args.steps):
        r, done, dt, _ = cpu_reference_rate(model, cfg, clip, Z, bounds, frames, tokens, n_rows, batch=32, threads=threads)
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "logprobs", cpu_reference_rate.last_outputs)
    total = sum(times)
    value = n_rows * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{wl.name}: {wl.description}", "sample_per_step": n_rows, "batch": 32},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "reference",
                         "sample": f"{n_rows} of {wl.num_coalitions} coalitions per step; transformers "
                                   f"{__import__('transformers').__version__} fp32 forward + log_softmax + gather, batch 32"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_b200(args):
    import torch.distributed as td
    from shap_transformer_asr_b200 import CoalitionCallback, Engine, dist as wdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, world = wdist.init_from_env("cuda") if world > 1 else (0, 1)
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    peaks = load_peaks()

    wl, cfg, clip, Z, kw = build_problem(args.workload)
    if args.coalitions > 0:
        Z, kw = Z[:args.coalitions], kw[:args.coalitions]
    model = make_hf_model(cfg)
    # batch tile: rows = B * T' should fill whole waves of 128-row tiles on 148 SMs (B = floor(148*128*k / T'))
    # (the library picks B = floor(148*128*k / T') with B >= 128 itself when max_batch is 0)
    eng = Engine(model, cfg, device=local, max_batch=max(0, args.batch), preln_fp32=args.preln_fp32,
                 graphs=not args.no_graph)
    eng.set_clip(clip, num_segments=wl.num_segments)
    # targets: per-character frames of the unmasked clip (all frames if the random-init transcript is empty)
    lg, frames, tokens = clip_targets(model, clip)
    eng.set_targets("logprob", frames, tokens)
    D = len(frames)
    K = Z.shape[0]
    bits = eng.bits_to_device(Z)
    out = torch.empty((K, D), dtype=torch.float32, device=dev)
    gathered = torch.empty((world * K, D), dtype=torch.float32, device=dev) if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def step():
        flush.fill_(1)                                                   # L2 flush between iterations (timed, ~0.1 ms)
        eng.eval_bits(bits, out)
        if world > 1:
            td.all_gather_into_tensor(gathered, out)                     # the path's single exchange

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        td.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    launches0 = eng.launch_count()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    launches = eng.launch_count() - launches0                            # counted inside the library at launch time
    if args.dump_outputs and rank == 0:                                  # the rows the last timed step handed back
        dump_outputs(args.dump_outputs, "logprobs", (gathered if world > 1 else out).cpu().numpy())
    if world > 1:
        td.barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms], device=dev)
        td.all_reduce(t, op=td.ReduceOp.MAX)
        ms = float(t.item())

    # ---- strong scaling, the split north_star names: ONE clip's K coalitions sharded over the ranks (rank r evaluates
    #      rows [r K/G, (r+1) K/G)), then the single all-gather of the output rows; same timing discipline ----
    lo, hi = wdist.shard_range(K, rank, world)
    per = (K + world - 1) // world
    shard_out = torch.zeros((per, D), dtype=torch.float32, device=dev)
    strong_all = torch.empty((world * per, D), dtype=torch.float32, device=dev) if world > 1 else None

    def strong_step():
        flush.fill_(1)
        if hi > lo:
            eng.eval_bits(bits[lo:hi], shard_out[:hi - lo])
        if world > 1:
            td.all_gather_into_tensor(strong_all, shard_out)

    for _ in range(args.warmup):
        strong_step()
    torch.cuda.synchronize()
    if world > 1:
        td.barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(args.steps):
        strong_step()
    s1.record()
    torch.cuda.synchronize()
    if world > 1:
        td.barrier()
    strong_ms = s0.elapsed_time(s1)
    if world > 1:
        t = torch.tensor([strong_ms], device=dev)
        td.all_reduce(t, op=td.ReduceOp.MAX)
        strong_ms = float(t.item())
        # the sharded outputs are the rows of the full evaluation (same kernels, other tile boundaries)
        assert torch.equal(strong_all[:K], gathered[rank * K:(rank + 1) * K]) or \
            (strong_all[:K] - gathered[rank * K:(rank + 1) * K]).abs().max().item() < 1e-3
    # ---- per-launch CUDA-event profile of the same K steps (events between launches cost ~3 us each, so this pass is
    #      kept out of the headline timing; the roofline numbers below come from it) ----
    eng.profile(True)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(args.steps):
        step()
    p1.record()
    torch.cuda.synchronize()
    prof = eng.profile_read()
    eng.profile(False)
    prof_ms = p0.elapsed_time(p1)
    value = world * K * args.steps / (ms / 1e3)

    # ---- e2e: the public callable with HOST buffers (pinned H2D of the coalition matrix, D2H of the outputs) ----
    cb = CoalitionCallback(eng)
    cb(Z[:64])
    torch.cuda.synchronize()
    if world > 1:
        td.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        y_host = cb(Z)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        td.all_reduce(t, op=td.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e = world * K * args.steps / e2e_s

    # ---- seconds per explained clip: sampler + target selection + all coalitions + all-gather + device WLS, end to end ----
    from shap_transformer_asr_b200 import KernelShapExplainer
    ex = KernelShapExplainer(eng, nsamples=wl.num_coalitions, seed=0)
    ex.explain(clip, num_segments=wl.num_segments)            # warm-up (plans for the sharded row counts)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = ex.explain(clip, num_segments=wl.num_segments)
    torch.cuda.synchronize()
    sec_per_clip = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([sec_per_clip], device=dev, dtype=torch.float64)
        td.all_reduce(t, op=td.ReduceOp.MAX)
        sec_per_clip = float(t.item())
    wls_status = int(res["status"].item())
    eng.set_clip(clip, num_segments=wl.num_segments)
    eng.set_targets("logprob", frames, tokens)

    if rank != 0:
        td.destroy_process_group()
        return
    # ---- roofline of the dominant kernel (the tcgen05 contraction kernel), from the live event profile ----
    # the dominant kernel FAMILY: every launch of the tcgen05 contraction kernels (gemm_tc2_kernel / gemm_tc_kernel /
    # posconv_kernel).  conv0 (mma.sync, HBM-bound), attention and the depthwise conv carry FLOPs too but are other
    # kernels with their own rows in kernel_breakdown.
    not_family = ("conv0", "attention", "depthwise")
    fam = {k: v for k, v in prof.items() if v["flops"] > 0 and k not in not_family}
    gemm_ms = sum(v["ms"] for v in fam.values())
    gemm_fl = sum(v["flops"] for v in fam.values())
    gemm_n = sum(v["launches"] for v in fam.values())
    total_prof_ms = sum(v["ms"] for v in prof.values())
    achieved = gemm_fl / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    launches_per_batch, tile = eng.kernel_count()
    traffic, traffic_detail = ncu_traffic(wl.name)
    n_batches = (K + tile - 1) // tile
    flops_fwd = eng.flops_per_forward()
    # every launch class with its own roofline number: tensor-bound classes against the sustained bf16 peak, the others
    # against the measured HBM copy bandwidth (conv0 carries both: it is bound by its output stream)
    breakdown = {}
    for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
        tf = (v["flops"] / (v["ms"] / 1e3) / 1e12) if v["flops"] and v["ms"] > 0 else None
        gb = (v["bytes"] / (v["ms"] / 1e3) / 1e9) if v["bytes"] and v["ms"] > 0 else None
        hbm_bound = gb is not None and (tf is None or k in ("conv0", "depthwise"))
        breakdown[k] = {"ms_per_step": v["ms"] / args.steps, "share": v["ms"] / total_prof_ms, "launches": v["launches"],
                        "tflops": tf, "gbs": gb, "bound": "hbm" if hbm_bound else "tensor",
                        "frac_of_peak": (gb / peaks["hbm"]) if hbm_bound else (tf / peaks["tf_sustained"] if tf else None)}

    # ---- CPU baseline on this box's host cores: bounded sample of the same workload ----
    cpu, parity = None, None
    if world == 1 and not args.no_cpu:
        from oracle import callback as CB
        bounds = CB.segment_bounds(wl.num_samples, wl.num_segments)
        r0, _, _, threads = cpu_reference_rate(model, cfg, clip, Z, bounds, frames, tokens, 8, batch=8)
        n_rows = int(max(16, min(K, (r0 * 20.0) // 8 * 8)))
        r, done, dt, threads = cpu_reference_rate(model, cfg, clip, Z, bounds, frames, tokens, n_rows, batch=32)
        cpu = {"value": r, "unit": UNIT, "cores": threads, "kind": "reference",
               "sample": f"{done} of {K} coalitions in {dt:.1f} s; transformers fp32 forward + log_softmax + gather, batch 32"}
        # the same rows as evaluated by the B200 path in the timed steps (first `done` rows of `out`), checked against
        # the CPU result -- the reference as checker only
        ref_rows = cpu_reference_rate.last_outputs
        gpu_rows = out[:done].cpu().numpy()
        tol = 0.025 * float(np.abs(lg).max())
        parity = {"rows": int(done), "outputs_per_row": int(D), "max_abs_err": float(np.abs(gpu_rows - ref_rows).max()),
                  "tolerance": tol, "what": "per-character log-probabilities, B200 path vs transformers fp32 on the same coalitions",
                  "ok": bool(np.abs(gpu_rows - ref_rows).max() < tol)}
        if not parity["ok"]:
            raise SystemExit(f"bench.py: parity check failed: {parity}")

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        # one clip's coalitions sharded over the N ranks + the all-gather (north_star's split), timed like `value`;
        # efficiency = what N ranks achieve on one clip / (N x what one rank achieves on the same clip, measured by the
        # weak leg of this very run, where every rank evaluates the full set)
        "strong": {"forwards_per_s": K * args.steps / (strong_ms / 1e3), "ms_per_clip_forward_part": strong_ms / args.steps,
                   "rows_per_rank": int(per), "efficiency_vs_n1": (ms / world) / strong_ms},
        "parity": parity,
        "config": {"workload": f"{wl.name}: {wl.description}", "coalitions_per_step_per_gpu": K, "outputs_per_coalition": D,
                   "batch_tile": tile, "gflop_per_forward": flops_fwd / 1e9,
                   "l2": "256 MB flush write between steps; per-step activation stream >> 126 MB L2",
                   "weights": "random-init (seed 0)", "sec_per_clip_forward_part": ms / args.steps / 1e3,
                   "sec_per_explained_clip": sec_per_clip, "sec_per_explained_clip_note":
                   f"KernelShapExplainer.explain on {world} GPU(s): host sampler + target selection + {K} coalitions sharded over ranks "
                   f"+ all-gather + device WLS (status {wls_status})"},
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(cb.h2d_bytes), "d2h_bytes_per_step": int(cb.d2h_bytes)},
        "gpu_launches": int(launches),
        "gpu_launches_note": f"counted by the library at launch time over the {args.steps} timed steps ({n_batches} tiles x "
                             f"{launches_per_batch} kernels per step; each tile's plan is replayed as one CUDA graph)",
        "roofline": {"bound": "tensor", "kernel": "gemm_tc2_kernel<256> and the other contraction launches (gemm_tc_kernel, posconv_kernel)", "achieved": achieved,
                     "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": achieved / peaks["tf_sustained"],
                     "traffic": traffic, "traffic_detail": traffic_detail,
                     "peak_source": peaks["source"] + " bf16_tflops_sustained",
                     "launches": int(gemm_n), "share_of_step": gemm_ms / total_prof_ms,
                     "profiled_ms_per_step": prof_ms / args.steps,
                     "whole_step_tflops": value * flops_fwd / 1e12 / world,
                     "whole_step_frac": value * flops_fwd / 1e12 / world / peaks["tf_sustained"]},
        "cpu_baseline": cpu,
        "kernel_breakdown": breakdown,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        td.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="C2")
    ap.add_argument("--batch", type=int, default=0, help="coalitions per batch tile (0 = fill whole waves)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--coalitions", type=int, default=0, help="profiling aid: evaluate only the first N coalitions per step")
    ap.add_argument("--preln-fp32", action="store_true", help="A/B: fp32 pre-LayerNorm tensors (W2S_FLAG_FP32_PRELN)")
    ap.add_argument("--no-graph", action="store_true", help="A/B: launch every kernel of a tile instead of replaying a graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        run_reference(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    run_b200(args)


if __name__ == "__main__":
    main()
