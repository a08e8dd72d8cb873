"""KernelSHAP over time-frequency cells at the C2 shape (wav2vec2-base, one 5 s clip, 2048 coalitions, per-character
log-probabilities): time-only coalitions against (segment, band) cells.

    python tools/bench_bands.py [--configs 100x1 25x4 50x8] [--steps 3] [--rounds 3] [--out FILE.json]

A config MxF is M time segments and F mel bands (F = 1: the time-only path bench.py times, no bands set).  For every
config it reports, from CUDA-event-timed eval_bits calls of all 2050 coalitions (the explainer's matrix: empty, full and
the 2048 sampled ones), the configs alternated round by round within this one process:
  coalitions_per_s      median over the rounds
  conv0_ms_per_tile / conv0_stats_ms_per_tile   those launches' time per batch tile (w2s_profile, a separate eager run)
  s_per_clip            one whole KernelShapExplainer.explain call (targets, evaluation, device solve), host clock
The GPU name and power limit are read in the same run and written beside the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from shap_transformer_asr_b200 import (MODELS, WORKLOADS, Engine, KernelShapExplainer, band_components, char_targets,  # noqa: E402
                                       mel_band_edges, sample_coalitions, synthetic_clip)
from shap_transformer_asr_b200.modelzoo import build_random_init_model  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["100x1", "25x4", "50x8"])
    ap.add_argument("--steps", type=int, default=3, help="eval_bits calls per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="timed windows per config, configs alternated")
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    args = ap.parse_args()
    wl = WORKLOADS["C2"]
    cfg = MODELS[wl.model]
    model = build_random_init_model(cfg, seed=0)
    clip = synthetic_clip(wl.num_samples)
    K = wl.num_coalitions
    eng = Engine(model, cfg, max_batch=0)
    eng.set_clip(clip, num_segments=wl.num_segments)
    eng.set_targets("logits")
    ones = np.ones((1, wl.num_segments), np.uint8)
    logits = eng.eval_bits(eng.bits_to_device(ones)).view(-1, cfg.vocab_size).cpu().numpy()
    frames, tokens = char_targets(logits)
    eng.set_targets("logprob", frames, tokens)

    configs = []
    for c in args.configs:
        M, F = (int(v) for v in c.split("x"))
        Z, _, _ = sample_coalitions(M * F, K, seed=0)
        Z = np.concatenate([np.zeros((1, M * F), np.uint8), np.ones((1, M * F), np.uint8), Z])
        comp = band_components(clip, mel_band_edges(F)) if F > 1 else None
        configs.append(dict(name=c, M=M, F=F, Z=Z, comp=comp, bits=None, times=[]))

    def select(c):
        eng.clear_bands()
        eng.set_clip(clip, num_segments=c["M"])
        if c["comp"] is not None:
            eng.set_bands(c["comp"])
        if c["bits"] is None:
            c["bits"] = eng.bits_to_device(c["Z"]).clone()

    for c in configs:                                     # warm-up: plans, graph capture
        select(c)
        eng.eval_bits(c["bits"])
    torch.cuda.synchronize()
    for _ in range(args.rounds):
        for c in configs:
            select(c)
            eng.eval_bits(c["bits"])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                eng.eval_bits(c["bits"])
            e1.record()
            torch.cuda.synchronize()
            c["times"].append(e0.elapsed_time(e1) / 1e3 / args.steps)

    results = []
    for c in configs:
        select(c)
        eng.profile(True)
        eng.eval_bits(c["bits"])
        torch.cuda.synchronize()
        prof = eng.profile_read()
        eng.profile(False)
        per_tile = {k: prof[k]["ms"] / prof[k]["launches"] for k in ("conv0", "conv0_stats") if k in prof}
        eng.clear_bands()
        ex = KernelShapExplainer(eng, nsamples=K, seed=0)
        edges = mel_band_edges(c["F"]) if c["F"] > 1 else None
        ex.explain(clip, num_segments=c["M"], targets=(frames, tokens), band_edges=edges)    # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = ex.explain(clip, num_segments=c["M"], targets=(frames, tokens), band_edges=edges)
        torch.cuda.synchronize()
        s_clip = time.perf_counter() - t0
        n = c["Z"].shape[0]
        s = float(np.median(c["times"]))
        r = dict(config=c["name"], segments=c["M"], bands=c["F"], features=c["M"] * c["F"], coalitions=n,
                 s_per_eval=s, coalitions_per_s=n / s, coalitions_per_s_rounds=[n / t for t in c["times"]],
                 conv0_ms_per_tile=per_tile.get("conv0"), conv0_stats_ms_per_tile=per_tile.get("conv0_stats"),
                 s_per_clip=s_clip, status=int(res["status"].item()))
        print(json.dumps(r))
        results.append(r)
    base = results[0]["coalitions_per_s"]
    for r in results:
        r["rate_vs_first"] = r["coalitions_per_s"] / base
    out = dict(workload="C2", model=wl.model, num_samples=wl.num_samples, targets=len(frames),
               batch_tile=eng.kernel_count()[1], steps=args.steps, rounds=args.rounds, gpu=gpu_info(), results=results)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))
    eng.close()


if __name__ == "__main__":
    main()
