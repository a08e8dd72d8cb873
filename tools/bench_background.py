"""KernelSHAP against a background dataset at the C2 shape (wav2vec2-base, one 5 s clip, 100 segments, 2048 coalitions,
per-character log-probabilities), for B background rows.

    python tools/bench_background.py [--rows 0 1 5 10] [--steps 3] [--out FILE.json]

For every B (0 = the zero fill bench.py times) it reports, from CUDA-event-timed eval_bits calls of all 2050 coalitions
(the explainer's matrix: empty, full and the 2048 sampled ones):
  row_forwards_per_s    coalitions * B rows evaluated per second (the zero fill's coalition-forwards/s when B = 0)
  coalitions_per_s      coalitions reported per second
  s_per_clip            one whole KernelShapExplainer.explain call (targets, evaluation, device solve), host clock
  bg_mean_ms            time of bg_mean_kernel in one call (w2s_profile, a separate eager run)
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
from shap_transformer_asr_b200 import (MODELS, WORKLOADS, Engine, KernelShapExplainer, char_targets, make_background,  # noqa: E402
                                       sample_coalitions, synthetic_clip)
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
    ap.add_argument("--rows", type=int, nargs="+", default=[0, 1, 5, 10])
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    args = ap.parse_args()
    wl = WORKLOADS["C2"]
    cfg = MODELS[wl.model]
    model = build_random_init_model(cfg, seed=0)
    clip = synthetic_clip(wl.num_samples)
    M, K = wl.num_segments, wl.num_coalitions
    eng = Engine(model, cfg, max_batch=0)
    eng.set_clip(clip, num_segments=M)
    eng.set_targets("logits")
    logits = eng.eval_bits(eng.bits_to_device(np.ones((1, M), np.uint8))).view(-1, cfg.vocab_size).cpu().numpy()
    frames, tokens = char_targets(logits)
    eng.set_targets("logprob", frames, tokens)
    Z, _, _ = sample_coalitions(M, K, seed=0)
    Z = np.concatenate([np.zeros((1, M), np.uint8), np.ones((1, M), np.uint8), Z])
    bits = eng.bits_to_device(Z).clone()
    n = Z.shape[0]
    results = []
    for B in args.rows:
        if B:
            eng.set_background(make_background(wl.num_samples, B, seed=0), np.linspace(1.0, 2.0, B))
        else:
            eng.clear_background()
        eng.eval_bits(bits)                                  # warm-up: plans, graph capture, scratch
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            eng.eval_bits(bits)
        e1.record()
        torch.cuda.synchronize()
        s = e0.elapsed_time(e1) / 1e3 / args.steps
        rows = n * max(1, B)
        bg_ms = None
        if B:
            eng.profile(True)
            eng.eval_bits(bits)
            torch.cuda.synchronize()
            prof = eng.profile_read()
            eng.profile(False)
            bg_ms = prof.get("bg_mean", {}).get("ms")
        ex = KernelShapExplainer(eng, nsamples=K, seed=0)
        bg = make_background(wl.num_samples, B, seed=0) if B else None
        ex.explain(clip, num_segments=M, targets=(frames, tokens), background=bg,
                   background_weights=np.linspace(1.0, 2.0, B) if B else None)    # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = ex.explain(clip, num_segments=M, targets=(frames, tokens), background=bg,
                         background_weights=np.linspace(1.0, 2.0, B) if B else None)
        torch.cuda.synchronize()
        s_clip = time.perf_counter() - t0
        r = dict(B=B, coalitions=n, rows=rows, s_per_eval=s, row_forwards_per_s=rows / s, coalitions_per_s=n / s,
                 s_per_clip=s_clip, bg_mean_ms=bg_ms, status=int(res["status"].item()))
        print(json.dumps(r))
        results.append(r)
    out = dict(workload="C2", model=wl.model, num_samples=wl.num_samples, segments=M, targets=len(frames),
               batch_tile=eng.kernel_count()[1], gpu=gpu_info(), results=results)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))
    eng.close()


if __name__ == "__main__":
    main()
