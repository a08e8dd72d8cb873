"""Cost of the transcript-level output (W2S_OUT_CTC) and of its gradient seed.

    python tools/bench_transcript.py [--steps 3] [--labels 70] [--out FILE.json]

KernelSHAP at the C2 shape (wav2vec2-base, one 5 s clip, 100 segments, 2048 coalitions + the empty and the full one):
  coalitions_per_s      eval_bits of all 2050 coalitions, CUDA events, logprob mode (per-character targets) and transcript
                        mode (one transcript of --labels labels), the two modes alternated --steps times
  head_reduce_ms_tile   time of the head reduction launch per batch tile (w2s_profile, a separate eager run)
Expected gradients at L = 183 600 (the recorded 11.5 s clip, T' = 573), 32 rows per call:
  passes_per_s          grad_transcripts rows per second against grad_waveforms (per-frame max logit)
  seed_share            share of the head_bwd step (the CTC seed kernels in transcript mode) in one call (w2s_profile)
  s_transcript_clip     one ExpectedGradientsExplainer.shap_values(x, transcripts=[y]) with 200 samples, host clock
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
from shap_transformer_asr_b200 import (MODELS, WORKLOADS, Engine, ExpectedGradientsExplainer, char_targets,  # noqa: E402
                                       make_background, sample_coalitions, synthetic_clip)
from shap_transformer_asr_b200.modelzoo import build_random_init_model  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except Exception:
        return None


def timed(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / steps


def profiled(eng, fn, key):
    eng.profile(True)
    fn()
    torch.cuda.synchronize()
    prof = eng.profile_read()
    eng.profile(False)
    total = sum(v["ms"] for v in prof.values())
    return prof.get(key, {}).get("ms"), prof.get(key, {}).get("launches"), total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--labels", type=int, default=70, help="labels of the explained transcript (about 14 per second)")
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    args = ap.parse_args()
    wl = WORKLOADS["C2"]
    cfg = MODELS[wl.model]
    model = build_random_init_model(cfg, seed=0)
    rng = np.random.default_rng(0)
    y = [int(v) for v in rng.integers(5, cfg.vocab_size, args.labels)]    # random letters: repeats as in text
    out = dict(gpu=gpu_info(), model=wl.model, labels=args.labels)

    # ---- KernelSHAP evaluation, C2 ----
    clip = synthetic_clip(wl.num_samples)
    M, K = wl.num_segments, wl.num_coalitions
    eng = Engine(model, cfg, max_batch=0)
    eng.set_clip(clip, num_segments=M)
    eng.set_targets("logits")
    logits = eng.eval_bits(eng.bits_to_device(np.ones((1, M), np.uint8))).view(-1, cfg.vocab_size).cpu().numpy()
    frames, tokens = char_targets(logits)
    Z, _, _ = sample_coalitions(M, K, seed=0)
    Z = np.concatenate([np.zeros((1, M), np.uint8), np.ones((1, M), np.uint8), Z])
    bits = eng.bits_to_device(Z).clone()
    n = Z.shape[0]
    modes = {"logprob": lambda: eng.set_targets("logprob", frames, tokens), "transcript": lambda: eng.set_transcripts([y])}
    times = {m: [] for m in modes}
    for m, setm in modes.items():      # warm-up of both
        setm()
        eng.eval_bits(bits)
    torch.cuda.synchronize()
    for _ in range(args.steps):
        for m, setm in modes.items():
            setm()
            times[m].append(timed(lambda: eng.eval_bits(bits), 1))
    tile = eng.kernel_count()[1]
    c2 = {}
    for m, setm in modes.items():
        setm()
        ms, launches, _ = profiled(eng, lambda: eng.eval_bits(bits), "head_reduce")
        s = float(np.median(times[m]))
        c2[m] = dict(s_per_eval=s, coalitions_per_s=n / s, all_s=times[m], head_reduce_ms_tile=ms / launches,
                     tiles=launches)
        print(json.dumps({m: c2[m]}))
    out["c2"] = dict(coalitions=n, batch_tile=tile, targets=len(frames), modes=c2)
    eng.close()

    # ---- expected gradients at L = 183 600 ----
    L = 183600
    eng = Engine(model, cfg, max_batch=0)
    T = eng.num_frames(L)
    x = torch.from_numpy(np.random.default_rng(1).standard_normal((32, L)).astype(np.float32)).cuda()
    eng.set_transcripts([y])
    which = np.zeros(32, np.int32)
    fr = np.arange(32, dtype=np.int32) % T
    calls = {"transcript": lambda: eng.grad_transcripts(x, which), "max_logit": lambda: eng.grad_waveforms(x, fr)}
    eg = {}
    for m, fn in calls.items():
        fn()
        torch.cuda.synchronize()
    gt = {m: [] for m in calls}
    for _ in range(args.steps):
        for m, fn in calls.items():
            gt[m].append(timed(fn, 1))
    for m, fn in calls.items():
        ms, _, total = profiled(eng, fn, "grad.head_bwd")
        s = float(np.median(gt[m]))
        eg[m] = dict(s_per_call=s, passes_per_s=32 / s, all_s=gt[m], head_bwd_ms=ms, seed_share=ms / total)
        print(json.dumps({m: eg[m]}))
    clip = synthetic_clip(L)
    ex = ExpectedGradientsExplainer(eng, make_background(L, 5, seed=0), nsamples=200, seed=0, batch=32)
    ex.shap_values(clip[:L], transcripts=[y])       # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    phi = ex.shap_values(clip[:L], transcripts=[y])
    torch.cuda.synchronize()
    s_clip = time.perf_counter() - t0
    out["expected_gradients"] = dict(num_samples=L, frames=T, rows_per_call=32, modes=eg, s_transcript_clip=s_clip,
                                     phi_finite=bool(np.isfinite(phi).all()))
    print(json.dumps(dict(s_transcript_clip=s_clip)))
    eng.close()
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
