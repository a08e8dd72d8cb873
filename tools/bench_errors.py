"""Cost of the recognition-error output (W2S_OUT_ERRORS) against the other modes of the head launch.

    python tools/bench_errors.py [--steps 5] [--labels 70] [--out FILE.json]

KernelSHAP at the C2 shape (wav2vec2-base, one 5 s clip, 100 segments, 2048 coalitions + the empty and the full one, the
automatic batch tile):
  coalitions_per_s      eval_bits of all 2050 coalitions, CUDA events, in four modes alternated --steps times:
                        logprob (per-character targets), transcript (one transcript of --labels labels), and the label and
                        word errors against the same labels as the reference (a space every 5 labels)
  head_reduce_ms_tile   time of the head reduction launch per batch tile (w2s_profile, a separate eager run per mode)
The GPU name and power limit are read in the same run and written beside the numbers."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from shap_transformer_asr_b200 import MODELS, WORKLOADS, Engine, char_targets, sample_coalitions, synthetic_clip  # noqa: E402
from shap_transformer_asr_b200.modelzoo import build_random_init_model  # noqa: E402
from bench_transcript import gpu_info, profiled, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--labels", type=int, default=70, help="labels of the transcript / reference (about 14 per second)")
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    args = ap.parse_args()
    wl = WORKLOADS["C2"]
    cfg = MODELS[wl.model]
    model = build_random_init_model(cfg, seed=0)
    rng = np.random.default_rng(0)
    y = [int(v) for v in rng.integers(5, cfg.vocab_size, args.labels)]
    y = [4 if i % 5 == 4 else v for i, v in enumerate(y)]          # words of four letters
    out = dict(gpu=gpu_info(), model=wl.model, labels=args.labels)

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
    modes = {"logprob": lambda: eng.set_targets("logprob", frames, tokens),
             "transcript": lambda: eng.set_transcripts([y]),
             "errors_labels": lambda: eng.set_references([y], unit="labels"),
             "errors_words": lambda: eng.set_references([y], unit="words")}
    times = {m: [] for m in modes}
    for m, setm in modes.items():      # warm-up of every mode
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
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
