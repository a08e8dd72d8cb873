"""A/B of the feature encoder's constant-frame skip on one workload (default C2): a dense-front-end engine
(W2S_FLAG_DENSE_FRONTEND) and the default engine on the same clip, coalitions and targets, timed alternately in one
process, then a per-launch CUDA-event profile of each arm.  The outputs of the two arms must be bit-identical.

    python tools/bench_frontend_skip.py [--workload C2] [--rounds 5] [--steps 3] [--out FILE]

Prints one JSON object (also written to --out): median ms per step of each arm and its spread over the rounds, the
per-launch breakdown of the encoder (conv0 .. conv6, the fills, the list kernel), the card, its power limit and SM clocks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload construction shared with the benchmark)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return r.stdout.strip().splitlines()[torch.cuda.current_device()]
    except Exception as e:  # the numbers are reported without it
        return f"unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="C2")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from shap_transformer_asr_b200 import Engine

    wl, cfg, clip, Z, _ = bench.build_problem(args.workload)
    model = bench.make_hf_model(cfg)
    _, frames, tokens = bench.clip_targets(model, clip)
    arms = {}
    for name, dense in (("dense", True), ("skip", False)):
        eng = Engine(model, cfg, dense_frontend=dense)
        eng.set_clip(clip, num_segments=wl.num_segments)
        eng.set_targets("logprob", frames, tokens)
        bits = eng.bits_to_device(Z)
        out = torch.empty((Z.shape[0], len(frames)), dtype=torch.float32, device="cuda")
        arms[name] = (eng, bits, out)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def step(name):
        eng, bits, out = arms[name]
        flush.fill_(1)
        eng.eval_bits(bits, out)

    for name in arms:
        for _ in range(2):
            step(name)
    torch.cuda.synchronize()
    same = torch.equal(arms["dense"][2], arms["skip"][2])
    times = {k: [] for k in arms}
    for _ in range(args.rounds):
        for name in ("dense", "skip"):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.steps):
                step(name)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.steps)
    same = same and torch.equal(arms["dense"][2], arms["skip"][2])
    breakdown = {}
    for name, (eng, _, _) in arms.items():
        eng.profile(True)
        step(name)
        torch.cuda.synchronize()
        prof = eng.profile_read()
        eng.profile(False)
        breakdown[name] = {k: dict(ms=round(v["ms"], 3), tflops=round(v["flops"] / 1e12, 2), gbytes=round(v["bytes"] / 1e9, 2))
                           for k, v in prof.items() if k.startswith(("conv", "frontend"))}
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = dict(workload=args.workload, card=card(), bit_identical=bool(same),
               ms_per_step={k: dict(median=round(med[k], 2), min=round(min(v), 2), max=round(max(v), 2),
                                    runs=[round(t, 2) for t in v]) for k, v in times.items()},
               speedup=round(med["dense"] / med["skip"], 4), breakdown_ms_one_step=breakdown)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    for eng, _, _ in arms.values():
        eng.close()
    if not same:
        sys.exit("outputs of the dense and skip arms differ")


if __name__ == "__main__":
    main()
