#!/usr/bin/env python
"""BASELINE config 5: controlled clean + noisy synthetic test set (64 clips x 3 SNRs) -> batch explanation sweep
feeding eta_raw / WER, on N B200s.

    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 tools/run_c5.py [--clips 64] [--out data_c5]

Clip-level sharding (SURVEY.md 8e): item i of the test set goes to rank i % N, so the data path has NO collective at
all; every rank explains its items with the whole coalition set on its own GPU and writes the reference's four .npy
files per item (shap_calculation.py:200-210).  The only exchange is the final gather of the per-item metric rows.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as td

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from shap_transformer_asr_b200 import (MODELS, Engine, dist as wdist, eta_raw_segments, explain_test_set, make_background,
                                       make_test_set, wer)
from shap_transformer_asr_b200.modelzoo import build_random_init_model


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=64)
    ap.add_argument("--samples", type=int, default=102400)     # 6.4 s >= 100 000 samples (shap_calculation.py:75)
    ap.add_argument("--segments", type=int, default=128)
    ap.add_argument("--coalitions", type=int, default=2048)
    ap.add_argument("--out", default="data_c5")
    ap.add_argument("--model", default="wav2vec2-base")
    ap.add_argument("--save-limit", type=int, default=-1, help="write the four .npy files of the first N items per rank "
                    "only (a 6.4 s item is 130 MB of attributions); -1 = all, as the reference does")
    ap.add_argument("--background", type=int, default=0, help="explain against the reference's noise background "
                    "(make_background: N rows of 0.01 * randn, shap_calculation.py:125-127) instead of zero fill; 0 = zero fill")
    args = ap.parse_args()
    rank, world = wdist.init_from_env("cuda") if int(os.environ.get("WORLD_SIZE", "1")) > 1 else (0, 1)
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    cfg = MODELS[args.model]
    model = build_random_init_model(cfg, seed=0)
    eng = Engine(model, cfg, device=local, max_batch=0)
    test_set = make_test_set(num_clips=args.clips, num_samples=args.samples, snrs=(5, 2, 1), seed=0)
    # keep each clip's clean item with its noisy versions on one rank (the clean transcript is their WER reference)
    mine = [i for i in range(len(test_set)) if (i // 4) % world == rank]
    torch.cuda.synchronize()
    wdist.barrier()
    t0 = time.perf_counter()
    rows = []

    def consume(k, item, phi, bounds, r):      # the downstream metrics of every item, from the segment-level attributions
        rows.append(dict(item=mine[k], type=item["type"], snr=item["snr"], status=r["status"],
                         eta_raw=eta_raw_segments(item["audio"] - item["noise"], item["noise"], phi, bounds, 16000),
                         wer=wer(r["text"], r["hypothesis"])))

    explain_test_set(eng, [test_set[i] for i in mine], out_dir=os.path.join(args.out, f"rank{rank}"),
                     num_segments=args.segments, nsamples=args.coalitions, seed=0,
                     save_limit=None if args.save_limit < 0 else args.save_limit, on_item=consume,
                     background=make_background(args.samples, args.background, seed=0) if args.background > 0 else None)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    gathered = [None] * world
    if world > 1:
        td.all_gather_object(gathered, (rows, dt))
    else:
        gathered = [(rows, dt)]
    if rank == 0:
        allrows = sorted((x for g in gathered for x in g[0]), key=lambda x: x["item"])
        wall = max(g[1] for g in gathered)
        by = {}
        for x in allrows:
            by.setdefault(str(x["snr"]), []).append(x)
        summary = {k: dict(n=len(v), eta_raw_mean=float(np.mean([x["eta_raw"] for x in v])),
                           wer_mean=float(np.mean([x["wer"] for x in v]))) for k, v in by.items()}
        print(json.dumps(dict(workload="C5", n_gpus=world, items=len(allrows), coalitions_per_item=args.coalitions,
                              wall_s=wall, items_per_s=len(allrows) / wall,
                              coalition_forwards_per_s=len(allrows) * (args.coalitions + 3) / wall,
                              wls_failures=sum(x["status"] for x in allrows), by_snr=summary)), flush=True)
    if world > 1:
        td.destroy_process_group()


if __name__ == "__main__":
    main()
