"""Generates tests/golden/tiny_wavlm.npz and tiny_wavlm_stable.npz from the installed ``transformers`` WavLMForCTC.

    python -m oracle.make_golden_wavlm

Writes these two files only (oracle/make_golden.py rewrites every other fixture, and the zip timestamps alone would
change their bytes).  Same recipe as the wav2vec2 fixtures: the wav2vec2-tiny sizes, seeded random init with the affine
terms perturbed, seeded noise in, full logits out, a weight checksum against RNG drift.
"""
from __future__ import annotations

import dataclasses
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import wavlm_forward as WL  # noqa: E402
from oracle.make_golden import OUT, TINY, weight_checksum  # noqa: E402

VARIANTS = {
    "tiny_wavlm": dataclasses.replace(TINY, kind="wavlm"),   # group-norm front end, post-LN encoder
    "tiny_wavlm_stable": dataclasses.replace(TINY, kind="wavlm", feat_extract_norm="layer", conv_bias=True,
                                             do_stable_layer_norm=True),
}


def build(cfg, seed=0):
    return WL.randomize_affine(WL.build_hf_model(cfg.to_dict(), seed=seed), seed=seed + 1)


def main():
    os.makedirs(OUT, exist_ok=True)
    for name, cfg in VARIANTS.items():
        model = build(cfg)
        g = torch.Generator().manual_seed(7)
        x = torch.randn(3, 4000, generator=g)
        with torch.no_grad():
            logits = model(x).logits.numpy()
        np.savez_compressed(os.path.join(OUT, f"{name}.npz"), x=x.numpy(), logits=logits, checksum=weight_checksum(model))
        print(name, logits.shape, float(np.abs(logits).mean()))


if __name__ == "__main__":
    main()
