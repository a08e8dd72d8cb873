"""Batch explanation sweep and the reference's on-disk format (SURVEY.md section 8, rows f2 / f4; BASELINE config 5).

* ``add_noise`` / ``make_test_set``  -- shap_calculation.py:55-108 with a SEEDED generator and synthetic clips (the
  reference pulls LibriSpeech from the hub and uses the unseeded global RNG).
* ``explain_test_set``               -- shap_calculation.py:170-210: one explanation per item, four ``.npy`` files per
  item named exactly as the reference names them, shap array ``[1, L, T']`` (evaluation.ipynb:503-504), so that
  visualization.py / calculate_metric.py / nraw_vs_wer.py can read them unmodified.
"""
from __future__ import annotations

import os
from typing import Dict, List

import numpy as np

from .kernelshap import KernelShapExplainer, expand_to_samples
from .metrics import greedy_ctc_decode
from .preprocess import normalize_clip, synthetic_clip
from .targets import greedy_transcript


def add_noise(audio: np.ndarray, snr_db: float, rng: np.random.Generator) -> np.ndarray:
    """White noise at the given SNR (shap_calculation.py:55-60)."""
    signal_power = np.mean(audio ** 2)
    noise_power = signal_power / (10 ** (snr_db / 10))
    return audio + rng.normal(0, np.sqrt(noise_power), len(audio))


def make_test_set(num_clips: int = 2, num_samples: int = 102400, snrs=(5, 2, 1), seed: int = 0) -> List[Dict]:
    """clean + noisy items per clip, in the reference's order and dict layout (shap_calculation.py:63-108);
    clips are at least 100 000 samples long as there (:75)."""
    rng = np.random.default_rng(seed)
    items = []
    for i in range(num_clips):
        audio = synthetic_clip(num_samples, seed=1000 + seed * 131 + i).astype(np.float64)
        items.append({"type": "clean", "audio": audio, "text": None, "snr": float("inf"), "noise": np.zeros_like(audio)})
        for snr in snrs:
            noisy = add_noise(audio, snr, rng)
            items.append({"type": "noisy", "audio": noisy, "text": None, "snr": snr, "noise": noisy - audio})
    return items


def explain_test_set(engine, test_set: List[Dict], out_dir: str = "data", num_segments: int = 128, nsamples=2048,
                     seed: int = 0, mode: str = "max", save_limit=None, on_item=None, background=None) -> List[Dict]:
    """Explain every item and write ``{shap_values,audio,noise,text}_sample_{i}_{type}_{snr}.npy``
    (shap_calculation.py:200-210).  ``mode="max"`` explains the max logit of every output frame, which is what the
    reference's wrapper returns (shap_calculation.py:50), so the saved array has the reference's ``[1, L, T']`` shape.
    The text of an item is the greedy transcript of its clip's clean version (random-init weights have no ground truth).

    Every item is explained on THIS rank's GPU (clip-level sharding: the caller hands each rank its items).
    ``save_limit``: write the files of the first N items only (a 6.4 s item is 130 MB of float32 attributions);
    ``on_item(index, item, phi, bounds, result)`` is called for every item, saved or not, with the segment-level
    attributions ``phi [M, T']`` (the ``[1, L, T']`` expansion is only materialised for the items that are written).
    ``background``: passed to every ``KernelShapExplainer.explain`` call -- an array [B, L] or a ``(data, weights)`` pair,
    e.g. the reference's noise background ``make_background(L, 5, seed)`` (shap_calculation.py:125-127) -- so the
    KernelSHAP attributions are taken against the same background as the expected-gradients ones; None fills the dropped
    segments with zeros.

    ``mode="errors"`` explains each item's word errors against its text, kept as label ids (the clean item's greedy
    transcript): the attributions of a noisy item then locate the audio that caused its WER.  The result of an item adds
    ``errors``, the device's word-error count of the unmasked item (``wer(text, hypothesis) * reference_words``), and
    ``reference_words``.  Items must come without a text of their own in this mode."""
    os.makedirs(out_dir, exist_ok=True)
    explainer = KernelShapExplainer(engine, nsamples=nsamples, seed=seed, shard_coalitions=False)
    results, clean_text = [], None
    for i, item in enumerate(test_set):
        x = normalize_clip(item["audio"])
        engine.set_clip(x, num_segments=num_segments)
        engine.set_targets("logits")
        ones = engine.bits_to_device(np.ones((1, num_segments), np.uint8))
        logits = engine.eval_bits(ones).view(-1, engine.config.vocab_size).cpu().numpy()
        hyp = greedy_ctc_decode(logits.argmax(-1))
        if item["type"] == "clean":
            clean_text, clean_ids = hyp, greedy_transcript(logits)
        text = item["text"] if item["text"] is not None else clean_text
        T = logits.shape[0]
        if mode == "errors":
            if item["text"] is not None:
                raise ValueError("mode='errors' explains against the clean item's greedy transcript: items carry no text")
            targets = [clean_ids]
        else:
            targets = ((), ()) if mode == "max" else (np.arange(T, dtype=np.int32), logits.argmax(-1).astype(np.int32))
        res = explainer.explain(x, num_segments=num_segments, mode=mode, targets=targets, background=background)
        phi = res["phi"].cpu().numpy()
        tag = f"sample_{i + 1}_{item['type']}_{item['snr']}"
        saved = save_limit is None or i < save_limit
        shape = (1, int(engine.bounds[-1]), phi.shape[1])
        if saved:
            shap_values = expand_to_samples(phi, engine.bounds).astype(np.float32)      # [1, L, T']
            np.save(os.path.join(out_dir, f"shap_values_{tag}"), shap_values)
            np.save(os.path.join(out_dir, f"audio_{tag}"), item["audio"])
            np.save(os.path.join(out_dir, f"noise_{tag}"), item["noise"])
            np.save(os.path.join(out_dir, f"text_{tag}.npy"), text)
        results.append(dict(tag=tag, hypothesis=hyp, text=text, shap_shape=shape, saved=saved,
                            status=int(res["status"].item())))
        if mode == "errors":
            results[-1].update(errors=float(res["fx"][0].item()), reference_words=res["reference_lengths"][0])
        if on_item is not None:
            on_item(i, item, phi, np.asarray(engine.bounds), results[-1])
    return results
