"""ORACLE (test infrastructure only): the transcript-level output W2S_OUT_CTC on the CPU.

``callback.reduce_logits`` extended by mode "transcript": out[r, d] = log p_CTC(y_d | logits[r]) in float64 through
``torch.nn.functional.ctc_loss`` -- the quantity HF's WavXForCTC(x, labels=y).loss computes (fp32 log_softmax, then
ctc_loss with blank = pad_token_id and reduction "sum"), negated.  ``evaluate`` / ``evaluate_coalitions`` are those of
``callback`` with this reduction, so ``kernelshap_ref.brute_force_shapley`` works for transcripts too.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from . import callback as CB
from . import w2v2_forward as W


def ctc_logp(logits: torch.Tensor, transcripts, blank: int = CB.PAD_ID) -> torch.Tensor:
    """logits [n, T, V] -> [n, D] float64: log p_CTC(y_d | logits[r]) over all T frames (natural log)."""
    lp = torch.log_softmax(logits.double(), dim=-1).transpose(0, 1)    # [T, n, V]
    T, n, _ = lp.shape
    cols = []
    for y in transcripts:
        y = torch.as_tensor(np.asarray(y, dtype=np.int64)).reshape(-1)
        tgt = y.repeat(n) if y.numel() else torch.zeros(0, dtype=torch.long)
        loss = F.ctc_loss(lp, tgt, torch.full((n,), T, dtype=torch.long), torch.full((n,), y.numel(), dtype=torch.long),
                          blank=blank, reduction="none", zero_infinity=False)
        cols.append(-loss)
    return torch.stack(cols, dim=1)


def reduce_logits(logits: torch.Tensor, mode: str, frames=None, tokens=None, transcripts=None,
                  blank: int = CB.PAD_ID) -> torch.Tensor:
    if mode == "transcript":
        return ctc_logp(logits, transcripts, blank)
    return CB.reduce_logits(logits, mode, frames, tokens)


@torch.no_grad()
def evaluate(sd, cfg: dict, X: np.ndarray, mode: str = "transcript", transcripts=None, blank: int = CB.PAD_ID,
             batch: int = 32, dtype=torch.float32, **kw) -> np.ndarray:
    """Waveforms X[n, L] -> reduced outputs [n, D] (float64 for transcripts)."""
    X = np.atleast_2d(np.asarray(X))
    outs = []
    for s in range(0, X.shape[0], batch):
        xb = torch.from_numpy(np.ascontiguousarray(X[s:s + batch])).to(dtype)
        outs.append(reduce_logits(W.ctc_logits(sd, cfg, xb), mode, transcripts=transcripts, blank=blank, **kw).double())
    return torch.cat(outs).numpy()


@torch.no_grad()
def evaluate_coalitions(sd, cfg, x, Z, bounds, baseline=0.0, **kw) -> np.ndarray:
    """f(Z[n, M]) -> [n, D] for the transcript reduction (callback.evaluate_coalitions with this module's evaluate)."""
    Z = np.atleast_2d(np.asarray(Z))
    batch = kw.pop("batch", 32)
    outs = []
    for s in range(0, Z.shape[0], batch):
        outs.append(evaluate(sd, cfg, CB.materialize(x, Z[s:s + batch], bounds, baseline), batch=batch, **kw))
    return np.concatenate(outs)
