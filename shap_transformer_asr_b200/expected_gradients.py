"""Expected gradients around the device input-gradient path -- the reference's production explainer.

``shap_calculation.py:125-162`` builds ``shap.GradientExplainer(wrapped_model, background, batch_size=1)`` over five
near-zero background clips and calls ``.shap_values(input_values)``; shap then loops over every output index (all T'
frames: ``ranked_outputs=None``) and ``nsamples = 200`` random (background, alpha) pairs, one forward + backward pass at
batch 1 each (traceback in ``feasability_tests/conformer_test.ipynb:95``): 114 600 passes for the recorded 11.5 s clip.

This module restates that estimator (shap is not installable here: algorithm FROM MEMORY of shap's
``_PyTorchGradient.shap_values``, as SURVEY.md Appendix A does for KernelExplainer -- parity with shap itself is
UNPINNED; what is pinned is the gradient, against torch autograd on the ``transformers`` model) and batches the passes:

    phi[:, j] = mean_s  d out_j / d x (x_s) * (x - bg_s),   x_s = bg_s + alpha_s (x - bg_s),  alpha_s ~ U(0, 1)

with the per-sample gradient rows evaluated by ``Engine.grad_waveforms`` in tiles.  Samples are drawn once per output
index from a seeded ``numpy`` generator, as shap reseeds per explained output.

Multi-GPU (one process per GPU, ``torch.distributed`` initialised): the passes of different output frames are
independent, so the OUTPUT FRAMES are split into contiguous blocks over the ranks -- no collective on the data path, every
rank accumulates only its own columns of phi, and one all-gather at the end assembles ``[D, L]`` on every rank.  Because a
column is produced by exactly one rank in the same order as on one GPU, the result is bit-identical for any world size.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import dist as wdist
from .targets import PAD_ID


def make_background(num_samples: int, num_background: int = 5, seed: Optional[int] = None) -> np.ndarray:
    """zeros + 0.01 * randn, the reference's background set (shap_calculation.py:125-127; unseeded there)."""
    rng = np.random.default_rng(seed)
    return (0.01 * rng.standard_normal((num_background, num_samples))).astype(np.float32)


class ExpectedGradientsExplainer:
    """phi[L, T'] for the ModelWrapper outputs (max logit per frame) of one clip."""

    def __init__(self, engine, background: np.ndarray, nsamples: int = 200, seed: int = 0, batch: int = 64,
                 shard_outputs: bool = True):
        self.engine = engine
        self.background = np.ascontiguousarray(background, dtype=np.float32)
        self.nsamples = int(nsamples)
        self.seed = seed
        self.batch = int(batch)
        self.shard_outputs = bool(shard_outputs)     # split the output frames over the ranks of torch.distributed

    def shap_values(self, x, frames=None, transcripts=None, blank: int = PAD_ID) -> np.ndarray:
        """x: normalised clip [L] -> attributions [1, L, D] (the reference's on-disk layout, D = T' when ``frames`` is
        None: every output frame, as ``ranked_outputs=None``).

        ``transcripts`` (a list of D label-id sequences, exclusive with ``frames``) explains transcript-level outputs
        instead: output d is log p_CTC(y_d | x) (-WavXForCTC(x, labels=y_d).loss, reduction "sum"; ``blank`` = the model's
        pad_token_id), one output per transcript, so 200 passes explain a whole transcript where the per-frame question
        takes T' x 200.  The transcripts are set on the engine (``Engine.set_transcripts``).  Draws are seeded per output
        index d as per frame; under torch.distributed the outputs are split over the ranks as the frames are, so with D
        smaller than the world size some ranks idle (sharding the samples of one output is not built).

        The (output, sample) passes of ALL outputs form one list that is cut into device calls of ``batch`` rows
        (every row carries its own target frame or transcript), so no call is ragged except the last."""
        eng = self.engine
        x = np.ascontiguousarray(np.asarray(x, dtype=np.float32).reshape(-1))
        L = x.size
        T = eng.num_frames(L)
        if transcripts is not None:
            if frames is not None:
                raise ValueError("frames and transcripts are mutually exclusive")
            eng.set_transcripts(transcripts, blank)
            frames = np.arange(len(eng.transcripts), dtype=np.int32)     # output d <-> transcript d
            grad_rows = eng.grad_transcripts
        else:
            frames = np.arange(T, dtype=np.int32) if frames is None else np.asarray(frames, dtype=np.int32)
            grad_rows = eng.grad_waveforms
        D, S = len(frames), self.nsamples
        bg = torch.from_numpy(self.background).to(eng.device)
        xt = torch.from_numpy(x).to(eng.device)
        # per output frame its own seeded draws (background index, alpha), as shap reseeds per explained output
        rind = np.empty((D, S), dtype=np.int64)
        alpha = np.empty((D, S), dtype=np.float32)
        for d, j in enumerate(frames):
            rng = np.random.default_rng([self.seed, int(j)])
            rind[d] = rng.integers(0, bg.shape[0], S)
            alpha[d] = rng.uniform(size=S).astype(np.float32)
        rind_t = torch.from_numpy(rind.reshape(-1)).to(eng.device)
        alpha_t = torch.from_numpy(alpha.reshape(-1)).to(eng.device)
        rank, world = wdist.rank_world() if self.shard_outputs else (0, 1)
        d_lo, d_hi = wdist.shard_range(D, rank, world)                         # this rank's output frames
        out_of = torch.arange(D, device=eng.device).repeat_interleave(S) - d_lo   # row -> local output slot
        row_frames = np.repeat(frames, S)
        phi = torch.zeros((d_hi - d_lo, L), dtype=torch.float32, device=eng.device)
        for r0 in range(d_lo * S, d_hi * S, self.batch):
            r1 = min(r0 + self.batch, d_hi * S)
            b = bg[rind_t[r0:r1]]
            delta = xt[None] - b
            xs = torch.addcmul(b, alpha_t[r0:r1, None], delta)
            g, _ = grad_rows(xs, row_frames[r0:r1])
            phi.index_add_(0, out_of[r0:r1], g * delta)
        phi /= S
        phi = wdist.all_gather_rows(phi, D, rank, world)                       # [D, L] on every rank
        return phi.t().contiguous()[None].cpu().numpy()
