"""KernelSHAP around the device callback: host coalition sampler, sharded evaluation, device solve.

The sampler restates ``shap.KernelExplainer.explain`` (shap is pinned only as ``>=0.40.0`` in the
reference's requirements.txt:4 and is not installed here; algorithm per SURVEY.md Appendix A).  It
draws from the GLOBAL legacy ``np.random`` state in shap's exact call order --
``np.random.choice(len(p), 4 * left, p=p)`` once, then one ``np.random.permutation(M)`` per draw --
so ``np.random.seed(s)`` fixes the coalition index sets exactly as it would for shap.  ``l1_reg`` is
pinned to ``False`` (plain constrained WLS, solved on the device by ``w2s_wls``).
"""
from __future__ import annotations

import ctypes as C
import itertools
from math import comb
from typing import Optional

import numpy as np
import torch

from . import _lib
from . import dist as wdist
from .engine import background_arrays
from .preprocess import band_components, check_band_edges
from .targets import MAX_TRANSCRIPT, PAD_ID, SPACE_ID, char_targets, greedy_transcript, reference_length


def unpack_coalitions(words: np.ndarray, M: int) -> np.ndarray:
    """uint32 words [K, ceil(M/32)] -> uint8 {0,1} matrix [K, M] (inverse of preprocess.pack_coalitions)."""
    w = np.ascontiguousarray(words, dtype=np.uint32)
    bits = np.unpackbits(w.view(np.uint8).reshape(w.shape[0], -1), axis=1, bitorder="little")
    return np.ascontiguousarray(bits[:, :M])


def sample_coalitions(M: int, nsamples="auto", seed: Optional[int] = None, packed: bool = False):
    """-> (Z uint8 [K, M] with 1 = segment kept, kernel weights float64 [K], info dict); ``packed=True`` returns the
    bit-packed uint32 words [K, ceil(M/32)] (what the device consumes) instead of Z.

    All floating-point work (size weights, ``np.random.choice``, weight scaling) is numpy's own; the per-draw
    ``np.random.permutation(M)`` loop runs natively on numpy's MT19937 state (``w2s_sample_rows``, csrc/sampler.cu)."""
    if seed is not None:
        np.random.seed(seed)
    M = int(M)
    if M < 2:
        raise ValueError("KernelSHAP needs at least 2 features")
    if M > 2048:
        raise ValueError("at most 2048 segments are supported")
    nsamples = 2 * M + 2 ** 11 if nsamples == "auto" else int(nsamples)
    max_samples = 2 ** 30
    if M <= 30:
        max_samples = 2 ** M - 2
        nsamples = min(nsamples, max_samples)
    W = (M + 31) // 32
    words = np.zeros((nsamples, W), dtype=np.uint32)
    kw = np.zeros(nsamples, dtype=np.float64)
    added = 0

    n_sizes = int(np.ceil((M - 1) / 2.0))
    n_paired = int(np.floor((M - 1) / 2.0))
    wv = np.array([(M - 1.0) / (i * (M - i)) for i in range(1, n_sizes + 1)])
    wv[:n_paired] *= 2
    wv /= np.sum(wv)

    # sizes that can be enumerated completely with the sample budget
    n_full = 0
    left = nsamples
    rem = wv.copy()
    full = np.uint32(0xFFFFFFFF)
    tail = np.uint32((1 << (M % 32)) - 1) if M % 32 else full
    for size in range(1, n_sizes + 1):
        nsub = float(comb(M, size))
        if size <= n_paired:
            nsub *= 2
        if left * rem[size - 1] / nsub >= 1.0 - 1e-8:
            n_full += 1
            left -= nsub
            if rem[size - 1] < 1.0:
                rem /= (1 - rem[size - 1])
            w = wv[size - 1] / comb(M, size)
            if size <= n_paired:
                w /= 2.0
            # itertools.combinations order, each subset followed by its complement when paired
            idx = np.fromiter(itertools.chain.from_iterable(itertools.combinations(range(M), size)), dtype=np.int64)
            idx = idx.reshape(-1, size)
            rows = np.zeros((idx.shape[0], W), dtype=np.uint32)
            r = np.repeat(np.arange(idx.shape[0]), size)
            np.bitwise_or.at(rows, (r, (idx >> 5).ravel()), (np.uint32(1) << (idx & 31).astype(np.uint32)).ravel())
            if size <= n_paired:
                comp = ~rows
                comp[:, -1] &= tail
                block = np.stack([rows, comp], axis=1).reshape(-1, W)
            else:
                block = rows
            words[added:added + block.shape[0]] = block
            kw[added:added + block.shape[0]] = w
            added += block.shape[0]
        else:
            break

    n_fixed = added
    samples_left = nsamples - added
    if n_full != n_sizes:
        rem = wv.copy()
        rem[:n_paired] /= 2
        rem = rem[n_full:]
        rem /= np.sum(rem)
        ind_set = np.ascontiguousarray(np.random.choice(len(rem), 4 * samples_left, p=rem), dtype=np.int64)
        # one np.random.permutation(M) per draw, de-duplication and complements: native, on numpy's own generator state
        lib = _lib.load()
        name, key, pos, has_gauss, cached = np.random.get_state()
        key = np.ascontiguousarray(key, dtype=np.uint32).copy()
        cpos = C.c_int32(int(pos))
        used = C.c_int64(0)
        new_added = lib.w2s_sample_rows(M, n_full, n_paired, ind_set.ctypes.data, len(ind_set), samples_left, added,
                                        key.ctypes.data, C.byref(cpos), words.ctypes.data, kw.ctypes.data, nsamples,
                                        C.byref(used))
        if new_added < 0:
            raise RuntimeError("w2s_sample_rows failed")
        np.random.set_state((name, key, int(cpos.value), has_gauss, cached))
        added = int(new_added)
        weight_left = np.sum(wv[n_full:])
        kw[n_fixed:added] *= weight_left / kw[n_fixed:added].sum()
    info = dict(nsamples=nsamples, n_fixed=n_fixed, n_full_sizes=n_full, max_samples=max_samples)
    words, kw = words[:added], kw[:added]
    return (words if packed else unpack_coalitions(words, M)), kw, info


class KernelShapExplainer:
    """Explains one clip: Shapley value of every waveform segment for every per-character output.

    ``engine`` is a :class:`~shap_transformer_asr_b200.engine.Engine`.  With ``torch.distributed``
    initialised, the coalition rows are sharded across ranks (no data-path collective), the
    per-coalition outputs are all-gathered once, and every rank solves the regression."""

    def __init__(self, engine, nsamples="auto", seed: int = 0, shard_coalitions: bool = True):
        """``shard_coalitions=False`` keeps every coalition of a clip on this rank even when torch.distributed is
        initialised -- the clip-level sharding of batch sweeps (BASELINE config 5), where ranks explain DIFFERENT clips
        and must not meet in a collective."""
        self.engine = engine
        self.nsamples = nsamples
        self.seed = seed
        self.shard_coalitions = shard_coalitions
        self._cache = {}

    def _coalitions(self, M: int):
        """The sampled coalition matrix depends on (M, nsamples, seed) only -- not on the clip -- so with a fixed seed a
        sweep over many clips draws it once: later calls reuse the packed rows, their device copy and the kernel weights,
        and leave numpy's global generator in the state the draw would have left it in (exactly what re-sampling does)."""
        key = (int(M), self.nsamples, self.seed)
        hit = self._cache.get(key) if self.seed is not None else None
        if hit is None:
            words, kw, info = sample_coalitions(M, self.nsamples, seed=self.seed, packed=True)
            head = np.zeros((2, words.shape[1]), dtype=np.uint32)      # rows 0 / 1: the empty and the full coalition
            head[1] = 0xFFFFFFFF
            if M % 32:
                head[1, -1] = (1 << (M % 32)) - 1
            hit = dict(words=words, kw=kw, info=info, state=np.random.get_state(), all_words=np.concatenate([head, words]),
                       bits_dev=None, w_dev=None)
            if self.seed is not None:
                self._cache = {key: hit}
        else:
            np.random.set_state(hit["state"])
        return hit

    def select_targets(self, mode: str = "logprob"):
        eng = self.engine
        eng.set_targets("logits")
        ones = eng.bits_to_device(np.ones((1, eng.num_segments), dtype=np.uint8))
        logits = eng.eval_bits(ones).view(-1, eng.config.vocab_size).cpu().numpy()
        frames, tokens = char_targets(logits)
        eng.set_targets(mode, frames, tokens)
        return frames, tokens, logits

    def _clip_logits(self, M: int, num_features: Optional[int] = None):
        """-> (logits [T', V] of the unmasked clip, the coalitions sampled over ``num_features`` (default M) features).
        The one-row forward (one graph replay) is asynchronous on the engine's stream: the coalitions are drawn on the host
        while it runs, the logits are read back afterwards."""
        eng = self.engine
        eng.set_targets("logits")
        logits_dev = eng.eval_bits(eng.bits_to_device(np.ones((1, M), dtype=np.uint8)))
        sampled = self._coalitions(num_features or M)
        return logits_dev.view(-1, eng.config.vocab_size).cpu().numpy(), sampled

    def _greedy_target(self, M: int, num_features: int, blank: int, what: str):
        """-> ([the greedy transcript of the unmasked clip], the sampled coalitions), from one _clip_logits pass"""
        logits, sampled = self._clip_logits(M, num_features)
        greedy = greedy_transcript(logits, blank)
        if greedy.size > MAX_TRANSCRIPT:
            raise ValueError(f"the greedy transcript of this clip has {greedy.size} labels, more than "
                             f"W2S_MAX_TRANSCRIPT = {MAX_TRANSCRIPT}: pass the {what} as targets")
        return [greedy], sampled

    def explain(self, clip, num_segments: int, mode: str = "logprob", targets=None, baseline: float = 0.0,
                check: bool = True, background=None, background_weights=None, blank: int = PAD_ID, band_edges=None,
                sr: int = 16000, unit: str = "words"):
        """-> dict(phi[M, D] fp64 device, fx, fnull, frames, tokens, Z, weights, y, status, info, background_weights,
        transcripts, phi_cells, band_edges, references, reference_lengths).

        ``mode="transcript"`` explains whole transcripts: output d is log p_CTC(y_d | clip), the log-likelihood the model
        was trained on (-WavXForCTC(x, labels=y_d).loss, reduction "sum"), with ``blank`` its pad_token_id.  ``targets``
        is then a list of label-id sequences; by default the greedy transcript of the unmasked clip (the model's own
        transcription, from the same one-row logits pass that selects per-character targets).  ``transcripts`` in the
        result lists them (None in the other modes).  A transcript holds at most W2S_MAX_TRANSCRIPT = 512 labels: when
        the greedy transcript of the clip is longer, explain raises ValueError (pass ``targets`` explicitly, e.g. the
        transcripts of shorter clips).

        ``mode="errors"`` explains recognition errors: output d is the edit distance between the greedy transcript of the
        (masked) clip and reference d, in ``unit`` "words" (split on the "|" label, targets.SPACE_ID; WER x N) or "labels".
        ``targets`` is then a list of label-id sequences, e.g. ground-truth transcripts; by default the greedy transcript of
        the unmasked clip, from the same one-row pass as in transcript mode, so the full coalition scores exactly 0 and phi
        attributes the errors the masking introduces.  The result's ``references`` lists them and ``reference_lengths`` their
        N in the unit (divide by N for rates).  Longer references than W2S_MAX_TRANSCRIPT labels are refused as transcripts
        are.  The engine is left with the references set.

        ``check`` reads the solve's status word back (one 4-byte D2H after the solve) and raises if the regression
        did not produce a usable answer; a rank-deficient design (status 2: fewer distinct coalitions than segments)
        is solved for the minimum-norm attributions exactly as shap's ``lstsq`` fallback does and only warns.

        ``background``: ``shap.KernelExplainer(f, data)``'s background set, an array [B, L] in the clip's normalised
        input space, or the ``(data, weights)`` pair :func:`kmeans_background` returns; ``background_weights`` (default
        uniform, or the pair's) weight its rows.  Every coalition (the empty and the full one included) is then
        evaluated once per background row with the dropped segments taken from that row, and its output is the
        weighted mean over the rows; ``baseline`` is not used.  The targets are selected on the clip itself.  With
        ``background=None`` dropped segments are filled with ``baseline``; ``background_weights`` in the result is then
        None, else the normalised float64 weights.

        ``band_edges`` (F + 1 edges in Hz from 0 to sr / 2, e.g. ``preprocess.mel_band_edges(F)``) explains time-frequency
        cells: the clip is split into F band components (``preprocess.band_components``) and feature s * F + b is band b
        of segment s, so M = num_segments * F.  The targets are selected on the clip itself; the coalitions are then
        evaluated with the bands set (a row is the sum of its kept cells' components, the empty coalition is silence, the
        full one the sum of all components) and the engine is left with time-only coalitions.  The result adds
        ``phi_cells`` = phi viewed as [num_segments, F, D] and the float64 ``band_edges`` (both None without bands).
        Bands cannot be combined with a background."""
        eng = self.engine
        eng.set_clip(clip, num_segments=num_segments, baseline=baseline)
        bg = None
        if background is not None:
            if isinstance(background, tuple):
                if background_weights is not None:
                    raise ValueError("pass the weights either in the (data, weights) pair or as background_weights")
                background, background_weights = background
            bg = background_arrays(background, background_weights, num_samples=eng.num_samples)
        elif background_weights is not None:
            raise ValueError("background_weights given without a background")
        edges = None
        if band_edges is not None:
            if bg is not None:
                raise ValueError("band_edges cannot be combined with a background")
            edges = check_band_edges(band_edges, sr)
            if eng.num_segments * (edges.size - 1) > 2048:
                raise ValueError(f"{eng.num_segments} segments x {edges.size - 1} bands = "
                                 f"{eng.num_segments * (edges.size - 1)} cells; at most 2048 are supported")
        if getattr(eng, "background_rows", 0):
            eng.clear_background()
        if getattr(eng, "num_bands", 0):
            eng.clear_bands()
        M = eng.num_segments
        Mf = M if edges is None else M * (edges.size - 1)     # features: segments, or time-frequency cells
        sampled = None
        transcripts = references = None
        if mode in ("max", "mean", "logits"):
            frames, tokens = (), ()
            eng.set_targets(mode)
        elif mode == "transcript":
            frames, tokens = (), ()
            if targets is None:
                targets, sampled = self._greedy_target(M, Mf, blank, "transcripts")
            eng.set_transcripts(targets, blank)
            transcripts = eng.transcripts
        elif mode == "errors":
            frames, tokens = (), ()
            if targets is None:
                targets, sampled = self._greedy_target(M, Mf, blank, "references")
            eng.set_references(targets, unit=unit, blank=blank, delimiter=SPACE_ID)
            references = eng.references
        elif targets is None:
            logits, sampled = self._clip_logits(M, Mf)
            frames, tokens = char_targets(logits)
            eng.set_targets(mode, frames, tokens)
        else:
            frames, tokens = targets
            eng.set_targets(mode, frames, tokens)
        if sampled is None:
            sampled = self._coalitions(Mf)
        words, kw, info = sampled["words"], sampled["kw"], sampled["info"]
        K = words.shape[0]
        if bg is not None:
            eng.set_background(*bg)
        if edges is not None:
            eng.set_bands(band_components(clip, edges, sr))
        # rows 0 / 1 of the evaluated matrix are the empty and the full coalition (fnull, fx): fx comes from the same
        # reduction kernel as every y row, so the efficiency constraint is consistent to the last bit
        rank, world = wdist.rank_world() if self.shard_coalitions else (0, 1)
        lo, hi = wdist.shard_range(K + 2, rank, world)
        if sampled["bits_dev"] is None or sampled["bits_dev"].device != eng.device:
            sampled["bits_dev"] = eng.bits_to_device(sampled["all_words"]).clone()     # own copy: survives later uploads
            sampled["w_dev"] = torch.from_numpy(kw).to(eng.device)
        bits_all = sampled["bits_dev"]
        y_local = eng.eval_bits(bits_all[lo:hi]) if hi > lo else torch.empty((0, eng.out_width()), device=eng.device)
        y_all = wdist.all_gather_rows(y_local, K + 2, rank, world)
        fnull = y_all[0].double()
        fx = y_all[1].double()
        phi, status = eng.wls(bits_all[2:], sampled["w_dev"], y_all[2:], fx, fnull, Mf)
        bg_w = None
        if bg is not None:
            bg_w = eng.background_weights
            eng.clear_background()      # the engine is left as it was found: baseline fill
        if edges is not None:
            eng.clear_bands()           # ... and time-only coalitions
        if check:
            st = int(status.item())
            if st == 1:
                raise RuntimeError("KernelSHAP regression did not converge (w2s_wls status 1)")
            if st == 2:
                import warnings
                warnings.warn(f"KernelSHAP design is rank deficient ({K} coalitions for {Mf} features): minimum-norm "
                              "attributions returned (shap's lstsq fallback)", RuntimeWarning)
        phi_cells = None if edges is None else phi.view(M, edges.size - 1, phi.shape[1])
        return dict(phi=phi, fx=fx, fnull=fnull, frames=frames, tokens=tokens, Z=unpack_coalitions(words, Mf), weights=kw,
                    y=y_all[2:], status=status, info=info, words=words, background_weights=bg_w, transcripts=transcripts,
                    phi_cells=phi_cells, band_edges=edges, references=references,
                    reference_lengths=None if references is None else
                    [reference_length(r, unit, SPACE_ID) for r in references])


def kmeans_background(X, k: int, round_values: bool = True):
    """``shap.kmeans(X, k, round_values)`` restated (from memory of shap's ``utils/_legacy.py``; shap is not installed, so
    parity with shap itself is unpinned): ``sklearn.cluster.KMeans(n_clusters=k, random_state=0)`` over the rows of
    ``X`` [n, L]; with ``round_values`` every centre coordinate is replaced by the nearest value its column takes in
    ``X``; the weights are the cluster sizes.  -> (data float32 [k, L], weights float64 [k]), the pair
    ``KernelShapExplainer.explain(background=...)`` accepts."""
    from sklearn.cluster import KMeans

    X = np.asarray(X, dtype=np.float64)
    if X.ndim != 2:
        raise ValueError(f"X must be [n, L], got shape {X.shape}")
    k = int(k)
    if k < 1 or k > X.shape[0]:
        raise ValueError(f"k = {k} clusters for {X.shape[0]} rows")
    km = KMeans(n_clusters=k, random_state=0).fit(X)
    centres = km.cluster_centers_.copy()
    if round_values:
        cols = np.arange(X.shape[1])
        for j0 in range(0, X.shape[1], 4096):     # [k, n, 4096] distances per chunk of columns
            c = cols[j0:j0 + 4096]
            nearest = np.abs(centres[:, None, c] - X[None, :, c]).argmin(axis=1)     # [k, chunk]: row index
            centres[:, c] = X[nearest, c[None, :]]
    weights = np.bincount(km.labels_, minlength=k).astype(np.float64)
    return centres.astype(np.float32), weights


def expand_to_samples(phi: np.ndarray, bounds: np.ndarray, per_sample: bool = False) -> np.ndarray:
    """phi[M, D] -> [1, L, D], the reference's on-disk layout (shap_calculation.py:200-210;
    evaluation.ipynb:503-504).  Each segment's value is repeated over its samples (or divided by the
    segment length when ``per_sample``); visualization.py:354 only uses relative magnitudes."""
    lens = np.diff(bounds)
    v = phi / lens[:, None] if per_sample else phi
    return np.repeat(v, lens, axis=0)[None]
