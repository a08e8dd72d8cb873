"""Python owner of one ``w2s_handle`` (include/w2s.h): weights, clip, targets and evaluation calls.

PyTorch is used only as plumbing here: device allocations, the current CUDA stream and
pinned host staging.  All arithmetic happens inside ``libw2s.so``.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from .config import ModelConfig
from .preprocess import pack_coalitions, segment_bounds
from .targets import PAD_ID, check_offsets, transcript_arrays


# ModelConfig.kind -> w2s_config.kind and the HF state_dict prefix of the encoder
KIND_IDS = {"wav2vec2": 0, "conformer": 1, "wavlm": 2}
PREFIXES = {"wav2vec2": "wav2vec2.", "conformer": "wav2vec2_conformer.", "wavlm": "wavlm."}


def _fold_pos_conv(sd: Dict[str, torch.Tensor], prefix: str) -> None:
    """weight_norm(dim=2) fold (HF wav2vec2/modeling_wav2vec2.py:337-354): w = g * v / ||v||_(0,1)."""
    p = prefix + "encoder.pos_conv_embed.conv."
    k0, k1 = p + "parametrizations.weight.original0", p + "parametrizations.weight.original1"
    if p + "weight" not in sd:
        if k0 in sd:
            g, v = sd[k0].float(), sd[k1].float()
        elif p + "weight_g" in sd:
            g, v = sd[p + "weight_g"].float(), sd[p + "weight_v"].float()
        else:
            return
        sd[p + "weight"] = v * (g / v.pow(2).sum(dim=(0, 1), keepdim=True).sqrt())


def background_arrays(bg, weights=None, num_samples: Optional[int] = None):
    """Validated background set: (rows float32 [B, L], weights float64 [B]).  ``bg`` is [B, L] (or one row [L]), numpy or
    torch; ``weights`` default to uniform.  Raises ValueError naming the problem: no rows, more than
    ``_lib.MAX_BACKGROUND``, a length other than ``num_samples``, or weights that are negative, not finite, of the wrong
    count or summing to zero.  Host only (the rows stay where they are when ``bg`` is a tensor)."""
    data = bg if isinstance(bg, torch.Tensor) else np.asarray(bg, dtype=np.float32)
    if data.ndim == 1:
        data = data[None]
    if data.ndim != 2:
        raise ValueError(f"background must be [B, L], got shape {tuple(data.shape)}")
    B, L = data.shape
    if B < 1 or B > _lib.MAX_BACKGROUND:
        raise ValueError(f"background has {B} rows; need 1 <= B <= {_lib.MAX_BACKGROUND}")
    if num_samples is not None and L != num_samples:
        raise ValueError(f"background rows have {L} samples, the clip has {num_samples}")
    w = np.ones(B, dtype=np.float64) if weights is None else np.ascontiguousarray(weights, dtype=np.float64).reshape(-1)
    if w.shape != (B,):
        raise ValueError(f"{w.size} background weights for {B} rows")
    if not np.all(np.isfinite(w)) or np.any(w < 0):
        raise ValueError("background weights must be finite and >= 0")
    if not w.sum() > 0:
        raise ValueError("background weights sum to zero")
    return data, np.ascontiguousarray(w)


def band_arrays(components, num_samples: Optional[int] = None, num_segments: Optional[int] = None,
                background_rows: int = 0):
    """Validated band components of time-frequency cells: [F, L] (numpy or torch; preprocess.band_components makes them).
    Raises ValueError naming the problem: not [F, L], F outside 1 .. ``_lib.MAX_BANDS``, a length other than
    ``num_samples``, ``num_segments * F`` above 2048 cells, or a background set.  Host only."""
    if components is None:
        raise ValueError("band components are None")
    data = components if isinstance(components, torch.Tensor) else np.asarray(components, dtype=np.float32)
    if data.ndim != 2:
        raise ValueError(f"band components must be [F, L], got shape {tuple(data.shape)}")
    F, L = data.shape
    if F < 1 or F > _lib.MAX_BANDS:
        raise ValueError(f"{F} bands; need 1 <= F <= {_lib.MAX_BANDS}")
    if num_samples is not None and L != num_samples:
        raise ValueError(f"band components have {L} samples, the clip has {num_samples}")
    if num_segments is not None and num_segments * F > 2048:
        raise ValueError(f"{num_segments} segments x {F} bands = {num_segments * F} cells; at most 2048 are supported")
    if background_rows:
        raise ValueError("a background is set: bands and a background cannot be combined (clear_background first)")
    return data


class Engine:
    """B200 evaluation engine for one model.  ``model`` may be a ``transformers`` Wav2Vec2ForCTC /
    Wav2Vec2ConformerForCTC / WavLMForCTC instance (what the reference builds at shap_calculation.py:218-219) or a
    plain ``state_dict`` with HF parameter names plus an explicit :class:`ModelConfig`."""

    def __init__(self, model, config: Optional[ModelConfig] = None, device: int = 0, max_batch: int = 0,
                 validate_gemm: bool = False, validate_attn: bool = False, preln_fp32: bool = False,
                 graphs: bool = True):
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device: the masked-coalition path has no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device)
        torch.cuda.set_device(self.device)
        if hasattr(model, "state_dict"):
            if config is None:
                config = ModelConfig.from_hf(model.config)
            sd = {k: v.detach() for k, v in model.state_dict().items()}
        else:
            if config is None:
                raise ValueError("a ModelConfig is required when passing a bare state_dict")
            sd = dict(model)
        self.config = config
        prefix = PREFIXES[config.kind]
        _fold_pos_conv(sd, prefix)
        keep = {}
        for k, v in sd.items():
            if not torch.is_floating_point(v):
                continue
            if "parametrizations" in k or k.endswith("weight_g") or k.endswith("weight_v"):
                continue
            if "quantizer" in k or "project_q" in k or "project_hid" in k or k.endswith("masked_spec_embed"):
                continue
            keep[k] = v.to(device=self.device, dtype=torch.float32).contiguous()
        cfg = _lib.W2SConfig()
        cfg.kind = KIND_IDS[config.kind]
        cfg.num_conv_layers = len(config.conv_dim)
        for i in range(len(config.conv_dim)):
            cfg.conv_dim[i] = config.conv_dim[i]
            cfg.conv_kernel[i] = config.conv_kernel[i]
            cfg.conv_stride[i] = config.conv_stride[i]
        cfg.conv_bias = int(config.conv_bias)
        cfg.feat_extract_norm = {"group": 0, "layer": 1}[config.feat_extract_norm]
        cfg.hidden_size = config.hidden_size
        cfg.num_hidden_layers = config.num_hidden_layers
        cfg.num_attention_heads = config.num_attention_heads
        cfg.intermediate_size = config.intermediate_size
        cfg.num_conv_pos_embeddings = config.num_conv_pos_embeddings
        cfg.num_conv_pos_embedding_groups = config.num_conv_pos_embedding_groups
        cfg.vocab_size = config.vocab_size
        cfg.layer_norm_eps = config.layer_norm_eps
        cfg.do_stable_layer_norm = int(config.do_stable_layer_norm)
        cfg.position_embeddings_type = {"relative": 1, "rotary": 2}.get(config.position_embeddings_type, 0) \
            if config.kind == "conformer" else 0
        cfg.conv_depthwise_kernel_size = config.conv_depthwise_kernel_size
        cfg.hidden_act = {"gelu": 0, "swish": 1, "silu": 1}[config.hidden_act]
        cfg.rotary_embedding_base = config.rotary_embedding_base
        cfg.num_buckets = config.num_buckets
        cfg.max_bucket_distance = config.max_bucket_distance
        cfg.max_batch = int(max_batch)
        cfg.flags = ((_lib.FLAG_VALIDATE_GEMM if validate_gemm else 0) | (_lib.FLAG_VALIDATE_ATTN if validate_attn else 0)
                     | (_lib.FLAG_FP32_PRELN if preln_fp32 else 0) | (0 if graphs else _lib.FLAG_NO_GRAPH))
        names = list(keep.keys())
        n = len(names)
        c_names = (C.c_char_p * n)(*[s.encode() for s in names])
        c_ptrs = (C.c_void_p * n)(*[keep[s].data_ptr() for s in names])
        c_num = (C.c_int64 * n)(*[keep[s].numel() for s in names])
        handle = C.c_void_p()
        rc = self.lib.w2s_create(C.byref(cfg), c_names, c_ptrs, c_num, n, device, C.byref(handle))
        if rc != 0:
            raise RuntimeError("w2s_create: " + self.lib.w2s_last_error(None).decode())
        self._h = handle
        self._cfg_struct = cfg
        self._pin_bits = None
        self._pin_event = torch.cuda.Event()
        self.max_batch = max_batch
        self.num_samples = 0
        self.num_segments = 0
        self.mode = "max"
        self.background_rows = 0
        self.background_weights = None
        self.num_bands = 0
        del keep

    # -- lifetime ----------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self.lib.w2s_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc != 0:
            raise RuntimeError(f"{what}: " + self.lib.w2s_last_error(self._h).decode())

    @staticmethod
    def _stream() -> int:
        return torch.cuda.current_stream().cuda_stream

    # -- state -------------------------------------------------------------------------------------
    def num_frames(self, num_samples: int) -> int:
        return int(self.lib.w2s_num_frames(self._h, int(num_samples)))

    def set_clip(self, x, num_segments: int = 1, bounds=None, baseline: float = 0.0):
        """x: normalised clip [L] (numpy or torch).  bounds: optional int32[M+1] segment boundaries."""
        xt = torch.as_tensor(x, dtype=torch.float32).reshape(-1).to(self.device).contiguous()
        L = xt.numel()
        if bounds is None:
            bounds = segment_bounds(L, num_segments)
        bounds = np.ascontiguousarray(bounds, dtype=np.int32)
        M = len(bounds) - 1
        self._check(self.lib.w2s_set_clip(self._h, xt.data_ptr(), L, bounds.ctypes.data_as(C.POINTER(C.c_int32)), M,
                                          float(baseline), self._stream()), "w2s_set_clip")
        self.num_samples, self.num_segments = L, M
        self.bounds = bounds

    def set_background(self, bg, weights=None):
        """Background dataset of ``shap.KernelExplainer(f, data)``: ``bg`` [B, L] (numpy or torch, the clip's normalised
        input space, L = the current clip's length) with ``weights`` [B] (default uniform; >= 0, positive sum).  Dropped
        segments of coalition k are then filled from each background row in turn, and ``eval_bits`` returns the weighted
        mean over the B rows (w2s_set_background).  The baseline of ``set_clip`` is ignored while a background is set."""
        data, w = background_arrays(bg, weights, num_samples=self.num_samples or None)
        if self.num_bands:
            raise ValueError("frequency bands are set: a background cannot be combined with them (clear_bands first)")
        bt = torch.as_tensor(data).to(device=self.device, dtype=torch.float32).contiguous()
        B, L = bt.shape
        self._check(self.lib.w2s_set_background(self._h, bt.data_ptr(), B, L, L, w.ctypes.data_as(C.POINTER(C.c_double)),
                                                self._stream()), "w2s_set_background")
        self.background_rows = B
        self.background_weights = w / w.sum()

    def clear_background(self):
        """Back to the baseline fill of ``set_clip`` (bit-identical to never having set a background)."""
        self._check(self.lib.w2s_set_background(self._h, None, 0, 0, 0, None, self._stream()), "w2s_set_background")
        self.background_rows = 0
        self.background_weights = None

    def set_bands(self, components):
        """Time-frequency cells (w2s_set_bands): ``components`` [F, L] are the clip's band components
        (preprocess.band_components; L = the current clip's length, 1 <= F <= 16, num_segments * F <= 2048).  Coalitions
        then have ``num_features`` = num_segments * F bits, bit s * F + b keeping cell (segment s, band b), and a row is the
        fp32 sum, in band order, of the kept cells' components.  The clip and the baseline are not read while bands are
        set; eval_waveforms and the gradient path ignore them."""
        data = band_arrays(components, self.num_samples or None, self.num_segments or None, self.background_rows)
        ct = torch.as_tensor(data).to(device=self.device, dtype=torch.float32).contiguous()
        F, L = ct.shape
        self._check(self.lib.w2s_set_bands(self._h, ct.data_ptr(), F, L, L, self._stream()), "w2s_set_bands")
        self.num_bands = F

    def clear_bands(self):
        """Back to time-only coalitions (bit-identical to never having set bands)."""
        self._check(self.lib.w2s_set_bands(self._h, None, 0, 0, 0, self._stream()), "w2s_set_bands")
        self.num_bands = 0

    @property
    def num_features(self) -> int:
        """Bits of one coalition row: num_segments, or num_segments * num_bands with time-frequency cells."""
        return self.num_segments * max(1, self.num_bands)

    def check_coalition_width(self, cols: int, packed: bool):
        """With bands set a coalition row must have num_features bits: a time-only row would be read as cells."""
        if not self.num_bands:
            return
        want = (self.num_features + 31) // 32 if packed else self.num_features
        if cols != want:
            raise ValueError(f"coalition rows have {cols} {'words' if packed else 'columns'}; with {self.num_segments} "
                             f"segments x {self.num_bands} bands they need {want}")

    def set_targets(self, mode: str = "max", frames=None, tokens=None):
        mid = _lib.MODE_IDS[mode]
        if mode in ("logit", "logprob"):
            f = np.ascontiguousarray(np.atleast_1d(frames), dtype=np.int32)
            t = np.ascontiguousarray(np.atleast_1d(tokens), dtype=np.int32)
            if f.shape != t.shape:
                raise ValueError("frames and tokens must have the same length")
            rc = self.lib.w2s_set_targets(self._h, f.ctypes.data_as(C.POINTER(C.c_int32)),
                                          t.ctypes.data_as(C.POINTER(C.c_int32)), int(f.size), mid, self._stream())
        else:
            rc = self.lib.w2s_set_targets(self._h, None, None, 0, mid, self._stream())
        self._check(rc, "w2s_set_targets")
        self.mode = mode

    def set_transcripts(self, transcripts, blank: int = PAD_ID, offsets=None):
        """Transcript-level output (w2s_set_transcripts): ``transcripts`` is a list of D label-id sequences (or, with
        ``offsets`` [D + 1], one flat label array).  Each evaluated row then yields D values, out[r, d] = log p_CTC(y_d |
        row r) = -WavXForCTC(x, labels=y_d).loss with ctc_loss_reduction="sum".  ``blank`` is the model's pad_token_id.
        Arguments are validated on the host before the library is called."""
        if offsets is not None:
            labels = np.ascontiguousarray(np.asarray(transcripts).reshape(-1), dtype=np.int32)
            offsets = check_offsets(offsets, labels.size)
            transcript_arrays([labels[a:b] for a, b in zip(offsets[:-1], offsets[1:])], blank, self.config.vocab_size)
        else:
            labels, offsets = transcript_arrays(transcripts, blank, self.config.vocab_size)
        self._check(self.lib.w2s_set_transcripts(self._h, labels.ctypes.data_as(C.POINTER(C.c_int32)),
                                                 offsets.ctypes.data_as(C.POINTER(C.c_int32)), len(offsets) - 1, int(blank),
                                                 self._stream()), "w2s_set_transcripts")
        self.mode = "transcript"
        self.transcripts = [labels[a:b].copy() for a, b in zip(offsets[:-1], offsets[1:])]
        self.blank = int(blank)

    def out_width(self, num_samples: Optional[int] = None) -> int:
        return int(self.lib.w2s_out_width(self._h, int(num_samples or self.num_samples)))

    # -- evaluation (device buffers) ------------------------------------------------------------------
    def eval_bits(self, zbits: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """zbits: int32/uint32 device tensor [K, ceil(M/32)] -> float32 device tensor [K, width]."""
        K = zbits.shape[0]
        self.check_coalition_width(zbits.shape[-1], packed=True)
        width = self.out_width()
        if out is None:
            out = torch.empty((K, width), dtype=torch.float32, device=self.device)
        self._check(self.lib.w2s_eval(self._h, zbits.data_ptr(), K, out.data_ptr(), self._stream()), "w2s_eval")
        return out

    def eval_waveforms(self, x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """x: float32 device tensor [n, L] (last dim contiguous) -> float32 device tensor [n, width]."""
        if x.dim() != 2 or x.stride(1) != 1 or x.dtype != torch.float32 or not x.is_cuda:
            raise ValueError("expected a float32 CUDA tensor [n, L] with contiguous rows")
        n, L = x.shape
        width = self.out_width(L)
        if out is None:
            out = torch.empty((n, width), dtype=torch.float32, device=self.device)
        self._check(self.lib.w2s_eval_waveforms(self._h, x.data_ptr(), n, L, x.stride(0), out.data_ptr(),
                                                self._stream()), "w2s_eval_waveforms")
        return out

    # -- input gradients (expected-gradients path) ----------------------------------------------------------
    def grad_waveforms(self, x: torch.Tensor, frames):
        """x: float32 device tensor [n, L]; frames: one output frame per row -> (grad [n, L] float32 device tensor of
        d out[r] / d x[r], out [n]) with out[r] = max_v logits[r, frames[r], v] -- the scalar the reference's
        GradientExplainer differentiates through ModelWrapper (shap_calculation.py:50, :133, :162)."""
        if x.dim() != 2 or x.stride(1) != 1 or x.dtype != torch.float32 or not x.is_cuda:
            raise ValueError("expected a float32 CUDA tensor [n, L] with contiguous rows")
        n, L = x.shape
        f = np.ascontiguousarray(np.broadcast_to(np.asarray(frames, dtype=np.int32), (n,)))
        grad = torch.empty((n, L), dtype=torch.float32, device=self.device)
        out = torch.empty((n,), dtype=torch.float32, device=self.device)
        self._check(self.lib.w2s_grad_waveforms(self._h, x.data_ptr(), n, L, x.stride(0),
                                                f.ctypes.data_as(C.POINTER(C.c_int32)), grad.data_ptr(), out.data_ptr(),
                                                self._stream()), "w2s_grad_waveforms")
        return grad, out

    def grad_transcripts(self, x: torch.Tensor, which):
        """x: float32 device tensor [n, L]; which: one transcript index per row (of the last ``set_transcripts``) ->
        (grad [n, L], out [n]) with out[r] = log p_CTC(y_which[r] | x[r]) and grad[r] = d out[r] / d x[r]."""
        if x.dim() != 2 or x.stride(1) != 1 or x.dtype != torch.float32 or not x.is_cuda:
            raise ValueError("expected a float32 CUDA tensor [n, L] with contiguous rows")
        n, L = x.shape
        w = np.ascontiguousarray(np.broadcast_to(np.asarray(which, dtype=np.int32), (n,)))
        grad = torch.empty((n, L), dtype=torch.float32, device=self.device)
        out = torch.empty((n,), dtype=torch.float32, device=self.device)
        self._check(self.lib.w2s_grad_transcripts(self._h, x.data_ptr(), n, L, x.stride(0),
                                                  w.ctypes.data_as(C.POINTER(C.c_int32)), grad.data_ptr(), out.data_ptr(),
                                                  self._stream()), "w2s_grad_transcripts")
        return grad, out

    def vjp_waveforms(self, x: torch.Tensor, gout: torch.Tensor) -> torch.Tensor:
        """Vector-Jacobian product of ModelWrapper's output [n, T'] (max logit per frame) w.r.t. the waveforms:
        gout [n, T'] float32 device tensor -> grad [n, L]."""
        if x.dim() != 2 or x.stride(1) != 1 or x.dtype != torch.float32 or not x.is_cuda:
            raise ValueError("expected a float32 CUDA tensor [n, L] with contiguous rows")
        n, L = x.shape
        gout = gout.to(device=self.device, dtype=torch.float32).contiguous()
        if tuple(gout.shape) != (n, self.num_frames(L)):
            raise ValueError(f"upstream gradient must be [n, T'] = {(n, self.num_frames(L))}, got {tuple(gout.shape)}")
        grad = torch.empty((n, L), dtype=torch.float32, device=self.device)
        self._check(self.lib.w2s_vjp_waveforms(self._h, x.data_ptr(), n, L, x.stride(0), gout.data_ptr(), grad.data_ptr(),
                                               None, self._stream()), "w2s_vjp_waveforms")
        return grad

    def grad_debug(self, snapshots: bool = True, simt_attention: bool = False, unfused_attention: bool = False):
        """Test hooks: keep per-stage snapshots (grad_peek); run attention backward on the CUDA-core cross-check kernels, or
        as batched tensor-core contractions + row kernels, instead of the fused tcgen05 kernel."""
        self.lib.w2s_grad_debug(self._h, int(bool(snapshots)) | (2 if simt_attention else 0) | (4 if unfused_attention else 0))

    GRAD_TILE_ROWS = 32       # rows per device tile of grad_waveforms (paired rows must fit one tile)

    def grad_rules(self, rescale_silu: bool = False, glu_placeholder: bool = False):
        """DeepLIFT handler rules of feasability_tests/custom_shap_handlers.py for the following grad_waveforms calls, whose
        rows must then be [explained | reference] halves (even count, at most GRAD_TILE_ROWS); both False: plain gradient."""
        self._check(self.lib.w2s_grad_rules(self._h, (1 if rescale_silu else 0) | (2 if glu_placeholder else 0)), "w2s_grad_rules")

    def grad_peek(self, name: str, shape, dtype=torch.float32) -> torch.Tensor:
        """Snapshot of an intermediate gradient of the last grad_waveforms call (tests; needs grad_debug(True))."""
        out = torch.empty(shape, dtype=dtype, device=self.device)
        got = self.lib.w2s_grad_peek(self._h, name.encode(), out.data_ptr(), out.numel() * out.element_size(), self._stream())
        if got != out.numel() * out.element_size():
            raise RuntimeError(f"w2s_grad_peek('{name}'): got {got} bytes for a buffer of {out.numel() * out.element_size()}")
        return out

    def mask(self, zbits: torch.Tensor) -> torch.Tensor:
        """The rows ``eval_bits`` evaluates: [K, L], or [K * B, L] (row k * B + b) with a background."""
        K = zbits.shape[0]
        self.check_coalition_width(zbits.shape[-1], packed=True)
        out = torch.empty((K * max(1, self.background_rows), self.num_samples), dtype=torch.float32, device=self.device)
        self._check(self.lib.w2s_mask(self._h, zbits.data_ptr(), K, out.data_ptr(), self._stream()), "w2s_mask")
        return out

    def wls(self, zbits: torch.Tensor, weights: torch.Tensor, y: torch.Tensor, fx: torch.Tensor,
            fnull: torch.Tensor, num_features: int):
        """Device KernelSHAP solve -> (phi[M, D] float64 device tensor, status int)."""
        K, D = y.shape
        phi = torch.empty((num_features, D), dtype=torch.float64, device=self.device)
        status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._check(self.lib.w2s_wls(self._h, zbits.data_ptr(), weights.data_ptr(), y.data_ptr(), K, num_features, D,
                                     fx.data_ptr(), fnull.data_ptr(), phi.data_ptr(), status.data_ptr(),
                                     self._stream()), "w2s_wls")
        return phi, status

    # -- convenience (host buffers) ---------------------------------------------------------------------
    def bits_to_device(self, Z) -> torch.Tensor:
        """Host {0,1} matrix [K, M] (or already packed uint32 words [K, ceil(M/32)]) -> device int32 words.  The
        pinned staging buffer is owned by the engine and re-used (grown geometrically) across calls."""
        Z = np.asarray(Z)
        self.check_coalition_width(Z.shape[-1], packed=Z.dtype == np.uint32)
        words = (Z if Z.dtype == np.uint32 else pack_coalitions(Z)).view(np.int32)
        n = words.size
        if self._pin_bits is None or self._pin_bits.numel() < n:
            self._pin_bits = torch.empty(max(n, 2 * (self._pin_bits.numel() if self._pin_bits is not None else 0)),
                                         dtype=torch.int32).pin_memory()
        else:
            # the previous upload from this buffer must have left the host before it is overwritten
            self._pin_event.synchronize()
        stage = self._pin_bits[:n].view(words.shape)
        stage.numpy()[...] = words
        dev = stage.to(self.device, non_blocking=True)
        self._pin_event.record(torch.cuda.current_stream())
        return dev

    def launch_count(self) -> int:
        """Kernel launches issued by eval_bits / eval_waveforms on this engine so far (counted in the library)."""
        return int(self.lib.w2s_launch_count(self._h))

    def flops_per_forward(self, num_samples: Optional[int] = None) -> float:
        return float(self.lib.w2s_flops_per_forward(self._h, int(num_samples or self.num_samples)))

    def profile(self, on: bool):
        self.lib.w2s_profile_enable(self._h, int(on))

    def profile_read(self):
        """-> {launch class: dict(ms, flops, bytes, launches)} accumulated since profile(True)."""
        cap, nmax = 1 << 16, 256
        names = C.create_string_buffer(cap)
        ms = (C.c_double * nmax)()
        fl = (C.c_double * nmax)()
        by = (C.c_double * nmax)()
        cn = (C.c_int64 * nmax)()
        n = self.lib.w2s_profile_read(self._h, names, cap, ms, fl, by, cn, nmax)
        if n < 0:
            raise RuntimeError("w2s_profile_read: buffer too small")
        keys = names.value.decode().split("\n")[:n]
        return {k: dict(ms=ms[i], flops=fl[i], bytes=by[i], launches=cn[i]) for i, k in enumerate(keys)}

    def kernel_count(self):
        a, b = C.c_int64(), C.c_int64()
        self.lib.w2s_kernel_count(self._h, C.byref(a), C.byref(b))
        return int(a.value), int(b.value)


def debug_gemm(a: torch.Tensor, w: torch.Tensor, bias=None, act: int = 0, out_fp32: bool = True, tcgen05: bool = True,
               residual=None, alpha: float = 1.0, accumulate_into=None):
    """out[M, N] = act(a[M, K] @ w[N, K]^T + bias) * alpha + residual through the library's contraction kernels
    (tests only).  ``accumulate_into`` (fp32 [M, N]): in-place accumulation, residual == out -- the case the CTA-pair
    kernel serves with TMA reduce-add."""
    lib = _lib.load()
    M, K = a.shape
    N = w.shape[0]
    if accumulate_into is not None:
        out, residual, out_fp32 = accumulate_into, accumulate_into, True
    else:
        out = torch.empty((M, N), dtype=torch.float32 if out_fp32 else torch.bfloat16, device=a.device)
    rc = lib.w2s_debug_gemm(int(tcgen05), a.data_ptr(), w.data_ptr(), bias.data_ptr() if bias is not None else None,
                            residual.data_ptr() if residual is not None else None,
                            int(residual is not None and residual.dtype == torch.float32), float(alpha),
                            out.data_ptr(), M, N, K, act, int(out_fp32), torch.cuda.current_stream().cuda_stream)
    if rc != 0:
        raise RuntimeError("w2s_debug_gemm: " + lib.w2s_last_error(None).decode())
    return out


def _check_buffer(name: str, t: torch.Tensor, dtype: torch.dtype, numel: int):
    if t.dtype != dtype or not t.is_cuda or not t.is_contiguous() or t.numel() < numel:
        raise ValueError(f"{name}: need a contiguous {dtype} CUDA tensor of at least {numel} elements")


def debug_attention(qkv: torch.Tensor, B: int, heads: int, pos_proj=None, scale: float = 0.125, tcgen05: bool = True,
                    with_lse: bool = False, ctx=None, lse=None):
    """Self-attention of one layer through the library's kernels (tests only): qkv [B*T, 3H] (q | k | v) or, with pos_proj
    [2T-1, H], [B*T, 4H] (q+u | q+v | k | v), bf16, H = 64 * heads.  tcgen05: the tensor-core kernel (attention_fa, or
    attention_rel with pos_proj), else the CUDA-core validation kernel.  Returns (ctx [B*T, H] bf16, lse [B, heads, T] fp32
    log2-domain log-sum-exp or None); ``ctx`` / ``lse`` may be caller buffers (at least that many elements)."""
    lib = _lib.load()
    H = 64 * heads
    T = qkv.shape[0] // B
    _check_buffer("qkv", qkv, torch.bfloat16, B * T * (4 if pos_proj is not None else 3) * H)
    if qkv.shape != (B * T, (4 if pos_proj is not None else 3) * H):
        raise ValueError(f"qkv: shape {tuple(qkv.shape)} does not fit B={B}, heads={heads}")
    if pos_proj is not None:
        _check_buffer("pos_proj", pos_proj, torch.bfloat16, (2 * T - 1) * H)
    if ctx is None:
        ctx = torch.empty((B * T, H), dtype=torch.bfloat16, device=qkv.device)
    _check_buffer("ctx", ctx, torch.bfloat16, B * T * H)
    if lse is None and with_lse:
        lse = torch.empty((B, heads, T), dtype=torch.float32, device=qkv.device)
    if lse is not None:
        _check_buffer("lse", lse, torch.float32, B * heads * T)
    rc = lib.w2s_debug_attention(int(tcgen05), qkv.data_ptr(), pos_proj.data_ptr() if pos_proj is not None else None,
                                 B, T, heads, float(scale), ctx.data_ptr(), lse.data_ptr() if lse is not None else None,
                                 torch.cuda.current_stream().cuda_stream)
    if rc != 0:
        raise RuntimeError("w2s_debug_attention: " + lib.w2s_last_error(None).decode())
    return ctx, lse


def debug_attention_bias(qkv: torch.Tensor, B: int, heads: int, rel_bias: torch.Tensor, gate: torch.Tensor,
                         scale: float = 0.125, tcgen05: bool = True, ctx=None, lse=None):
    """`debug_attention` with WavLM's gated relative-position bias (tests only): score[b, h, i, j] += gate[b, h, i] *
    rel_bias[h, T - 1 + j - i], with rel_bias [heads, 2T-1] and gate [B, heads, T] fp32 in natural units.  The bias
    variant writes no log-sum-exp: passing ``lse`` raises.  Returns ctx [B*T, H] bf16 (``ctx`` may be a caller buffer)."""
    lib = _lib.load()
    H = 64 * heads
    T = qkv.shape[0] // B
    _check_buffer("qkv", qkv, torch.bfloat16, B * T * 3 * H)
    if qkv.shape != (B * T, 3 * H):
        raise ValueError(f"qkv: shape {tuple(qkv.shape)} does not fit B={B}, heads={heads}")
    _check_buffer("rel_bias", rel_bias, torch.float32, heads * (2 * T - 1))
    _check_buffer("gate", gate, torch.float32, B * heads * T)
    if ctx is None:
        ctx = torch.empty((B * T, H), dtype=torch.bfloat16, device=qkv.device)
    _check_buffer("ctx", ctx, torch.bfloat16, B * T * H)
    rc = lib.w2s_debug_attention_bias(int(tcgen05), qkv.data_ptr(), rel_bias.data_ptr(), gate.data_ptr(), B, T, heads,
                                      float(scale), ctx.data_ptr(), lse.data_ptr() if lse is not None else None,
                                      torch.cuda.current_stream().cuda_stream)
    if rc != 0:
        raise RuntimeError("w2s_debug_attention_bias: " + lib.w2s_last_error(None).decode())
    return ctx


def debug_ctc(logits: torch.Tensor, transcripts, blank: int = PAD_ID, which=None, grad: bool = False):
    """The library's CTC code on caller logits (tests only): logits fp32 [n, T, V] (CUDA) -> out [n, D] =
    log p_CTC(y_d | logits[r]) through the head reduction kernel; with ``grad``, also d out[r, which[r]] / d logits[r] as
    [n, T, V] from the gradient seed kernel (``which`` defaults to 0 for every row)."""
    lib = _lib.load()
    n, T, V = logits.shape
    _check_buffer("logits", logits, torch.float32, n * T * V)
    labels, offsets = transcript_arrays(transcripts, blank, V)
    D = len(offsets) - 1
    out = torch.empty((n, D), dtype=torch.float32, device=logits.device)
    dl = torch.empty((n, T, V), dtype=torch.float32, device=logits.device) if grad else None
    w = np.ascontiguousarray(np.broadcast_to(np.asarray(0 if which is None else which, dtype=np.int32), (n,)))
    rc = lib.w2s_debug_ctc(logits.data_ptr(), n, T, V, V, labels.ctypes.data_as(C.POINTER(C.c_int32)),
                           offsets.ctypes.data_as(C.POINTER(C.c_int32)), D, int(blank), w.ctypes.data_as(C.POINTER(C.c_int32)),
                           out.data_ptr(), dl.data_ptr() if dl is not None else None, torch.cuda.current_stream().cuda_stream)
    if rc != 0:
        raise RuntimeError("w2s_debug_ctc: " + lib.w2s_last_error(None).decode())
    return (out, dl) if grad else out


def relative_buckets(T: int, num_buckets: int = 320, max_distance: int = 800) -> np.ndarray:
    """WavLM's relative-position buckets for a clip of T frames as the library computes them (host, no device):
    int32 [2T-1], entry r for relative position r - (T - 1)."""
    lib = _lib.load()
    out = np.empty(2 * T - 1, dtype=np.int32)
    if lib.w2s_relative_buckets(int(T), int(num_buckets), int(max_distance), out.ctypes.data) != 0:
        raise ValueError("w2s_relative_buckets: bad argument")
    return out


def debug_attention_bwd(qkv: torch.Tensor, dctx: torch.Tensor, B: int, heads: int, ctx=None, lse=None, scale: float = 0.125,
                        tcgen05: bool = True, dqkv=None):
    """Backward of `debug_attention` without relative positions (tests only): d ctx [B*T, H] -> dqkv [B*T, 3H] bf16.
    tcgen05: the gradient path's fused kernel, which needs the forward's ``ctx`` and ``lse``; else the CUDA-core
    cross-check kernels.  ``dqkv`` may be a caller buffer."""
    lib = _lib.load()
    H = 64 * heads
    T = qkv.shape[0] // B
    _check_buffer("qkv", qkv, torch.bfloat16, B * T * 3 * H)
    if qkv.shape != (B * T, 3 * H):
        raise ValueError(f"qkv: shape {tuple(qkv.shape)} does not fit B={B}, heads={heads}")
    _check_buffer("dctx", dctx, torch.bfloat16, B * T * H)
    if tcgen05:
        if ctx is None or lse is None:
            raise ValueError("the fused backward needs the forward's ctx and lse")
        _check_buffer("ctx", ctx, torch.bfloat16, B * T * H)
        _check_buffer("lse", lse, torch.float32, B * heads * T)
    if dqkv is None:
        dqkv = torch.empty((B * T, 3 * H), dtype=torch.bfloat16, device=qkv.device)
    _check_buffer("dqkv", dqkv, torch.bfloat16, B * T * 3 * H)
    rc = lib.w2s_debug_attention_bwd(int(tcgen05), qkv.data_ptr(), ctx.data_ptr() if ctx is not None else None,
                                     dctx.data_ptr(), lse.data_ptr() if lse is not None else None, B, T, heads, float(scale),
                                     dqkv.data_ptr(), torch.cuda.current_stream().cuda_stream)
    if rc != 0:
        raise RuntimeError("w2s_debug_attention_bwd: " + lib.w2s_last_error(None).decode())
    return dqkv
