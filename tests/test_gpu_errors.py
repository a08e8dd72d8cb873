"""GPU: the recognition-error output W2S_OUT_ERRORS, out[r, d] = the edit distance between row r's greedy transcript and
reference d, in labels or words.

Every comparison is exact: the output is a count computed by integer and compare operations from the row's logits, so
the device must reproduce the oracle (oracle/errors_ref.py) applied to the same fp32 logits bit for bit.

Kernel level: w2s_debug_errors on designed logits -- hypotheses that are edits of the references, exact ties inside a
lane (ids v and v + 32) and across lanes, all-blank rows, delimiter runs at both ends, hypothesis words longer than every
reference word, reference words that are permutations and prefixes of each other, and reference lengths on both sides of
every 32-unit boundary.  These cases catch, among others, the highest id winning a tie, blanks dropped before repeats are
collapsed, empty words counted, and an off-by-one in the cross-lane carry or shift.

Model level: w2s_eval in errors mode against the oracle on the same rows' W2S_OUT_LOGITS output; tile independence; the
background mean; bands; and the decoded labels against the transformers fp32 forward on rows whose every frame's top-2
margin exceeds twice the measured logit deviation, where the argmax cannot differ.
"""
import numpy as np
import pytest
import torch

from helpers import VARIANTS, build_model
from oracle import background_ref as BR
from oracle import callback as CB
from oracle import errors_ref as ER
from oracle.kernelshap_ref import brute_force_shapley
from oracle.make_golden_wavlm import VARIANTS as WAVLM_VARIANTS, build as build_wavlm
from shap_transformer_asr_b200 import metrics
from shap_transformer_asr_b200.targets import greedy_transcript, reference_length
from test_gpu_background import host_bg_mean

pytestmark = pytest.mark.gpu

DELIM = 4


@pytest.fixture(scope="module")
def P():
    import shap_transformer_asr_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


def fast_levenshtein(a, b):
    """ER.levenshtein with each DP row in numpy (the long cases have 512 x 1031 cells)"""
    b = np.asarray([hash(v) for v in b], dtype=np.int64)
    prev = np.arange(len(b) + 1)
    ar = np.arange(len(b) + 1)
    for i, x in enumerate(a, 1):
        cur = np.empty_like(prev)
        cur[0] = i
        cur[1:] = np.minimum(prev[1:] + 1, prev[:-1] + (b != hash(x)))
        prev = np.minimum.accumulate(cur - ar) + ar
    return int(prev[-1])


def oracle(logits, refs, unit, blank, delim=DELIM):
    out = np.zeros((logits.shape[0], len(refs)))
    for r in range(logits.shape[0]):
        hyp = ER.greedy_ids(logits[r], blank)
        for d, y in enumerate(refs):
            a, b = (hyp, y) if unit == "labels" else (ER.split_words(hyp, delim), ER.split_words(y, delim))
            out[r, d] = fast_levenshtein(a, b)
    return out


def test_fast_levenshtein_is_the_oracle():
    rng = np.random.default_rng(0)
    for _ in range(200):
        a, b = list(rng.integers(0, 4, rng.integers(0, 12))), list(rng.integers(0, 4, rng.integers(0, 12)))
        assert fast_levenshtein(a, b) == ER.levenshtein(a, b)


# ---------------------------------------------------------------------------------------------------------------------
# kernel level
# ---------------------------------------------------------------------------------------------------------------------
def word_ref(words, delim=DELIM, lead=0, trail=0):
    out = [delim] * lead
    for i, w in enumerate(words):
        out += list(w) + ([delim] if i + 1 < len(words) else [])
    return out + [delim] * trail


def make_refs(rng, V, blank, unit):
    """references of 0 .. 512 labels; in words, word counts on both sides of 32 and 64, permutations and prefixes"""
    letters = [v for v in range(V) if v not in (blank, DELIM)]
    refs = []
    for U in (0, 1, 31, 32, 33, 63, 64, 65, 511, 512):
        if unit == "labels":
            refs.append([int(v) for v in rng.choice(letters[:6] + [DELIM], U)])
    if unit == "words":
        a, b, c = letters[0], letters[1], letters[2]
        refs.append(word_ref([(a, b), (b, a), (a, b, c), (a,), (a, b)], lead=2, trail=3))   # permutations, prefixes
        for n in (1, 31, 32, 33, 63, 64, 65, 256):          # 256 one-letter words: 511 labels
            refs.append(word_ref([tuple(int(v) for v in rng.choice(letters[:4], rng.integers(1, 3 if n < 256 else 2)))
                                  for _ in range(n)]))
        refs.append([])
        refs.append([DELIM] * 5)                                                                # no words at all
        refs.append(word_ref([tuple(int(v) for v in rng.choice(letters[:5], 120)) for _ in range(4)]))  # 4 words, 483 labels
    return refs


def frames_for(seq, T, blank, rng):
    """a frame labelling whose greedy decode is seq (repeats broken by blanks, random extra repeats and blanks),
    truncated or blank-padded to T frames"""
    fr = []
    for i, v in enumerate(seq):
        if fr and fr[-1] == v:
            fr.append(blank)
        fr += [v] * int(rng.integers(1, 3))
        if rng.random() < 0.3:
            fr.append(blank)
    fr = fr[:T]
    return fr + [blank] * (T - len(fr))


def design_rows(rng, T, V, blank, refs, n):
    letters = [v for v in range(V) if v not in (blank, DELIM)]
    rows = []
    for r in range(n):
        kind = r % 6
        if kind == 0:       # an edited reference
            y = list(refs[r % len(refs)])
            for _ in range(int(rng.integers(0, 6))):
                i = int(rng.integers(0, len(y) + 1))
                if rng.random() < 0.4 and i < len(y):
                    del y[i]
                else:
                    y.insert(i, int(rng.choice(letters[:6] + [DELIM])))
            fr = frames_for(y, T, blank, rng)
        elif kind == 1:     # all blank
            fr = [blank] * T
        elif kind == 2:     # delimiter runs at the start and the end around words
            fr = frames_for([DELIM] * 3 + word_ref([(letters[0], letters[1]), (letters[1], letters[0])]) + [DELIM] * 4,
                            T, blank, rng)
        elif kind == 3:     # one hypothesis word longer than every reference word
            fr = frames_for([letters[i % 3] for i in range(T)], T, blank, rng)
        else:               # random frames from a small alphabet with the blank and the delimiter
            fr = [int(v) for v in rng.choice(letters[:4] + [blank, blank, DELIM], T)]
        rows.append(fr)
    z = (0.5 * rng.standard_normal((n, T, V))).astype(np.float32)
    for r, fr in enumerate(rows):
        z[r, np.arange(T), fr] = 4.0
        for t in range(T):
            u = rng.random()
            if u < 0.15:                        # exact tie inside a lane: v and v +- 32 (or the wrap of the block)
                z[r, t, (fr[t] + 32) % V] = 4.0
            elif u < 0.3:                       # exact tie across lanes, lower or higher id
                z[r, t, int(rng.integers(0, V))] = 4.0
    return z


KERNEL_T = [1, 2, 31, 32, 33, 249, 1031]


@pytest.mark.parametrize("T", KERNEL_T)
@pytest.mark.parametrize("V,blank", [(32, 0), (33, 7), (128, 0), (128, 77)])
@pytest.mark.parametrize("unit", ["labels", "words"])
def test_debug_errors_equal_the_oracle(P, T, V, blank, unit):
    rng = np.random.default_rng([T, V, blank, unit == "words"])
    refs = make_refs(rng, V, blank, unit)
    n = 30
    z = design_rows(rng, T, V, blank, refs, n)
    zt = torch.from_numpy(z).cuda()
    want = oracle(z, refs, unit, blank)
    got = np.concatenate([P.debug_errors(zt, refs[d0:d0 + 8], unit=unit, blank=blank).cpu().numpy()
                          for d0 in range(0, len(refs), 8)], axis=1)               # D up to 8 per call
    bad = np.argwhere(got != want)
    assert bad.size == 0, (bad[:5].tolist(), got[tuple(bad[0])], want[tuple(bad[0])], len(refs[bad[0][1]]))
    # the value of a row does not depend on its position or on the other references
    one = P.debug_errors(zt[5:6].contiguous(), [refs[-1]], unit=unit, blank=blank).cpu().numpy()
    assert one[0, 0] == want[5, -1]
    print(f"T={T} V={V} blank={blank} {unit}: {len(refs)} references, errors range [{want.min():.0f}, {want.max():.0f}]")


def test_debug_errors_refuses_bad_arguments(P):
    z = torch.zeros((1, 4, 32), device="cuda")
    with pytest.raises(ValueError, match="delimiter"):
        P.debug_errors(z, [[5]], unit="words", delimiter=0)
    with pytest.raises(ValueError, match="at most 512"):
        P.debug_errors(z, [[5] * 513])


# ---------------------------------------------------------------------------------------------------------------------
# model level
# ---------------------------------------------------------------------------------------------------------------------
def _model(name):
    if name in WAVLM_VARIANTS:
        cfg = WAVLM_VARIANTS[name]
        return build_wavlm(cfg), cfg
    return build_model(VARIANTS[name]), VARIANTS[name]


def _refs(lg, V):
    """the greedy transcript of one row, an edit of it with a word boundary, a fixed one and the empty one"""
    g = greedy_transcript(lg).tolist()
    return [g, g[:len(g) // 2] + [DELIM, 5, 6] + g[len(g) // 2:], [5, 6, DELIM, 7, DELIM, DELIM, 5, 6], []]


@pytest.mark.parametrize("name,validate", [("tiny_group", False), ("tiny_layer_stable", False),
                                           ("tiny_conformer_rel", False), ("tiny_wavlm", False), ("tiny_group", True)])
def test_eval_errors_equal_the_oracle_on_the_engines_own_logits(P, name, validate):
    model, cfg = _model(name)
    L, M = 9000, 12
    eng = P.Engine(model, cfg, max_batch=16, validate_gemm=validate, validate_attn=validate)
    eng.set_clip(P.synthetic_clip(L), num_segments=M)
    Z, _, _ = P.sample_coalitions(M, 40, seed=1)
    bits = eng.bits_to_device(np.concatenate([np.ones((1, M), np.uint8), Z]))
    T, V = cfg.num_frames(L), cfg.vocab_size
    eng.set_targets("logits")
    own = eng.eval_bits(bits).view(-1, T, V).cpu().numpy()
    refs = _refs(own[0], V)
    for unit in ("labels", "words"):
        eng.set_references(refs, unit=unit)
        assert eng.out_width() == len(refs)
        got = eng.eval_bits(bits).cpu().numpy()
        want = oracle(own, refs, unit, 0)
        assert np.array_equal(got, want), (unit, np.argwhere(got != want)[:5].tolist())
        assert got[0, 0] == 0
        print(f"{name} validate={validate} {unit}: errors range [{want.min():.0f}, {want.max():.0f}] over {len(own)} rows")
    eng.close()


def test_errors_are_bit_identical_across_tiles(P):
    model, cfg = _model("tiny_group")
    L = 9000
    x = torch.from_numpy(np.random.default_rng(1).standard_normal((37, L)).astype(np.float32)).cuda()
    refs = [[5, 6, DELIM, 7], [], [8] * 40]
    outs = []
    for mb in (7, 32, 0):
        eng = P.Engine(model, cfg, max_batch=mb)
        eng.set_references(refs, unit="labels")
        a = eng.eval_waveforms(x).clone()
        b = eng.eval_waveforms(x).clone()
        alone = eng.eval_waveforms(x[11:12].contiguous())
        torch.cuda.synchronize()
        assert torch.equal(a, b) and torch.equal(alone[0], a[11])
        outs.append(a.cpu())
        eng.close()
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


def test_background_errors_mean_equals_the_host_replay(P):
    model, cfg = _model("tiny_group")
    L, M = 12000, 10
    eng = P.Engine(model, cfg, max_batch=16)
    clip = P.synthetic_clip(L)
    eng.set_clip(clip, num_segments=M)
    eng.set_targets("logits")
    lg = eng.eval_bits(eng.bits_to_device(np.ones((1, M), np.uint8))).view(-1, cfg.vocab_size).cpu().numpy()
    refs = [greedy_transcript(lg).tolist(), [5, 6, DELIM, 7]]
    eng.set_references(refs, unit="words")
    Z, _, _ = P.sample_coalitions(M, 30, seed=0)
    bits = eng.bits_to_device(Z)
    B = 3
    bg = P.make_background(L, B, seed=5)
    bounds = CB.segment_bounds(L, M)
    per_row = []
    for b in range(B):
        eng.set_background(bg[b:b + 1])
        fused = eng.eval_bits(bits).clone()
        explicit = eng.eval_waveforms(torch.from_numpy(BR.materialize_background(clip, Z, bounds, bg[b:b + 1])).cuda())
        torch.cuda.synchronize()
        assert torch.equal(fused, explicit)
        per_row.append(explicit.cpu().numpy())
    w = np.array([0.5, 2.0, 1.0])
    eng.set_background(bg, w)
    y = eng.eval_bits(bits).cpu().numpy()
    rows = np.stack(per_row, axis=1).reshape(-1, y.shape[1])
    assert np.array_equal(y, host_bg_mean(rows, (w / w.sum()).astype(np.float32), B))
    eng.close()


def test_errors_with_bands_equal_the_oracle(P):
    model, cfg = _model("tiny_group")
    L, M, F = 9000, 6, 3
    eng = P.Engine(model, cfg, max_batch=16)
    clip = P.synthetic_clip(L)
    eng.set_clip(clip, num_segments=M)
    eng.set_bands(P.band_components(clip, P.mel_band_edges(F)))
    Z, _, _ = P.sample_coalitions(M * F, 30, seed=2)
    bits = eng.bits_to_device(Z)
    T, V = cfg.num_frames(L), cfg.vocab_size
    eng.set_targets("logits")
    own = eng.eval_bits(bits).view(-1, T, V).cpu().numpy()
    refs = _refs(own[0], V)
    eng.set_references(refs, unit="words")
    got = eng.eval_bits(bits).cpu().numpy()
    assert np.array_equal(got, oracle(own, refs, "words", 0))
    eng.close()


def test_decoded_labels_agree_with_transformers_where_the_margin_allows(P):
    model, cfg = _model("tiny_group")
    L, n = 3000, 48
    x = np.random.default_rng(3).standard_normal((n, L)).astype(np.float32)
    with torch.no_grad():
        hf = model(torch.from_numpy(x)).logits.numpy()
    eng = P.Engine(model, cfg, max_batch=8)
    xt = torch.from_numpy(x).cuda()
    eng.set_targets("logits")
    own = eng.eval_waveforms(xt).view(hf.shape).cpu().numpy()
    refs = [greedy_transcript(hf[0]).tolist(), []]
    eng.set_references(refs, unit="labels")
    got = eng.eval_waveforms(xt).cpu().numpy()
    srt = np.sort(hf, -1)
    margin = srt[..., -1] - srt[..., -2]                          # [n, T']
    dev = np.abs(own - hf).max(axis=(1, 2))                       # measured deviation per row
    ok = np.all(margin > 2 * dev[:, None], axis=1)
    print(f"transformers parity: {ok.sum()} of {n} rows with every frame's top-2 margin above 2 x the row's deviation "
          f"(max deviation {dev.max():.3g})")
    assert ok.sum() >= 1
    for r in np.nonzero(ok)[0]:
        assert ER.greedy_ids(own[r]) == ER.greedy_ids(hf[r])
    assert np.array_equal(got[ok], oracle(hf[ok], refs, "labels", 0))
    eng.close()


def test_references_and_transcripts_are_kept_apart(P):
    """w2s_set_references selects the errors mode without touching the transcripts: w2s_grad_transcripts still uses the
    transcripts last set by w2s_set_transcripts, and refuses to run when only references were set."""
    model, cfg = _model("tiny_group")
    L = 9000
    x = torch.from_numpy(np.random.default_rng(4).standard_normal((2, L)).astype(np.float32)).cuda()
    eng = P.Engine(model, cfg, max_batch=4)
    eng.set_references([[5, 6]], unit="labels")
    with pytest.raises(RuntimeError, match="no transcripts set"):
        eng.grad_transcripts(x, [0, 0])
    eng.set_transcripts([[7, 8]])
    _, want = eng.grad_transcripts(x, [0, 0])
    eng.set_references([[5, 6, 6, 6], [9]], unit="labels")
    assert eng.out_width(L) == 2
    _, got = eng.grad_transcripts(x, [0, 0])
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    with pytest.raises(RuntimeError, match="transcript index 1"):
        eng.grad_transcripts(x, [0, 1])
    # w2s_set_targets still refuses the errors mode
    assert eng.lib.w2s_set_targets(eng._h, None, None, 0, 6, eng._stream()) != 0
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------
# KernelSHAP
# ---------------------------------------------------------------------------------------------------------------------
def test_full_enumeration_errors_kernelshap_equals_brute_force_of_the_device_game(P):
    model, cfg = _model("tiny_group")
    L, M = 12000, 10
    clip = P.synthetic_clip(L)
    eng = P.Engine(model, cfg, max_batch=64)
    res = P.KernelShapExplainer(eng, nsamples=2 ** M, seed=0).explain(clip, num_segments=M, mode="errors", unit="labels")
    assert res["Z"].shape[0] == 2 ** M - 2 and int(res["status"].item()) == 0
    fx, fnull = res["fx"].cpu().numpy(), res["fnull"].cpu().numpy()
    assert fx[0] == 0.0                                              # the default reference is the clip's own transcript
    f = lambda Zm: eng.eval_bits(eng.bits_to_device(np.atleast_2d(Zm).astype(np.uint8))).cpu().numpy().astype(np.float64)
    exact = brute_force_shapley(f, M)
    phi = res["phi"].cpu().numpy()
    err = np.abs(phi - exact).max()
    print(f"errors KernelSHAP, full enumeration M={M}, N={res['reference_lengths']}: f(empty) = {fnull[0]:.0f}, "
          f"max |phi - brute force| {err:.3e}, max |phi| {np.abs(exact).max():.3g}")
    assert np.abs(exact).max() > 0
    assert err <= 1e-6 * max(1.0, np.abs(exact).max())
    assert np.abs(phi.sum(0) - (fx - fnull)).max() <= 1e-6 * max(1.0, np.abs(fx - fnull).max())
    assert eng.mode == "errors"
    eng.close()


def test_explain_errors_default_words_scores_zero_on_the_full_coalition(P):
    model, cfg = _model("tiny_layer_stable")
    eng = P.Engine(model, cfg, max_batch=32)
    res = P.KernelShapExplainer(eng, nsamples=200, seed=1).explain(P.synthetic_clip(16000), num_segments=16, mode="errors")
    assert float(res["fx"][0]) == 0.0 and res["phi"].shape == (16, 1)
    assert res["reference_lengths"] == [reference_length(res["references"][0], "words", DELIM)]
    eng.close()


def test_explain_test_set_errors_match_metrics_wer(P, tmp_path):
    model, cfg = _model("tiny_group")
    eng = P.Engine(model, cfg, max_batch=64)
    items = P.make_test_set(num_clips=1, num_samples=16000, snrs=(5, 1, -5), seed=0)
    res = P.explain_test_set(eng, items, out_dir=str(tmp_path), num_segments=16, nsamples=100, mode="errors",
                             save_limit=0)
    for r in res:
        n = r["reference_words"]
        assert n == len(r["text"].split())
        want = metrics.wer(r["text"], r["hypothesis"]) * n if n else len(r["hypothesis"].split())
        print(f"{r['tag']}: {r['errors']:.0f} word errors of {n} (WER {metrics.wer(r['text'], r['hypothesis']):.3f})")
        assert r["errors"] == round(want)
    assert res[0]["errors"] == 0
    eng.close()
