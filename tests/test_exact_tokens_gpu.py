"""GPU: EXACT token identity with the reference CPU path over whole free-running transcripts (>= 200 tokens), greedy AND beam search
with 5 beams, F16 and Q5_0 -- on synthetic models that are WELL-CONDITIONED in the sense a trained checkpoint is.

Why a conditioned model.  With plain random weights the top-2 logit gap is below the noise between two correct implementations at a few
percent of the steps (gap ~ Exp(0.21 sigma) for 51864 Gaussian logits), so free-running transcripts part ways at the first near-tie.
"Noise" is not this engine's alone: the reference differs FROM ITSELF by 4e-2 of the logits' std when only n_threads changes
(tests/test_reference_noise_cpu.py: its CPU flash attention accumulates P.V in F16 and cuts the 1536 cross keys into one chunk per thread,
ggml-cpu/ops.cpp:8585-8600, 9122-9157; its encoder output moves by 5.6e-3 for Q5_0).  synth.conditioned() attenuates the one part of the
decoder whose reference arithmetic cannot be reproduced bit for bit -- what the attention VALUE path adds to the residual stream -- and
sharpens the softmax (final LayerNorm gain x100), so every decision has a margin far above the remaining noise.  Seeds were chosen on the
CPU (reference only) such that the reference's own smallest top-2 margin over the whole transcript is >= 2e-3 sigma, the transcript uses
>= 40 distinct ids, and -- for attn > 0 -- another audio clip changes the transcript (the audio path is attenuated, not cut).

  F16,  attn 1e-3 : reference noise across thread counts 1.4e-4 sigma; seeds 3 and 16: the reference gives the same transcript on 1 / 4 / 8
                    threads (greedy and beam), 427 .. 525 tokens, 6 .. 8 segments with real timestamp tokens, ragged windows
  Q5_0, attn 0    : the value path removed; everything else (token + position embeddings, 3 x (LN, int8 GEMVs, GELU table), logits
                    GEMV, filters, samplers, KV bookkeeping, timestamp rules, seek loop) is live; exact
  Q5_0, attn 1e-4 : int8 activation blocks make tiny perturbations occasionally jump (one rounding flip = up to 1e-2 sigma): in a search
                    over 30 seeds the reference never reproduced its own 4-thread transcript on 1 thread.  Asserted instead: this engine
                    follows the 4-thread reference at least as far as the 1-thread reference does
Everything that is not attention is mirrored arithmetic (Q8_0 activation blocks, integer block dots, f16 GELU table), so identity is
expected and asserted token for token, with segment times.
"""
import ctypes as C
import os

import numpy as np
import pytest

from wbtest import data_file, F16, Q5_0, TokenData
from e2e_util import Side, synth

pytestmark = pytest.mark.gpu
vp = C.c_void_p

# (weight type, model seed, attenuation of the attention value path, final-LN gain, strategy, what is asserted)
# The model is "test-3l.en": three text layers, so that whisper_full keeps timestamps on (two text layers + an English vocabulary count as
# "distilled" and force no_timestamps).
#   exact   : token-for-token and segment-time identity over the whole transcript
#   margin  : identical until the first sampling step where the reference's own top-2 margin is below 1e-2 sigma (Q5_0: this engine's
#             f32 summation orders differ from the AVX2 kernels' at the 1e-7 level; once in a few hundred steps that flips one int8
#             activation rounding, which moves a logit by up to ~6e-3 sigma -- measured, scripts/dbg_beam.py)
#   yardstick: stays with the 4-thread reference at least as long as the 1-thread reference does
# Beam search is run with gain 3000: sample_token_topk DRAWS its candidates from softmax(logits) with a seeded mt19937, and once two
# candidates' cumulative log-probabilities are within the logit noise their order -- hence which decoder's RNG stream continues which
# hypothesis -- is a coin toss for any two implementations.  With the sharper softmax every draw is the arg-max, candidates tie exactly and
# the reference's own tie-break (decoder index) decides: what is pinned is the beam machinery (candidate expansion, de-duplication, KV
# sequence copies, 5-row decode passes, scoring and selection of the best decoder), free of coin tosses.
CASES = [(F16, 3, 1e-3, 100.0, 0, "exact"), (F16, 16, 1e-3, 100.0, 0, "exact"),
         (F16, 3, 1e-3, 3000.0, 1, "exact"), (F16, 16, 1e-3, 3000.0, 1, "exact"),
         (Q5_0, 0, 0.0, 100.0, 0, "margin"), (Q5_0, 7, 1e-4, 100.0, 0, "yardstick")]


def _model(tmp_path, wt, seed, attn, gain):
    stub = data_file("for-tests-ggml-tiny.en.bin")
    path = str(tmp_path / ("cond-%d-%d-%g-%g.bin" % (wt, seed, attn, gain)))
    synth.write_model(path, "test-3l.en", wt, seed=seed, vocab_from=stub, scale=lambda n: synth.conditioned(n, attn, gain))
    return path


LOGITS_CB = C.CFUNCTYPE(None, vp, vp, C.POINTER(TokenData), C.c_int, C.POINTER(C.c_float), vp)


def _run(S, pcm, strategy, n_threads=4, record=None):
    L = S.L
    fp = L.whisper_full_default_params(strategy); fp.print_progress = False; fp.temperature_inc = 0.0; fp.greedy.best_of = 1; fp.n_threads = n_threads
    if strategy == 1:
        fp.beam_search.beam_size = 5
    cb = None
    if record is not None:                               # (token history, top-2 margin in units of the logits' std) of every sampling step
        V = S.n_vocab

        def rec(c, st, toks, nt, logits, ud):
            x = np.ctypeslib.as_array(logits, (V,)); fin = x[np.isfinite(x)]
            top = np.partition(fin, -2)[-2:]
            record.append((tuple(toks[k].id for k in range(nt)), float(top[1] - top[0]) / float(fin.std())))
        cb = LOGITS_CB(rec)
        fp.logits_filter_callback = C.cast(cb, vp)
    assert L.whisper_full(S.ctx, fp, pcm.ctypes.data_as(vp), len(pcm)) == 0
    segs = []
    for i in range(L.whisper_full_n_segments(S.ctx)):
        segs.append((L.whisper_full_get_segment_t0(S.ctx, i), L.whisper_full_get_segment_t1(S.ctx, i),
                     [L.whisper_full_get_token_id(S.ctx, i, j) for j in range(L.whisper_full_n_tokens(S.ctx, i))]))
    return segs


def _common(a, b):
    k = 0
    while k < min(len(a), len(b)) and a[k] == b[k]:
        k += 1
    return k


@pytest.mark.parametrize("wt,seed,attn,gain,strategy,mode", CASES)
def test_free_running_transcripts_are_token_identical(lib, ref, tmp_path, wt, seed, attn, gain, strategy, mode):
    path = _model(tmp_path, wt, seed, attn, gain)
    pcm = synth.synth_audio(seed=500 + seed, seconds=60.0)
    A = Side(lib, path, False); B = Side(ref, path, True)
    try:
        # every case runs twice: on a FRESH state the reference reads an all-zero row 0 for the no-speech probability of the first window
        # (wb_state.h, whisper_state::lrows) -- with this model's huge logits that is +inf and the window is dropped -- on a used state not
        for name in ("fresh state", "used state"):
            sa = _run(A, pcm, strategy); sb = _run(B, pcm, strategy)
            ta = [t for s in sa for t in s[2]]; tb = [t for s in sb for t in s[2]]
            k = _common(ta, tb)
            print("%s, strategy %d: %d tokens (reference %d), %d distinct, %d segments, identical prefix %d" % (name, strategy, len(ta), len(tb), len(set(tb)), len(sb), k))
            assert len(tb) >= 200
            if mode == "exact":
                assert ta == tb, (name, k, ta[max(0, k - 3):k + 3], tb[max(0, k - 3):k + 3])
                assert [(s[0], s[1]) for s in sa] == [(s[0], s[1]) for s in sb]
            elif mode == "yardstick":
                t1 = [t for s in _run(B, pcm, strategy, n_threads=1) for t in s[2]]
                print("   reference 1 thread vs 4 threads: identical prefix %d" % _common(t1, tb))
                assert k >= min(_common(t1, tb), len(tb)), (name, k, _common(t1, tb))
        if mode == "margin":
            ra, rb = [], []
            _run(A, pcm, strategy, record=ra); _run(B, pcm, strategy, record=rb)
            c = 0
            while c < min(len(ra), len(rb)) and ra[c][0] == rb[c][0]:
                c += 1
            print("   sampling steps with identical history: %d of %d" % (c, len(rb)))
            assert c >= 100
            if c < min(len(ra), len(rb)):                # histories part at step c: the decision of step c-1 differed
                assert rb[c - 1][1] < 1e-2, (c, rb[c - 1][1])
        if attn > 0 and strategy == 0:                   # the audio path is attenuated, not cut: another clip changes the transcript
            other = synth.synth_audio(seed=9000 + seed, seconds=60.0)
            assert _run(A, other, 0) != _run(A, pcm, 0)
    finally:
        A.free(); B.free()
