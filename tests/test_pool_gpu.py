"""GPU: the context-level device pool behind the whisper.h entry points (wb_state.h, Group).

whisper.h allows concurrent whisper_full_with_state calls on DISTINCT states of one context (include/whisper.h:45-46) and
whisper_full_parallel is exactly that (src/whisper.cpp:7813-7941).  In this engine such calls rendezvous into lock-step batched
passes.  Asserted here, through the C ABI only:
  * 8 threads x whisper_full_with_state on 8 states give, chunk by chunk, the tokens of the same chunks run one by one, and the
    passes really were shared (rows per decode pass > 1);
  * whisper_full_parallel(n = 4) on the GPU equals the REFERENCE's whisper_full_parallel segment for segment, token for token
    (id / p / plog / t0 / t1 ...) when both are driven by the same scripted logits_filter_callback (the model is taken out of the
    equation exactly like tests/test_full_scripted_cpu.py does on the CPU);
  * 64 ragged chunks through the pool == one by one, and == the reference's tokens wherever the reference's own top-2 margin
    exceeds the logit noise;
  * states can be created and freed while others are transcribing (pool growth keeps KV contents).
"""
import ctypes as C
import os
import threading

import numpy as np
import pytest

from wbtest import data_file, F16, Q5_0, FullParams, TokenData, read_wav_f32
from e2e_util import Side, synth
from test_full_scripted_cpu import Script, collect

pytestmark = pytest.mark.gpu
vp = C.c_void_p


def _model(tmp_path, cfg, wt, seed):
    stub = data_file("for-tests-ggml-tiny.en.bin" if cfg.endswith(".en") else "for-tests-ggml-tiny.bin")
    path = str(tmp_path / f"{cfg}-{wt}-{seed}.bin")
    synth.write_model(path, cfg, wt, seed=seed, vocab_from=stub)
    return path


def _tokens_from_state(L, st):
    return [[L.whisper_full_get_token_id_from_state(st, s, j) for j in range(L.whisper_full_n_tokens_from_state(st, s))]
            for s in range(L.whisper_full_n_segments_from_state(st))]


def _tokens(L, ctx):
    return [[L.whisper_full_get_token_id(ctx, s, j) for j in range(L.whisper_full_n_tokens(ctx, s))] for s in range(L.whisper_full_n_segments(ctx))]


def _counters(L):
    L.wb200_counters.argtypes = [C.POINTER(C.c_double), C.c_int]
    a = (C.c_double * 8)(); L.wb200_counters(a, 8)
    return [a[i] for i in range(8)]


def test_concurrent_full_with_state_equals_one_by_one(lib, tmp_path):
    path = _model(tmp_path, "test-2l.en", Q5_0, 5)
    A = Side(lib, path, False)
    try:
        L = A.L
        secs = (30.0, 11.0, 47.0, 30.0, 3.0, 21.5, 8.0, 30.0)
        chunks = [synth.synth_audio(seed=40 + i, seconds=s) for i, s in enumerate(secs)]
        fp = L.whisper_full_default_params(0); fp.print_progress = False; fp.temperature_inc = 0.0; fp.greedy.best_of = 1
        single = []
        for c in chunks:
            assert L.whisper_full(A.ctx, fp, c.ctypes.data_as(vp), len(c)) == 0
            single.append(_tokens(L, A.ctx))
        states = [L.whisper_init_state(A.ctx) for _ in chunks]
        assert all(states), L.wb200_last_error()
        rcs = [None] * len(chunks)

        def work(i):
            rcs[i] = L.whisper_full_with_state(A.ctx, states[i], fp, chunks[i].ctypes.data_as(vp), len(chunks[i]))
        c0 = _counters(L)
        th = [threading.Thread(target=work, args=(i,)) for i in range(len(chunks))]
        for t in th: t.start()
        for t in th: t.join()
        c1 = _counters(L)
        assert rcs == [0] * len(chunks), (rcs, L.wb200_last_error())
        conc = [_tokens_from_state(L, st) for st in states]
        assert conc == single
        assert sum(len(t) for c in conc for t in c) > 50
        passes, rows = c1[0] - c0[0], c1[1] - c0[1]
        assert rows / passes > 2.0, (passes, rows)                 # the calls really shared their passes
        # a second round on the same states after freeing half of them and creating new ones (slot reuse)
        for st in states[::2]: L.whisper_free_state(st)
        states[::2] = [L.whisper_init_state(A.ctx) for _ in states[::2]]
        th = [threading.Thread(target=work, args=(i,)) for i in range(len(chunks))]
        for t in th: t.start()
        for t in th: t.join()
        assert [_tokens_from_state(L, st) for st in states] == single
        for st in states: L.whisper_free_state(st)
    finally:
        A.free()


def test_pool_grows_while_a_state_is_transcribing(lib, tmp_path):
    """whisper_init_state / beam search on other states re-lay the pool out (more slots, more KV cells per slot) while one state is in
    the middle of whisper_full: its transcript must not change."""
    path = _model(tmp_path, "test-2l.en", Q5_0, 6)
    A = Side(lib, path, False)
    try:
        L = A.L
        pcm = synth.synth_audio(seed=77, seconds=75.0)
        fp = L.whisper_full_default_params(0); fp.print_progress = False; fp.temperature_inc = 0.0; fp.greedy.best_of = 1
        assert L.whisper_full(A.ctx, fp, pcm.ctypes.data_as(vp), len(pcm)) == 0
        want = _tokens(L, A.ctx)
        extra = []
        ENC = C.CFUNCTYPE(C.c_bool, vp, vp, vp)

        def on_window(ctx, st, ud):                                  # encoder_begin_callback of the transcribing state: grow the pool from inside
            s = L.whisper_init_state(A.ctx)
            assert s
            extra.append(s)
            if len(extra) == 2:                                       # ... and make another state need 5 decoders (cells per slot grow)
                short = synth.synth_audio(seed=78, seconds=2.0)
                bp = L.whisper_full_default_params(1); bp.print_progress = False; bp.temperature_inc = 0.0; bp.beam_search.beam_size = 5
                assert L.whisper_full_with_state(A.ctx, s, bp, short.ctypes.data_as(vp), len(short)) == 0
            return True
        cb = ENC(on_window)
        fp.encoder_begin_callback = C.cast(cb, vp)
        assert L.whisper_full(A.ctx, fp, pcm.ctypes.data_as(vp), len(pcm)) == 0
        assert len(extra) >= 2
        assert _tokens(L, A.ctx) == want
        for s in extra: L.whisper_free_state(s)
    finally:
        A.free()


@pytest.mark.parametrize("n_proc", [4])
def test_full_parallel_equals_reference_scripted(lib, ref, tmp_path, n_proc):
    path = _model(tmp_path, "test-2l.en", F16, 9)
    pcm = synth.synth_audio(seed=31, seconds=118.0)
    A = Side(lib, path, False); B = Side(ref, path, True)
    try:
        out = []
        for S in (A, B):
            L = S.L
            sc = Script(L, S.ctx, 4242, "peaked", use_segments=False)
            sc.tap = None; sc.tap_att = None                          # the batch taps exist only on engine-less test contexts
            fp = L.whisper_full_default_params(0); fp.print_progress = False; fp.greedy.best_of = 1; fp.temperature_inc = 0.0
            fp.n_threads = 2; fp.no_speech_thold = 2.0                # no_speech_prob comes from the real (different-noise) logits
            fp.logits_filter_callback = C.cast(sc.cb, vp)
            rc = L.whisper_full_parallel(S.ctx, fp, pcm.ctypes.data_as(vp), len(pcm), n_proc)
            assert rc == 0
            out.append(collect(L, S.ctx))
            assert sc.calls > 100
        assert len(out[0]) == len(out[1]) and len(out[0]) >= n_proc
        for sa, sb in zip(out[0], out[1]):
            assert sa == sb
    finally:
        A.free(); B.free()


def test_64_ragged_chunks_through_the_pool(lib, ref, tmp_path):
    path = _model(tmp_path, "test-2l.en", Q5_0, 5)
    A = Side(lib, path, False); B = Side(ref, path, True)
    try:
        L = A.L
        n = 64
        secs = [2.0 + 1.37 * ((i * 7) % 23) for i in range(n)]        # 2 .. 32 s: one or two windows, ragged ends
        chunks = [synth.synth_audio(seed=300 + i, seconds=s) for i, s in enumerate(secs)]
        fp = L.whisper_full_default_params(0); fp.print_progress = False; fp.temperature_inc = 0.0; fp.greedy.best_of = 1
        L.wb200_full_batch.argtypes = [vp, FullParams, C.POINTER(vp), C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
        ptrs = (vp * n)(*[c.ctypes.data for c in chunks]); lens = (C.c_int * n)(*[len(c) for c in chunks]); outs = (vp * n)()
        c0 = _counters(L)
        assert L.wb200_full_batch(A.ctx, fp, ptrs, lens, n, outs) == 0, L.wb200_last_error()
        c1 = _counters(L)
        batched = []
        for i in range(n):
            batched.append(_tokens_from_state(L, outs[i]))
            L.whisper_free_state(outs[i])
        assert (c1[1] - c0[1]) / (c1[0] - c0[0]) > 16.0               # rows per pass: the 64 sequences shared their launches
        single = []
        for c in chunks:
            assert L.whisper_full(A.ctx, fp, c.ctypes.data_as(vp), len(c)) == 0
            single.append(_tokens(L, A.ctx))
        assert batched == single
        # against the reference on a subset.  Both sides run with a logits_filter_callback that only RECORDS: the token history of every
        # sampling step and the top-2 margin of the logits it is shown.  The histories must be identical call by call until the first
        # step where the reference's own decision is within the logit noise (random weights: near-ties are frequent, SURVEY fact 7).
        R = B.L
        LOGITS_CB = C.CFUNCTYPE(None, vp, vp, C.POINTER(TokenData), C.c_int, C.POINTER(C.c_float), vp)
        V = A.n_vocab

        def run_recorded(Lx, ctx, pcm):
            log = []

            def rec(c, st, toks, nt, logits, ud):
                x = np.ctypeslib.as_array(logits, (V,))
                fin = x[np.isfinite(x)]
                top = np.partition(fin, -2)[-2:]
                log.append((tuple(toks[k].id for k in range(nt)), float(top[1] - top[0]) / float(fin.std())))
            cb = LOGITS_CB(rec)
            rp = Lx.whisper_full_default_params(0); rp.print_progress = False; rp.temperature_inc = 0.0; rp.greedy.best_of = 1; rp.n_threads = 4
            rp.logits_filter_callback = C.cast(cb, vp)
            assert Lx.whisper_full(ctx, rp, pcm.ctypes.data_as(vp), len(pcm)) == 0
            return log, _tokens(Lx, ctx)
        agree = total = 0
        for i in range(0, n, 8):
            rlog, _ = run_recorded(R, B.ctx, chunks[i])
            mlog, mtok = run_recorded(L, A.ctx, chunks[i])
            assert mtok == single[i]                                  # host sampler (callback present) == on-device sampler
            k = 0
            while k < min(len(rlog), len(mlog)) and rlog[k][0] == mlog[k][0]:
                k += 1
            agree += k; total += len(rlog)
            if k < min(len(rlog), len(mlog)):
                # histories differ at call k: the decision of call k-1 differed; the reference's margin there is within the noise
                assert rlog[k - 1][1] < 0.35, (i, k, rlog[k - 1][1])
        print("reference agreement on 8 chunks: %d of %d sampling steps before the first near-tie" % (agree, total))
        assert agree >= 8 * 4
    finally:
        A.free(); B.free()
