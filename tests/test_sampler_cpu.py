"""CPU (no GPU): the host logits filter + greedy pick of libwhisper_b200.so (wb_full.cpp: process_logits / sample_token, the
restatement of src/whisper.cpp:6196-6543) against the UNMODIFIED reference (oracle/_ref, wref_process_logits) on injected
logits -- rows a9/a10 of SURVEY.md 8.  Bit-exact: same float formulas in the same order, integer token ids, tie rule."""
import ctypes as C
import os
import numpy as np
import pytest

from wbtest import data_file, FullParams, TokenData, bind_whisper_api

vp = C.c_void_p


def _setup(lib, ref, stub):
    L = bind_whisper_api(lib); R = bind_whisper_api(ref)
    path = data_file(stub).encode()
    cp = R.whisper_context_default_params(); cp.use_gpu = False
    rctx = R.whisper_init_from_file_with_params(path, cp)
    assert rctx
    R.wref_ctx_state.restype = vp; R.wref_ctx_state.argtypes = [vp]
    sig = [C.POINTER(FullParams), C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.c_float, vp, vp, vp, vp, C.POINTER(TokenData)]
    R.wref_process_logits.argtypes = [vp, vp] + sig
    L.wb200_dbg_process_logits.argtypes = [C.c_char_p] + sig
    return L, R, path, rctx


def _run_both(L, R, path, rctx, fp, hist, has_ts, seek_delta, temp, logits):
    n = len(logits)
    h = (C.c_int * max(1, len(hist)))(*hist)
    outs = []
    for which in (0, 1):
        lo = np.empty(n, np.float32); lp = np.empty(n, np.float32); pr = np.empty(n, np.float32); td = TokenData()
        args = (C.byref(fp), h, len(hist), has_ts, seek_delta, C.c_float(temp), logits.ctypes.data_as(vp), lo.ctypes.data_as(vp),
                lp.ctypes.data_as(vp), pr.ctypes.data_as(vp), C.byref(td))
        rc = L.wb200_dbg_process_logits(path, *args) if which == 0 else R.wref_process_logits(rctx, R.wref_ctx_state(rctx), *args)
        assert rc == 0
        outs.append((lo, lp, pr, td))
    return outs


@pytest.mark.parametrize("stub", ["for-tests-ggml-tiny.en.bin", "for-tests-ggml-tiny.bin"])
def test_logits_filter_and_greedy_pick_match_reference(lib, ref, stub):
    L, R, path, rctx = _setup(lib, ref, stub)
    n_vocab = R.whisper_n_vocab(rctx)
    beg, eot = R.whisper_token_beg(rctx), R.whisper_token_eot(rctx)
    rng = np.random.default_rng(5)
    cases = []
    for trial in range(24):
        fp = R.whisper_full_default_params(0)
        fp.suppress_nst = bool(trial & 1)
        fp.no_timestamps = trial % 7 == 3
        fp.max_initial_ts = 1.0 if trial % 5 else 0.0
        fp.max_tokens = 6 if trial % 6 == 2 else 0
        kind = trial % 4
        if kind == 0:
            hist, has_ts, sd = [], 0, 0                                             # initial step: blank / max_initial_ts rules
        elif kind == 1:
            hist, has_ts, sd = [100, 200, beg + 50], 1, 100                        # last token is a timestamp, penultimate is text
        elif kind == 2:
            hist, has_ts, sd = [100, beg + 10, beg + 60], 1, 120                   # two timestamps in a row
        else:
            hist, has_ts, sd = [int(x) for x in rng.integers(0, eot, 9)], 0, 0      # plain text history (max_tokens rule when set)
        logits = rng.standard_normal(n_vocab).astype(np.float32) * 3.0
        if trial % 3 == 0:
            logits[beg:] += 4.0                                                    # timestamp mass > best text token
        if trial % 8 == 5:
            j = int(rng.integers(0, eot - 1)); logits[j] = logits[j + 1] = logits.max() + 1.0   # exact tie: lowest index wins
        temp = 0.0 if trial % 2 == 0 else 0.6
        cases.append((fp, hist, has_ts, sd, temp, logits))
    for fp, hist, has_ts, sd, temp, logits in cases:
        (lo_a, lp_a, pr_a, td_a), (lo_b, lp_b, pr_b, td_b) = _run_both(L, R, path, rctx, fp, hist, has_ts, sd, temp, logits)
        assert np.array_equal(lo_a, lo_b)                   # same -inf pattern and same finite values
        assert np.array_equal(lp_a, lp_b) and np.array_equal(pr_a, pr_b)
        assert (td_a.id, td_a.tid) == (td_b.id, td_b.tid)
        assert td_a.p == td_b.p and td_a.plog == td_b.plog and td_a.pt == td_b.pt and td_a.ptsum == td_b.ptsum
    R.whisper_free(rctx)


@pytest.mark.parametrize("stub", ["for-tests-ggml-tiny.en.bin", "for-tests-ggml-tiny.bin"])
def test_beam_candidates_match_reference(lib, ref, stub):
    """beam search draws its k candidates per beam from std::discrete_distribution(probs) with std::mt19937(j)
    (whisper_sample_token_topk, src/whisper.cpp:6545-6618): same probabilities + same libstdc++ => the same draws."""
    L, R, path, rctx = _setup(lib, ref, stub)
    if not hasattr(R, "wref_sample_topk"):
        pytest.skip("oracle/_ref predates wref_sample_topk (rebuild with make -C oracle)")
    n_vocab = R.whisper_n_vocab(rctx)
    beg, eot = R.whisper_token_beg(rctx), R.whisper_token_eot(rctx)
    K = 5
    R.wref_sample_topk.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(TokenData)]
    L.wb200_dbg_sample_topk.argtypes = [C.c_char_p, C.POINTER(FullParams), C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.c_float, vp,
                                        C.c_int, C.c_int, C.POINTER(TokenData)]
    rng = np.random.default_rng(9)
    for trial in range(12):
        fp = R.whisper_full_default_params(1)
        hist, has_ts, sd = ([], 0, 0) if trial % 3 == 0 else ([100, 200, beg + 20], 1, 40) if trial % 3 == 1 else ([int(x) for x in rng.integers(0, eot, 5)], 0, 0)
        logits = (rng.standard_normal(n_vocab) * (3.0 if trial % 2 else 8.0)).astype(np.float32)      # flat and peaked distributions
        temp = 0.0 if trial % 4 else 0.4
        _run_both(L, R, path, rctx, fp, hist, has_ts, sd, temp, logits)               # leaves the distribution in the reference's decoder 0
        h = (C.c_int * max(1, len(hist)))(*hist)
        a = (TokenData * K)(); b = (TokenData * K)()
        assert R.wref_sample_topk(rctx, R.wref_ctx_state(rctx), K, trial, b) == 0
        assert L.wb200_dbg_sample_topk(path, C.byref(fp), h, len(hist), has_ts, sd, C.c_float(temp), logits.ctypes.data_as(vp), K, trial, a) == 0
        for i in range(K):
            assert (a[i].id, a[i].tid) == (b[i].id, b[i].tid), (trial, i)
            assert a[i].p == b[i].p and a[i].plog == b[i].plog and a[i].pt == b[i].pt and a[i].ptsum == b[i].ptsum
        # the same candidates when the uniforms are taken from the generator BEFORE the decode (what whisper_full does so that the draws
        # can run on the device): running sums + lower_bound as libstdc++'s discrete_distribution forms them
        c = (TokenData * K)()
        assert L.wb200_dbg_sample_topk(path, C.byref(fp), h, len(hist), has_ts, sd, C.c_float(temp), logits.ctypes.data_as(vp), -K, trial, c) == 0
        for i in range(K):
            assert (c[i].id, c[i].tid, c[i].p, c[i].plog, c[i].pt, c[i].ptsum) == (b[i].id, b[i].tid, b[i].p, b[i].plog, b[i].pt, b[i].ptsum), (trial, i)
    R.whisper_free(rctx)
