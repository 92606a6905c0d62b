"""CPU: experimental token-level timestamps (params.token_timestamps) and max_len segment wrapping of libwhisper_b200.so against
the reference (src/whisper.cpp:8500-8820, 6096-6147) on injected segments: token t0/t1, voice lengths, the carried t_beg / t_last /
tid_last state and the wrapped pieces must be identical."""
import ctypes as C
import os
import numpy as np
import pytest

from wbtest import data_file, bind_whisper_api

vp = C.c_void_p
SIG = [vp, vp, vp, vp, C.c_int, C.c_int64, C.c_int64, vp, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int]


def test_signal_energy_matches_reference(lib, ref):
    if not hasattr(ref, "wref_signal_energy"):
        pytest.skip("oracle/_ref predates wref_signal_energy (rebuild with make -C oracle)")
    rng = np.random.default_rng(0)
    pcm = (rng.standard_normal(5000) * np.hanning(5000)).astype(np.float32)
    a = np.empty_like(pcm); b = np.empty_like(pcm)
    for fn, out in ((lib.wb200_dbg_signal_energy, a), (ref.wref_signal_energy, b)):
        fn.argtypes = [vp, C.c_int, C.c_int, vp]
        assert fn(pcm.ctypes.data, len(pcm), 32, out.ctypes.data) == 0
    assert np.array_equal(a, b)


@pytest.mark.parametrize("stub", ["for-tests-ggml-tiny.en.bin", "for-tests-ggml-tiny.bin"])
def test_token_timestamps_and_wrapping_match_reference(lib, ref, stub):
    if not hasattr(ref, "wref_token_timestamps"):
        pytest.skip("oracle/_ref predates wref_token_timestamps (rebuild with make -C oracle)")
    R = bind_whisper_api(ref)
    path = data_file(stub).encode()
    cp = R.whisper_context_default_params(); cp.use_gpu = False
    rctx = R.whisper_init_from_file_with_params(path, cp)
    assert rctx
    R.wref_ctx_state.restype = vp; R.wref_ctx_state.argtypes = [vp]
    R.wref_token_timestamps.argtypes = [vp, vp] + SIG
    lib.wb200_dbg_token_timestamps.argtypes = [C.c_char_p] + SIG
    R.whisper_tokenize.argtypes = [vp, C.c_char_p, vp, C.c_int]
    beg, eot = R.whisper_token_beg(rctx), R.whisper_token_eot(rctx)
    rng = np.random.default_rng(3)
    n_energy = 16000 * 12
    t = np.arange(n_energy) / 16000.0
    energy = (np.abs(np.sin(2 * np.pi * 0.7 * t)) * (0.2 + 0.8 * (rng.random(n_energy) > 0.3))).astype(np.float32) * 0.1   # bursts and pauses
    texts = [" And so my fellow Americans, ask not what your country can do for you.", " 1, 2, 3... go! Why? Because: naïve café 東京、こんにちは。",
             " one", " a b c d e f g h i j k l m n o p"]
    carry_a = np.zeros(3, np.int64); carry_b = np.zeros(3, np.int64)
    seg_t0 = 0
    for case, text in enumerate(texts * 2):
        buf = (C.c_int * 256)()
        nt = R.whisper_tokenize(rctx, text.encode("utf-8"), buf, 256)
        assert nt > 0
        ids = list(buf[:nt])
        with_ts = case % 2 == 0
        if with_ts:
            ids = [beg + seg_t0 // 2 % 1400] + ids + [beg + (seg_t0 // 2 + 140) % 1400]      # segment framed by timestamp tokens
        n = len(ids)
        ids = np.asarray(ids, np.int32)
        tids = (beg + np.sort(rng.integers(seg_t0 // 2, seg_t0 // 2 + 150, n))).astype(np.int32)  # non-decreasing timestamp guesses
        tids[ids >= beg] = ids[ids >= beg]
        pt = rng.random(n).astype(np.float32) * (rng.random(n) > 0.4)                          # some confident, some not
        ptsum = rng.random(n).astype(np.float32)
        seg_t1 = seg_t0 + 300
        max_len = (0, 12, 25, 7)[case % 4]; split_on_word = case % 3 == 0
        outs = []
        for which, carry in ((0, carry_a), (1, carry_b)):
            tok = np.full((n, 2), -7, np.int64); vlen = np.zeros(n, np.float32); pieces = np.full((32, 3), -7, np.int64)
            args = (ids.ctypes.data, tids.ctypes.data, pt.ctypes.data, ptsum.ctypes.data, n, seg_t0, seg_t1, energy.ctypes.data, n_energy,
                    C.c_float(0.01), C.c_float(0.01), max_len, int(split_on_word), carry.ctypes.data, tok.ctypes.data, vlen.ctypes.data, pieces.ctypes.data, 32)
            npieces = lib.wb200_dbg_token_timestamps(path, *args) if which == 0 else R.wref_token_timestamps(rctx, R.wref_ctx_state(rctx), *args)
            assert npieces >= 1
            outs.append((npieces, tok, vlen, pieces))
        assert outs[0][0] == outs[1][0], case
        assert np.array_equal(outs[0][1], outs[1][1]), case
        assert np.array_equal(outs[0][2], outs[1][2]), case
        assert np.array_equal(outs[0][3], outs[1][3]), case
        assert np.array_equal(carry_a, carry_b), case
        if max_len:
            assert outs[0][0] > 1 or n < 4
        seg_t0 = seg_t1
    R.whisper_free(rctx)
