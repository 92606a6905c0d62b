"""GPU: the on-device logits filter + greedy pick (k_greedy_sample) against the host restatement (which tests/test_sampler_cpu.py
pins bit for bit to the reference): token ids and timestamp ids identical, probabilities to f32 summation order."""
import ctypes as C
import os
import numpy as np
import pytest

from wbtest import data_file, FullParams, TokenData, bind_whisper_api

pytestmark = pytest.mark.gpu
vp = C.c_void_p


@pytest.mark.parametrize("stub", ["for-tests-ggml-tiny.en.bin", "for-tests-ggml-tiny.bin"])
def test_device_sampler_matches_host_filter(lib, stub):
    L = bind_whisper_api(lib)
    path = data_file(stub).encode()
    sig = [C.POINTER(FullParams), C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int]
    L.wb200_dbg_process_logits.argtypes = [C.c_char_p] + sig + [C.c_float, vp, vp, vp, vp, C.POINTER(TokenData)]
    L.wb200_dbg_greedy_sample.argtypes = [C.c_char_p] + sig + [vp, C.POINTER(TokenData)]
    multilingual = stub.endswith("tiny.bin")
    n_vocab = 51865 if multilingual else 51864
    eot = 50257 if multilingual else 50256
    beg = eot + (107 if multilingual else 107)          # token_beg = 50363 (.en) / 50364 (multilingual)
    rng = np.random.default_rng(11)
    n_ts = 0
    for trial in range(32):
        fp = L.whisper_full_default_params(0)
        fp.suppress_nst = bool(trial & 1)
        fp.no_timestamps = trial % 7 == 3
        fp.max_initial_ts = 1.0 if trial % 5 else 0.0
        fp.max_tokens = 6 if trial % 6 == 2 else 0
        kind = trial % 4
        if kind == 0:
            hist, has_ts, sd = [], 0, 0
        elif kind == 1:
            hist, has_ts, sd = [100, 200, beg + 50], 1, 100
        elif kind == 2:
            hist, has_ts, sd = [100, beg + 10, beg + 60], 1, 120
        else:
            hist, has_ts, sd = [int(x) for x in rng.integers(0, eot, 9)], 0, 0
        logits = (rng.standard_normal(n_vocab) * 3.0).astype(np.float32)
        if trial % 3 == 0:
            logits[beg:] += 4.0
        if trial % 8 == 5:
            j = int(rng.integers(0, eot - 1)); logits[j] = logits[j + 1] = logits.max() + 1.0
        h = (C.c_int * max(1, len(hist)))(*hist)
        host = TokenData(); dev = TokenData()
        assert L.wb200_dbg_process_logits(path, C.byref(fp), h, len(hist), has_ts, sd, C.c_float(0.0), logits.ctypes.data_as(vp), None, None, None, C.byref(host)) == 0
        assert L.wb200_dbg_greedy_sample(path, C.byref(fp), h, len(hist), has_ts, sd, logits.ctypes.data_as(vp), C.byref(dev)) == 0, L.wb200_last_error()
        assert (dev.id, dev.tid) == (host.id, host.tid), trial
        for a, b in ((dev.p, host.p), (dev.pt, host.pt), (dev.ptsum, host.ptsum)):
            assert abs(a - b) <= 2e-4 * max(abs(b), 1e-3), (trial, a, b)      # f32 sum of 51k exponentials in a different order: ~4e-5
        assert abs(dev.plog - host.plog) <= 2e-4 * max(1.0, abs(host.plog))
        n_ts += int(host.id >= beg)
    assert 0 < n_ts < 32                                # both text and timestamp picks were exercised


@pytest.mark.gpu
@pytest.mark.parametrize("stub", ["for-tests-ggml-tiny.en.bin", "for-tests-ggml-tiny.bin"])
def test_device_categorical_draws_match_host_sampler(lib, stub):
    """beam search: the k draws of std::discrete_distribution(probs) per decoder (whisper_sample_token_topk, src/whisper.cpp:6545-6618) made
    on the device from host-drawn uniforms, against the host sampler (pinned to the reference bit for bit in test_sampler_cpu)."""
    L = bind_whisper_api(lib)
    path = data_file(stub).encode()
    sig = [C.POINTER(FullParams), C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int]
    L.wb200_dbg_sample_topk.argtypes = [C.c_char_p] + sig + [C.c_float, vp, C.c_int, C.c_int, C.POINTER(TokenData)]
    L.wb200_dbg_draw_sample.argtypes = [C.c_char_p] + sig + [vp, C.c_int, C.c_int, C.POINTER(TokenData)]
    multilingual = stub.endswith("tiny.bin")
    n_vocab = 51865 if multilingual else 51864
    eot = 50257 if multilingual else 50256
    beg = eot + 107
    rng = np.random.default_rng(5)
    n_same = n_all = 0
    for trial in range(24):
        fp = L.whisper_full_default_params(1)
        fp.suppress_nst = bool(trial & 1)
        kind = trial % 3
        hist, has_ts, sd = ([], 0, 0) if kind == 0 else ([100, 200, beg + 20], 1, 40) if kind == 1 else ([int(x) for x in rng.integers(0, eot, 5)], 0, 0)
        logits = (rng.standard_normal(n_vocab) * (3.0 if trial % 2 else 8.0)).astype(np.float32)      # flat and peaked distributions
        K = 5 if trial % 4 else 40
        h = (C.c_int * max(1, len(hist)))(*hist)
        a = (TokenData * K)(); b = (TokenData * K)()
        assert L.wb200_dbg_sample_topk(path, C.byref(fp), h, len(hist), has_ts, sd, C.c_float(0.0), logits.ctypes.data_as(vp), K, trial, b) == 0
        assert L.wb200_dbg_draw_sample(path, C.byref(fp), h, len(hist), has_ts, sd, logits.ctypes.data_as(vp), K, trial, a) == 0, L.wb200_last_error()
        for i in range(K):
            n_all += 1
            assert (a[i].id, a[i].tid) == (b[i].id, b[i].tid), (trial, i, a[i].id, b[i].id)
            n_same += 1
            for x, y in ((a[i].p, b[i].p), (a[i].pt, b[i].pt), (a[i].ptsum, b[i].ptsum)):
                assert abs(x - y) <= 2e-4 * max(abs(y), 1e-3), (trial, i, x, y)
            assert abs(a[i].plog - b[i].plog) <= 2e-4 * max(1.0, abs(b[i].plog))
    assert n_same == n_all
