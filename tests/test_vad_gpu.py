"""GPU: the VAD kernels (k_vad_features + k_vad_lstm) through the whisper_vad_* C ABI against the reference's CPU graph, and
params.vad through whisper_full.  The host restatement of the same phases and all integer logic are pinned on CPU by
tests/test_vad_cpu.py; this file checks the device execution of those phases.
Tolerance on probabilities: 1.5e-3 (one F16 rounding flip of an activation; see test_vad_cpu.py), median below 5e-5."""
import ctypes as C
import os
import numpy as np
import pytest

from wbtest import DATA_DIR, data_file, Q5_0, bind_whisper_api, read_wav_f32
from e2e_util import Side, synth
from vad_synth import write_vad_model, speechy_audio
from test_vad_cpu import bind_vad, ref_probs, GOLDEN, SILERO

pytestmark = pytest.mark.gpu
vp = C.c_void_p


def _probs(L, vctx, pcm, pieces=None):
    return ref_probs(L, vctx, pcm, pieces)            # same whisper_vad_* calls on either library


def test_vad_device_real_silero_weights_golden(lib):
    """device kernels on the Silero weights of the reference's tests/test-vad.cpp: the committed reference probabilities
    (tests/golden/vad_r01.npz) and the reference's own KAT -- 344 probabilities, 4 segments with the default parameters"""
    if not os.path.exists(SILERO):
        pytest.skip("oracle/_ref/data lacks the silero fixture")
    bind_vad(lib)
    g = np.load(GOLDEN)
    pcm = np.ascontiguousarray(read_wav_f32(os.path.join(DATA_DIR, "jfk.wav")), np.float32)
    lv = lib.whisper_vad_init_from_file_with_params(SILERO.encode(), lib.whisper_vad_default_context_params())
    assert lv, lib.wb200_last_error()
    got = _probs(lib, lv, pcm)
    assert len(got) == 344
    d = np.abs(got - g["probs"])
    print("silero v6.2.0 on jfk.wav (device): max|d|=%.2e median %.2e" % (d.max(), np.median(d)))
    assert d.max() < 1.5e-3 and np.median(d) < 5e-5
    lib.whisper_vad_segments_from_probs.restype = vp
    lib.whisper_vad_segments_from_probs.argtypes = [vp, type(lib.whisper_vad_default_params())]
    segs = lib.whisper_vad_segments_from_probs(lv, lib.whisper_vad_default_params())
    n = lib.whisper_vad_segments_n_segments(segs)
    assert n == 4
    assert [int(lib.whisper_vad_segments_get_segment_t0(segs, i)) for i in range(n)] == g["seg_t0"].tolist()
    assert [int(lib.whisper_vad_segments_get_segment_t1(segs, i)) for i in range(n)] == g["seg_t1"].tolist()
    lib.whisper_vad_free_segments(segs); lib.whisper_vad_free(lv)


def test_vad_device_probs_match_reference(lib, ref, tmp_path):
    bind_vad(lib); bind_vad(ref)
    lib.wb200_dbg_vad_probs.argtypes = [C.c_char_p, vp, C.c_int, C.c_int, vp, C.c_int]
    for seed, gain in [(1, 1.0), (2, 1.6)]:
        path = write_vad_model(str(tmp_path / ("vad%d.bin" % seed)), seed=seed, gain=gain).encode()
        rv = ref.whisper_vad_init_from_file_with_params(path, ref.whisper_vad_default_context_params())
        lv = lib.whisper_vad_init_from_file_with_params(path, lib.whisper_vad_default_context_params())
        assert rv and lv, lib.wb200_last_error()
        for pcm in (read_wav_f32(os.path.join(DATA_DIR, "jfk.wav")), speechy_audio(31.7, seed), np.zeros(100, np.float32)):
            pcm = np.ascontiguousarray(pcm, np.float32)
            want = _probs(ref, rv, pcm)
            got = _probs(lib, lv, pcm)
            assert len(got) == len(want) == (len(pcm) + 511) // 512
            d = np.abs(got - want)
            print("vad device: n=%d  max|d|=%.2e  median %.2e" % (len(got), d.max(), np.median(d)))
            assert d.max() < 1.5e-3 and np.median(d) < 5e-5
            emu = np.empty(len(want) + 8, np.float32)                       # the host walk of the same phases
            n = lib.wb200_dbg_vad_probs(path, pcm.ctypes.data_as(vp), len(pcm), 0, emu.ctypes.data_as(vp), len(emu))
            assert n == len(got) and np.abs(emu[:n] - got).max() < 1.5e-3
        # streaming: state carried across calls == one shot
        pcm = np.ascontiguousarray(speechy_audio(12.0, seed + 10)[: 512 * 300])
        one = _probs(lib, lv, pcm)
        parts = _probs(lib, lv, pcm, pieces=512 * 77)
        assert np.array_equal(one, parts)
        ref.whisper_vad_free(rv); lib.whisper_vad_free(lv)


def test_whisper_full_with_vad_cuts_the_same_audio(lib, ref, tmp_path):
    """params.vad through whisper_full on both libraries: real Silero weights + jfk.wav with the default VAD parameters (no window of
    that clip is within 6e-3 of either hysteresis threshold, so the 1.5e-3 tolerance on device probabilities cannot move a boundary)"""
    if not os.path.exists(SILERO):
        pytest.skip("oracle/_ref/data lacks the silero fixture")
    bind_vad(lib); bind_vad(ref)
    g = np.load(GOLDEN)
    vpath = SILERO.encode()
    mpath = str(tmp_path / "m.bin")
    synth.write_model(mpath, "test-2l.en", Q5_0, seed=5, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    pcm = np.ascontiguousarray(read_wav_f32(os.path.join(DATA_DIR, "jfk.wav")), np.float32)
    A, B = Side(lib, mpath, False), Side(ref, mpath, True)
    try:
        out = []
        for S in (A, B):
            L = S.L
            for fn in ("whisper_full_get_vad_segment_t0", "whisper_full_get_vad_segment_t1"):
                getattr(L, fn).restype = C.c_int64; getattr(L, fn).argtypes = [vp, C.c_int]
            L.whisper_full_n_vad_segments.argtypes = [vp]
            L.whisper_full_get_segment_t0.restype = C.c_int64; L.whisper_full_get_segment_t1.restype = C.c_int64
            fp = L.whisper_full_default_params(0)
            fp.print_progress = False; fp.temperature_inc = 0.0; fp.greedy.best_of = 1; fp.no_timestamps = True; fp.max_tokens = 8
            fp.vad = True; fp.vad_model_path = vpath
            assert L.whisper_full(S.ctx, fp, pcm.ctypes.data_as(vp), len(pcm)) == 0
            nv = L.whisper_full_n_vad_segments(S.ctx)
            segs = [(L.whisper_full_get_vad_segment_t0(S.ctx, i), L.whisper_full_get_vad_segment_t1(S.ctx, i)) for i in range(nv)]
            ns = L.whisper_full_n_segments(S.ctx)
            times = [(L.whisper_full_get_segment_t0(S.ctx, i), L.whisper_full_get_segment_t1(S.ctx, i)) for i in range(ns)]
            out.append((segs, times))
        assert out[0][0] == out[1][0]                                       # identical speech segments (centiseconds, original timeline)
        assert out[0][0] == list(zip(g["seg_t0"].tolist(), g["seg_t1"].tolist()))   # = the reference's VAD known answer for this clip
        assert len(out[0][1]) >= 1 and all(0 <= a <= b <= len(pcm) // 160 + 100 for a, b in out[0][1])
        if len(out[0][1]) == len(out[1][1]):
            assert out[0][1][0][0] == out[1][1][0][0]                       # first segment starts where the first speech starts
    finally:
        A.free(); B.free()
