"""GPU: DTW token timestamps through the C ABI (flash_attn = false, dtw_token_timestamps = true, like the reference requires): the
alignment-head cross-attention weights this engine computes (kernel chain with the queries captured per layer + k_dtw_qk) against the
reference's own aheads_cross_QKs on the same synthetic 3-text-layer model and the same scripted transcript; every text token gets a
t_dtw, and t_dtw equals what the host DTW code -- pinned exactly against the reference on CPU, tests/test_dtw_cpu.py -- makes of those
weights.  (Written after the GPU budget of round 1 was spent: not yet run on a GPU.)"""
import ctypes as C
import os
import numpy as np
import pytest

from wbtest import DATA_DIR, data_file, F16, Q5_0, TokenData, bind_whisper_api, read_wav_f32
from e2e_util import synth
from test_full_scripted_cpu import Script, LOG_CB, _quiet

pytestmark = pytest.mark.gpu
vp = C.c_void_p


def _run(X, path, pcm, use_gpu):
    X.whisper_log_set.argtypes = [LOG_CB, vp]; X.whisper_log_set(_quiet, None)
    cp = X.whisper_context_default_params()
    cp.use_gpu = use_gpu; cp.flash_attn = False; cp.dtw_token_timestamps = True; cp.dtw_aheads_preset = 1; cp.dtw_n_top = 2
    ctx = X.whisper_init_from_file_with_params(path.encode(), cp)
    assert ctx, (X.wb200_last_error() if use_gpu else "reference init failed")
    fp = X.whisper_full_default_params(0)
    fp.print_progress = False; fp.n_threads = 4; fp.no_speech_thold = 2.0; fp.greedy.best_of = 1; fp.temperature_inc = 0.0
    script = Script(X, ctx, 77, "peaked")
    fp.logits_filter_callback = C.cast(script.cb, vp)
    assert X.whisper_full(ctx, fp, pcm.ctypes.data_as(vp), len(pcm)) == 0
    toks = []
    for i in range(X.whisper_full_n_segments(ctx)):
        toks.append([X.whisper_full_get_token_data(ctx, i, j) for j in range(X.whisper_full_n_tokens(ctx, i))])
    return ctx, [[(t.id, t.t_dtw) for t in seg] for seg in toks]


@pytest.mark.parametrize("wt,tol", [(F16, 2e-2), (Q5_0, 8e-2)])
def test_dtw_weights_and_timestamps(lib, ref, tmp_path, wt, tol):
    L = bind_whisper_api(lib); R = bind_whisper_api(ref)
    L.wb200_last_error.restype = C.c_char_p
    path = str(tmp_path / "m.bin")
    synth.write_model(path, (51864, 1500, 384, 6, 1, 448, 384, 6, 3, 80), wt, seed=9, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    pcm = np.ascontiguousarray(read_wav_f32(os.path.join(DATA_DIR, "jfk.wav")), np.float32)
    lctx, mine = _run(L, path, pcm, True)
    rctx, theirs = _run(R, path, pcm, False)
    try:
        assert [[t[0] for t in s] for s in mine] == [[t[0] for t in s] for s in theirs]        # the scripted transcript is the same on both sides
        eot = L.whisper_token_eot(lctx)
        # weights
        L.wb200_ctx_state.restype = vp; L.wb200_ctx_state.argtypes = [vp]
        L.wb200_dbg_last_dtw_qks.restype = C.c_int64; L.wb200_dbg_last_dtw_qks.argtypes = [vp, vp, C.c_int64, vp]
        shape = (C.c_int * 3)()
        n = L.wb200_dbg_last_dtw_qks(L.wb200_ctx_state(lctx), None, 0, shape)
        a = np.empty(n, np.float32)
        assert L.wb200_dbg_last_dtw_qks(L.wb200_ctx_state(lctx), a.ctypes.data, n, shape) == n
        R.wref_ctx_state.restype = vp; R.wref_ctx_state.argtypes = [vp]
        R.wref_dtw_qks.restype = C.c_int64; R.wref_dtw_qks.argtypes = [vp, vp, C.c_int64, vp, vp, vp]
        nt, na, nh = C.c_int(), C.c_int(), C.c_int()
        m = R.wref_dtw_qks(R.wref_ctx_state(rctx), None, 0, C.byref(nt), C.byref(na), C.byref(nh))
        b = np.empty(m, np.float32)
        assert R.wref_dtw_qks(R.wref_ctx_state(rctx), b.ctypes.data, m, C.byref(nt), C.byref(na), C.byref(nh)) == m
        assert (shape[0], shape[1], shape[2]) == (nt.value, na.value, nh.value) and n == m
        err = float(np.sqrt(((a - b) ** 2).mean()) / np.sqrt((b ** 2).mean()))
        print("dtw alignment-head weights: %d x %d x %d, relative rms error %.2e" % (nt.value, na.value, nh.value, err))
        assert err < tol
        assert np.allclose(a.reshape(nh.value, na.value, nt.value).sum(axis=1), 1.0, atol=1e-4)     # each (head, token) is a distribution over time
        # timestamps: every text token stamped, inside the clip, and exactly what the (CPU-pinned) host code makes of these weights
        flat = [t for s in mine for t in s]
        text = [t for t in flat if t[0] < eot]
        assert all(0 <= t[1] <= len(pcm) // 160 + 2 for t in text)
        ids = np.asarray([t[0] for t in flat], np.int32); sizes = np.asarray([len(s) for s in mine], np.int32)
        got = (C.c_int64 * len(ids))()
        L.wb200_dbg_dtw.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, vp]
        L.whisper_n_len.argtypes = [vp]
        n_frames = min(3000, L.whisper_n_len(lctx))
        assert L.wb200_dbg_dtw(a.ctypes.data, shape[0], shape[1], shape[2], n_frames, 1, 0, eot, ids.ctypes.data, sizes.ctypes.data, len(sizes), got) > 0
        assert list(got) == [t[1] for t in flat]
        # reported only: with random weights the alignment cost surface is nearly flat, so the reference's own path moves under 1e-3 weight noise
        d = np.abs(np.asarray([t[1] for t in text]) - np.asarray([t[1] for s in theirs for t in s if t[0] < eot]))
        print("dtw t_dtw vs reference: median |d| = %.0f cs, 90%% = %.0f cs, identical %d / %d" % (np.median(d), np.quantile(d, 0.9), int((d == 0).sum()), len(d)))
    finally:
        L.whisper_free(lctx); R.whisper_free(rctx)
