"""CPU: DTW token timestamps (whisper_context_params.dtw_token_timestamps, src/whisper.cpp:8856-9167).  The reference runs its whole DTW path
on the CPU (flash_attn off, a synthetic 3-text-layer model, transcript scripted through logits_filter_callback so that there is text to
align); the alignment-head cross-attention weights it computed are read back (oracle tap wref_dtw_qks) and fed to this library's host
code (normalisation, median filter, mean over heads, dynamic time warping, backtrace, assignment): t_dtw of every token must be
IDENTICAL.  (The device part -- producing those weights -- is tests/test_dtw_gpu.py.)"""
import ctypes as C
import os
import numpy as np
import pytest

from wbtest import DATA_DIR, data_file, F16, TokenData, bind_whisper_api, read_wav_f32
from e2e_util import synth
from test_full_scripted_cpu import Script, LOG_CB, _quiet

vp = C.c_void_p


class Ahead(C.Structure):
    _fields_ = [("n_text_layer", C.c_int), ("n_head", C.c_int)]


@pytest.mark.parametrize("preset", ["n_top_2", "n_top_1", "custom"])
def test_dtw_host_math_matches_reference(lib, ref, tmp_path, preset):
    if not hasattr(ref, "wref_dtw_qks"):
        pytest.skip("oracle/_ref predates wref_dtw_qks (rebuild with make -C oracle)")
    R = bind_whisper_api(ref)
    R.whisper_log_set.argtypes = [LOG_CB, vp]; R.whisper_log_set(_quiet, None)
    path = str(tmp_path / "m.bin")
    synth.write_model(path, (51864, 1500, 384, 6, 1, 448, 384, 6, 3, 80), F16, seed=9, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    cp = R.whisper_context_default_params(); cp.use_gpu = False; cp.flash_attn = False; cp.dtw_token_timestamps = True
    keep = None
    if preset == "custom":
        keep = (Ahead * 5)(Ahead(2, 3), Ahead(0, 1), Ahead(1, 5), Ahead(2, 0), Ahead(1, 2))
        cp.dtw_aheads_preset = 2; cp.dtw_aheads.n_heads = 5; cp.dtw_aheads.heads = C.cast(keep, vp)
    else:
        cp.dtw_aheads_preset = 1; cp.dtw_n_top = int(preset[-1])
    ctx = R.whisper_init_from_file_with_params(path.encode(), cp)
    assert ctx
    pcm = np.ascontiguousarray(read_wav_f32(os.path.join(DATA_DIR, "jfk.wav")), np.float32)
    fp = R.whisper_full_default_params(0)
    fp.print_progress = False; fp.n_threads = 4; fp.no_speech_thold = 2.0; fp.greedy.best_of = 1; fp.temperature_inc = 0.0
    script = Script(R, ctx, 77, "peaked")
    fp.logits_filter_callback = C.cast(script.cb, vp)
    assert R.whisper_full(ctx, fp, pcm.ctypes.data_as(vp), len(pcm)) == 0
    R.wref_ctx_state.restype = vp; R.wref_ctx_state.argtypes = [vp]
    st = R.wref_ctx_state(ctx)
    R.wref_dtw_qks.restype = C.c_int64; R.wref_dtw_qks.argtypes = [vp, vp, C.c_int64, vp, vp, vp]
    nt, na, nh = C.c_int(), C.c_int(), C.c_int()
    n = R.wref_dtw_qks(st, None, 0, C.byref(nt), C.byref(na), C.byref(nh))
    assert n == nt.value * na.value * nh.value > 0
    qk = np.empty(n, np.float32)
    assert R.wref_dtw_qks(st, qk.ctypes.data, n, C.byref(nt), C.byref(na), C.byref(nh)) == n
    assert nh.value == {"n_top_2": 12, "n_top_1": 6, "custom": 5}[preset]
    eot = R.whisper_token_eot(ctx)
    ids, sizes, want = [], [], []
    for i in range(R.whisper_full_n_segments(ctx)):
        toks = [R.whisper_full_get_token_data(ctx, i, j) for j in range(R.whisper_full_n_tokens(ctx, i))]
        sizes.append(len(toks)); ids += [t.id for t in toks]; want += [t.t_dtw for t in toks]
    n_text = sum(1 for t in ids if t < eot)
    assert n_text > 20 and nt.value == n_text + 3                       # sot, not, text..., eot (English-only model: no language token)
    assert sum(1 for w in want if w >= 0) == n_text                     # the reference stamped every text token
    n_frames = min(3000, len(pcm) // 160 + 1)                           # one window: min(30 s, seek_delta, seek_end - seek), src/whisper.cpp:7755
    R.whisper_n_len.argtypes = [vp]
    n_frames = min(3000, R.whisper_n_len(ctx))
    got = (C.c_int64 * len(ids))()
    lib.wb200_dbg_dtw.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, vp]
    ids_a = np.asarray(ids, np.int32); sizes_a = np.asarray(sizes, np.int32)
    npath = lib.wb200_dbg_dtw(qk.ctypes.data, nt.value, na.value, nh.value, n_frames, 1, 0, eot, ids_a.ctypes.data, sizes_a.ctypes.data, len(sizes), got)
    assert npath > 0
    assert list(got) == want, [(a, b) for a, b in zip(got, want) if a != b][:8]
    R.whisper_free(ctx)


def test_dtw_qk_kernel_phases_match_numpy(lib):
    """the phases of k_dtw_qk walked on the host (wb200_dbg_dtw_qk): softmax over the audio positions of f16(q) . K^T * 64^-1/4, for alignment
    heads spread over several layers, written [head][audio][token] like the reference's host copy"""
    rng = np.random.default_rng(3)
    d, Tp, n_ctx, n_tok, n_layers = 384, 1536, 1500, 7, 3
    heads = [(0, 1, 4), (0, 1, 0), (1, 2, 5)]                       # (captured-layer slot, text layer, head)
    q = (rng.standard_normal((2, n_tok, d)) * 3).astype(np.float32)
    k = (rng.standard_normal((n_layers, Tp, d)) * 0.5).astype(np.float16)
    out = np.empty((len(heads), n_ctx, n_tok), np.float32)
    tri = np.asarray(heads, np.int32)
    scale = np.float32(64.0) ** np.float32(-0.25)
    lib.wb200_dbg_dtw_qk.argtypes = [vp, vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_float, vp]
    assert lib.wb200_dbg_dtw_qk(q.ctypes.data, k.ctypes.data, Tp, d, tri.ctypes.data, len(heads), n_tok, n_ctx, C.c_float(float(scale)), out.ctypes.data) == 0
    for e, (ls, ly, hd) in enumerate(heads):
        qh = q[ls, :, 64 * hd:64 * hd + 64].astype(np.float16).astype(np.float64)
        kh = k[ly, :n_ctx, 64 * hd:64 * hd + 64].astype(np.float64)
        s = (qh @ kh.T) * float(scale)
        p = np.exp(s - s.max(axis=1, keepdims=True)); p /= p.sum(axis=1, keepdims=True)
        assert np.abs(out[e].T - p).max() < 2e-6 * max(1.0, p.max() * 1e3), e
        assert np.allclose(out[e].sum(axis=0), 1.0, atol=1e-5)


def test_alignment_head_tables_and_order_match_reference(lib, ref):
    """every preset of whisper_alignment_heads_preset resolves to the same (layer, head) list, in the same order, as the reference's tables"""
    if not hasattr(ref, "wref_dtw_heads"):
        pytest.skip("oracle/_ref predates wref_dtw_heads")
    from wbtest import ContextParams
    R = bind_whisper_api(ref)
    sig = [ContextParams, C.c_int, C.c_int, vp, C.c_int]
    ref.wref_dtw_heads.argtypes = sig; lib.wb200_dbg_dtw_heads.argtypes = sig
    shapes = {3: (4, 6), 4: (4, 6), 5: (6, 8), 6: (6, 8), 7: (12, 12), 8: (12, 12), 9: (24, 16), 10: (24, 16), 11: (32, 20), 12: (32, 20), 13: (32, 20), 14: (4, 20)}
    n_checked = 0
    for preset, (n_layer, n_head) in shapes.items():
        cp = R.whisper_context_default_params(); cp.dtw_token_timestamps = True; cp.dtw_aheads_preset = preset
        a = (C.c_int * 256)(); b = (C.c_int * 256)()
        na = lib.wb200_dbg_dtw_heads(cp, n_layer, n_head, a, 128); nb = ref.wref_dtw_heads(cp, n_layer, n_head, b, 128)
        assert na == nb > 0 and list(a[: 2 * na]) == list(b[: 2 * nb]), preset
        n_checked += na
    assert n_checked == 8 + 6 + 5 + 8 + 19 + 10 + 18 + 6 + 9 + 23 + 10 + 6
    cp = R.whisper_context_default_params(); cp.dtw_aheads_preset = 1; cp.dtw_n_top = 3
    a = (C.c_int * 256)(); b = (C.c_int * 256)()
    assert lib.wb200_dbg_dtw_heads(cp, 6, 8, a, 128) == ref.wref_dtw_heads(cp, 6, 8, b, 128) == 24 and list(a[:48]) == list(b[:48])
    cp.dtw_n_top = 7
    assert lib.wb200_dbg_dtw_heads(cp, 6, 8, a, 128) == -2                          # more layers than the model has
    cp.dtw_aheads_preset = 0
    assert lib.wb200_dbg_dtw_heads(cp, 6, 8, a, 128) == -2                          # DTW without a selection
    cp.dtw_aheads_preset = 5                                                        # base.en heads on a 4-layer model
    assert lib.wb200_dbg_dtw_heads(cp, 4, 6, a, 128) == -2
