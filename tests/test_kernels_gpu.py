"""Kernel-level parity on the GPU (through the wb200_dbg_* C entry points of libwhisper_b200.so).

Oracles: the compiled reference (oracle/_ref) for log-mel, oracle/ref_numpy.py (pinned to the reference in
test_oracle_cpu.py) for the integer GEMV, LayerNorm and the decode attention.  Tolerances are stated per test.
"""
import ctypes as C
import os
import numpy as np
import pytest

from wbtest import (F16, Q4_0, Q5_0, Q8_0, Q4_K, Q5_K, ref_quantize, bind_whisper_api, read_wav_f32, DATA_DIR, data_file,
                    parse_model_header)
from oracle import ref_numpy as rn

pytestmark = pytest.mark.gpu
vp = C.c_void_p


def _ptr(a):
    return a.ctypes.data_as(vp) if a is not None else None


def test_log_mel_matches_reference_on_jfk(lib, ref):
    """device STFT+mel vs whisper_pcm_to_mel (src/whisper.cpp:3178-3272).  Both are f32 pipelines with different
    summation orders (direct DFT vs radix-2 recursion): abs tol 2e-3 on the normalised log-mel, mean 2e-5."""
    bind_whisper_api(ref)
    ref.wref_ctx_state.restype = vp; ref.wref_ctx_state.argtypes = [vp]
    ref.wref_mel_copy.argtypes = [vp, vp, C.c_int64]
    ref.wref_mel_n_len.argtypes = [vp]
    cp = ref.whisper_context_default_params(); cp.use_gpu = False
    model = data_file("for-tests-ggml-tiny.en.bin")
    ctx = ref.whisper_init_from_file_with_params(model.encode(), cp)
    _, filt = parse_model_header(model)
    pcm_full = read_wav_f32(os.path.join(DATA_DIR, "jfk.wav"))
    for n in (len(pcm_full), 16000, 150, 1, 479999 % len(pcm_full)):
        pcm = np.ascontiguousarray(pcm_full[:n])
        assert ref.whisper_pcm_to_mel(ctx, _ptr(pcm), n, 4) == 0
        st = ref.wref_ctx_state(ctx)
        n_len = ref.wref_mel_n_len(st)
        want = np.empty((80, n_len), np.float32)
        assert ref.wref_mel_copy(st, _ptr(want), want.size) == 0
        got = np.empty((80, n_len), np.float32)
        rc = lib.wb200_dbg_mel(_ptr(pcm), n, _ptr(filt), 80, _ptr(got), C.c_int64(got.size))
        assert rc == n_len, (rc, lib.wb200_last_error())
        err = np.abs(got - want)
        assert err.max() < 2e-3 and err.mean() < 2e-5, (n, err.max(), err.mean())
    ref.whisper_free(ctx)


def test_layernorm(lib):
    rng = np.random.default_rng(3)
    for rows, d in ((7, 384), (1500, 1280), (3, 512)):
        x = (rng.standard_normal((rows, d)) * 3 + 0.5).astype(np.float32)
        w = (1 + 0.1 * rng.standard_normal(d)).astype(np.float32)
        b = (0.1 * rng.standard_normal(d)).astype(np.float32)
        o32 = np.empty((rows, d), np.float32); o16 = np.empty((rows, d), np.uint16)
        assert lib.wb200_dbg_layernorm(_ptr(x), _ptr(w), _ptr(b), C.c_float(1e-5), rows, d, _ptr(o32), _ptr(o16)) == 0
        want = rn.layernorm(x, w, b)
        assert np.abs(o32 - want).max() < 2e-5            # f32 summation order only
        assert np.array_equal(o16.view(np.float16), o32.astype(np.float16))


@pytest.mark.parametrize("v2", [0, 4])
@pytest.mark.parametrize("wtype", [Q4_0, Q5_0, Q8_0, F16])
@pytest.mark.parametrize("N,K,n_tok", [(384, 384, 1), (1280, 1280, 1), (1000, 5120, 3), (51864, 384, 1), (640, 1280, 8), (1290, 1280, 5)])
def test_gemv_integer_dot_matches_reference_arithmetic(lib, ref, wtype, N, K, n_tok, v2):
    """same integer arithmetic as the CPU mul_mat (Q8_0 activations, int dot, f32 block sums): only the f32
    summation order differs -> rel tol 2e-5 of the output scale."""
    rng = np.random.default_rng(N + K + n_tok + wtype)
    w = (rng.standard_normal((N, K)) * 0.05).astype(np.float32)
    x = rng.standard_normal((n_tok, K)).astype(np.float32)
    bias = rng.standard_normal(N).astype(np.float32)
    scale = (0.5 + rng.random(N)).astype(np.float32)
    res = rng.standard_normal((n_tok, N)).astype(np.float32)
    raw = ref_quantize(ref, wtype, w)
    out = np.empty((n_tok, N), np.float32)
    rawb = np.frombuffer(raw, dtype=np.uint8)
    rc = lib.wb200_dbg_gemv(wtype, N, K, n_tok, _ptr(rawb), _ptr(x), _ptr(bias), _ptr(scale), _ptr(res), None, None, _ptr(out), v2)
    assert rc == 0, lib.wb200_last_error()
    y = rn.mul_mat_f16(raw, N, K, x) if wtype == F16 else rn.mul_mat_q(wtype, raw, N, K, x)
    want = (y + bias[None, :]) * scale[None, :] + res
    tol = 2e-5 * (np.abs(y).max() + 1.0)
    assert np.abs(out - want).max() < tol, np.abs(out - want).max()


@pytest.mark.parametrize("v2", [0, 4])
@pytest.mark.parametrize("wtype", [Q4_K, Q5_K])
def test_gemv_kquants_within_activation_quantisation_noise(lib, ref, wtype, v2):
    """K-quant GEMV uses Q8_K activations like the reference (ggml-quants.c:2768-2805); checked against exact math
    with the reference's own int8 noise budget (1e-2 of the output scale)."""
    rng = np.random.default_rng(5)
    N, K, n_tok = 512, 1280, 2
    w = (rng.standard_normal((N, K)) * 0.05).astype(np.float32)
    x = rng.standard_normal((n_tok, K)).astype(np.float32)
    raw = ref_quantize(ref, wtype, w)
    wd = rn.dequantize(wtype, raw, N, K).astype(np.float64)
    out = np.empty((n_tok, N), np.float32)
    rawb = np.frombuffer(raw, dtype=np.uint8)
    rc = lib.wb200_dbg_gemv(wtype, N, K, n_tok, _ptr(rawb), _ptr(x), None, None, None, None, None, _ptr(out), v2)
    assert rc == 0, lib.wb200_last_error()
    want = x.astype(np.float64) @ wd.T
    assert np.abs(out - want).max() < 1e-2 * np.abs(want).max()


@pytest.mark.parametrize("v2", [0, 4])
def test_gemv_fused_layernorm_and_gelu(lib, ref, v2):
    rng = np.random.default_rng(11)
    N, K, n_tok = 1536, 384, 2
    w = (rng.standard_normal((N, K)) * 0.05).astype(np.float32)
    x = (rng.standard_normal((n_tok, K)) * 2 + 1).astype(np.float32)
    lw = (1 + 0.1 * rng.standard_normal(K)).astype(np.float32); lb = (0.1 * rng.standard_normal(K)).astype(np.float32)
    bias = rng.standard_normal(N).astype(np.float32)
    raw = ref_quantize(ref, Q5_0, w)
    out = np.empty((n_tok, N), np.float32)
    rawb = np.frombuffer(raw, dtype=np.uint8)
    rc = lib.wb200_dbg_gemv(Q5_0, N, K, n_tok, _ptr(rawb), _ptr(x), _ptr(bias), None, None, _ptr(lw), _ptr(lb), _ptr(out), 3 | v2)
    assert rc == 0, lib.wb200_last_error()
    xn = rn.layernorm(x, lw, lb)
    want = rn.gelu(rn.mul_mat_q(Q5_0, raw, N, K, xn) + bias[None, :])
    # LN summation order can move an activation across an int8 rounding edge: allow 1e-3 of the scale, but require
    # that the bulk agrees to f16-ulp level
    err = np.abs(out - want)
    assert err.max() < 5e-3 * (np.abs(want).max() + 1) and np.median(err) < 1e-4


def test_attention_decode_kernels(lib):
    rng = np.random.default_rng(2)
    n_head, d = 6, 384
    n_cells, n_tok, ld = 40, 3, 32
    kc = (rng.standard_normal((n_cells, d))).astype(np.float16); vc = rng.standard_normal((n_cells, d)).astype(np.float16)
    q = rng.standard_normal((n_tok, d)).astype(np.float32)
    n_kv = np.array([5, 17, 32], np.int32)
    idx = np.zeros((n_tok, ld), np.int32)
    for t in range(n_tok):
        idx[t, :n_kv[t]] = rng.permutation(n_cells)[:n_kv[t]]
    out = np.empty((n_tok, d), np.float32)
    assert lib.wb200_dbg_attn_self(_ptr(q), _ptr(kc), _ptr(vc), _ptr(idx), ld, _ptr(n_kv), n_tok, n_head, n_cells, _ptr(out)) == 0, lib.wb200_last_error()
    for t in range(n_tok):
        cells = idx[t, :n_kv[t]]
        for h in range(n_head):
            sl = slice(h * 64, h * 64 + 64)
            want = rn.attention(q[t:t + 1, sl], kc[cells][:, sl].astype(np.float32), vc[cells][:, sl].astype(np.float32), 1.0)
            assert np.abs(out[t, sl] - want[0]).max() < 1e-4
    # cross attention over 1536 keys of which the last 36 are all-zero and NOT masked (SURVEY.md fact 4)
    n_keys = 1536
    kx = np.zeros((n_tok, n_keys, d), np.float16); vx = np.zeros((n_tok, n_keys, d), np.float16)
    kx[:, :1500] = (rng.standard_normal((n_tok, 1500, d)) * 0.3).astype(np.float16)
    vx[:, :1500] = rng.standard_normal((n_tok, 1500, d)).astype(np.float16)
    scale = 64.0 ** -0.25
    assert lib.wb200_dbg_attn_cross(_ptr(q), _ptr(kx), _ptr(vx), n_keys, n_tok, n_head, C.c_float(scale), _ptr(out)) == 0, lib.wb200_last_error()
    for t in range(n_tok):
        for h in range(n_head):
            sl = slice(h * 64, h * 64 + 64)
            want = rn.attention(q[t:t + 1, sl], kx[t, :1500, sl].astype(np.float32), vx[t, :1500, sl].astype(np.float32), scale, n_zero_keys=36)
            assert np.abs(out[t, sl] - want[0]).max() < 1e-4


def test_encoder_flash_attention_kernel(lib):
    """fattn_enc_kernel (wb_fattn.cu) alone against a float64 softmax(Q K^T) V over the 1536 padded keys: 1500 real + 36 all-zero rows that take
    part in the softmax (SURVEY.md fact 4).  Two windows, ragged last query tile (1500 = 11 x 128 + 92).  Tolerance: the kernel rounds the
    probabilities to f16 for the tensor core (2^-11 relative each) and the output to f16."""
    rng = np.random.default_rng(11)
    T, Tp, H, n_win = 1500, 1536, 3, 2
    d = H * 64
    q = (rng.standard_normal((n_win, T, d)) * 1.5).astype(np.float32); k = rng.standard_normal((n_win, T, d)).astype(np.float32)
    v = rng.standard_normal((n_win, T, d)).astype(np.float32)
    out = np.empty((n_win, T, d), np.float32)
    scale = 1.0 / 8.0
    lib.wb200_dbg_fattn.restype = C.c_int
    assert lib.wb200_dbg_fattn(_ptr(q), _ptr(k), _ptr(v), T, Tp, H, n_win, C.c_float(scale), _ptr(out)) == 0, lib.wb200_last_error()
    q16 = q.astype(np.float16).astype(np.float64); k16 = k.astype(np.float16).astype(np.float64); v16 = v.astype(np.float16).astype(np.float64)
    worst = 0.0
    for w in range(n_win):
        for h in range(H):
            sl = slice(h * 64, h * 64 + 64)
            s_ = q16[w, :, sl] @ k16[w, :, sl].T * scale                                   # [T][T]
            s_ = np.concatenate([s_, np.zeros((T, Tp - T))], axis=1)                        # the zero keys score 0
            p_ = np.exp(s_ - s_.max(axis=1, keepdims=True)); p_ /= p_.sum(axis=1, keepdims=True)
            want = p_[:, :T] @ v16[w, :, sl]
            worst = max(worst, float(np.abs(out[w, :, sl] - want).max()))
    print("encoder attention kernel: worst abs error %.2e" % worst)
    assert worst < 4e-3


def test_whisper_bench_entry_points_measure_the_device(lib):
    """whisper_bench_memcpy_str / whisper_bench_ggml_mul_mat_str (whisper.h:746-753, `whisper-bench -w 1|2`) report device copy bandwidth
    and tcgen05 GEMM throughput"""
    import ctypes as C
    import re
    lib.whisper_bench_memcpy_str.restype = C.c_char_p; lib.whisper_bench_ggml_mul_mat_str.restype = C.c_char_p
    s = lib.whisper_bench_memcpy_str(1).decode()
    gbs = [float(x) for x in re.findall(r"([\d.]+) GB/s", s)]
    assert gbs and gbs[0] > 1000.0, s
    s = lib.whisper_bench_ggml_mul_mat_str(1).decode()
    tf = [float(x) for x in re.findall(r"([\d.]+) TFLOP/s", s)]
    assert len(tf) == 6 and max(tf) > 300.0, s
    print(s)
