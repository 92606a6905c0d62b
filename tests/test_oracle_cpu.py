"""CPU tests (no GPU): pin the NumPy restatement (oracle/ref_numpy.py) against the UNMODIFIED reference build
(oracle/_ref/libwhisper_ref.so) -- the reference ships no numeric golden vectors for this path (SURVEY.md 8c)."""
import ctypes as C
import os
import numpy as np
import pytest

from wbtest import (F16, Q4_0, Q5_0, Q8_0, Q4_K, Q5_K, ref_quantize, ref_dequantize, bind_whisper_api, read_wav_f32,
                    DATA_DIR, data_file, parse_model_header, ContextParams)
from oracle import ref_numpy as rn


@pytest.mark.parametrize("wtype", [Q4_0, Q5_0, Q8_0, Q4_K, Q5_K, F16])
def test_block_decoders_match_ggml(ref, wtype):
    rng = np.random.default_rng(wtype)
    w = (rng.standard_normal((16, 512)) * 0.1).astype(np.float32)
    w[3, :64] = 0.0
    raw = ref_quantize(ref, wtype, w)
    want = ref_dequantize(ref, wtype, raw, 16, 512)
    got = rn.dequantize(wtype, raw, 16, 512)
    assert np.array_equal(got, want)           # bit-exact: same f32 operations


def test_gelu_table_semantics(ref):
    ref.wref_fp16_round.restype = C.c_float
    ref.wref_fp16_round.argtypes = [C.c_float]
    x = np.linspace(-12, 12, 4001).astype(np.float32)
    y = rn.gelu(x)
    assert y[0] == 0.0 and y[-1] == x[-1]
    # the table output is an f16 value
    assert np.array_equal(y[(x > -10) & (x < 10)].astype(np.float16).astype(np.float32), y[(x > -10) & (x < 10)])


def _ref_ctx(ref, model):
    bind_whisper_api(ref)
    cp = ref.whisper_context_default_params()
    cp.use_gpu = False
    ctx = ref.whisper_init_from_file_with_params(os.path.join(DATA_DIR, model).encode(), cp)
    assert ctx
    return ctx


def test_log_mel_float64_restatement_vs_reference(ref):
    ref.wref_ctx_state.restype = C.c_void_p
    ref.wref_ctx_state.argtypes = [C.c_void_p]
    ref.wref_mel_copy.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    ref.wref_mel_n_len.argtypes = [C.c_void_p]
    ctx = _ref_ctx(ref, "for-tests-ggml-tiny.en.bin")
    pcm = read_wav_f32(os.path.join(DATA_DIR, "jfk.wav"))
    assert ref.whisper_pcm_to_mel(ctx, pcm.ctypes.data, len(pcm), 4) == 0
    st = ref.wref_ctx_state(ctx)
    n_len = ref.wref_mel_n_len(st)
    assert n_len == (len(pcm) + 480000) // 160
    mel = np.empty((80, n_len), np.float32)
    assert ref.wref_mel_copy(st, mel.ctypes.data, mel.size) == 0
    _, filt = parse_model_header(data_file("for-tests-ggml-tiny.en.bin"))
    want = rn.log_mel(pcm, filt)
    assert want.shape == mel.shape
    # reference computes the FFT in f32: agreement to ~1e-4 except in bins far below the frame energy
    assert np.abs(mel - want).max() < 2e-3
    assert np.abs(mel - want).mean() < 2e-5
    ref.whisper_free(ctx)


def test_q8_0_dot_restatement_matches_exact_math_within_quantisation_noise(ref):
    rng = np.random.default_rng(7)
    w = (rng.standard_normal((64, 256)) * 0.05).astype(np.float32)
    x = rng.standard_normal((3, 256)).astype(np.float32)
    for wtype in (Q4_0, Q5_0, Q8_0):
        raw = ref_quantize(ref, wtype, w)
        wd = rn.dequantize(wtype, raw, 64, 256)
        y = rn.mul_mat_q(wtype, raw, 64, 256, x)
        exact = x.astype(np.float64) @ wd.astype(np.float64).T
        rel = np.abs(y - exact).max() / np.abs(exact).max()
        assert rel < 2e-2      # the reference's own int8 activation noise (SURVEY.md fact 3)


@pytest.mark.parametrize("wtype,tol", [(F16, 8e-3), (Q5_0, 3e-2)])   # Q5_0: int8 activation rounding amplifies the f32-vs-f64 attention difference
def test_decoder_step_restatement_vs_reference(ref, tmp_path, wtype, tol):
    """oracle/ref_numpy.DecoderOracle (the text decoder of src/whisper.cpp:2466-2844 in NumPy, CPU arithmetic incl. the Q8_0
    activation quantisation) against the reference's own logits on the synthetic 2-layer model, fed with the reference's cross KV.

    Single-token steps agree to ~5e-3 of the logit std.  A multi-token (prompt) call does not, and not because of the restatement:
    the reference itself gives different logits for the same tokens fed in one batch or one by one (6-7e-2, asserted below) --
    its CPU flash-attention takes the split-KV path only for 1 query row (ops.cpp:9126) and otherwise accumulates P.V of all 1536
    cross keys in F16 (flash_attn_ext_f16_one_chunk, ops.cpp:8640-8660).  The restatement (f64 accumulation) sits at the
    single-row result; so do the CUDA kernels (tests/test_e2e_gpu.py)."""
    import importlib.util
    from wbtest import ROOT
    spec = importlib.util.spec_from_file_location("wb_synth", os.path.join(ROOT, "whisper.cpp_b200", "synth.py"))
    synth = importlib.util.module_from_spec(spec); spec.loader.exec_module(synth)
    path = str(tmp_path / "m.bin")
    synth.write_model(path, "test-2l.en", wtype, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    bind_whisper_api(ref)
    cp = ref.whisper_context_default_params(); cp.use_gpu = False
    ctx = ref.whisper_init_from_file_with_params(path.encode(), cp)
    assert ctx
    pcm = synth.synth_audio(seed=3, seconds=2.0)
    assert ref.whisper_pcm_to_mel(ctx, pcm.ctypes.data, len(pcm), 4) == 0
    assert ref.whisper_encode(ctx, 0, 4) == 0
    ref.wref_ctx_state.restype = C.c_void_p; ref.wref_ctx_state.argtypes = [C.c_void_p]
    st = ref.wref_ctx_state(ctx)
    L, d, Tp = 2, 384, 1536
    for nme in ("wref_kv_cross_k", "wref_kv_cross_v"):
        getattr(ref, nme).restype = C.c_int64; getattr(ref, nme).argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    kc = np.empty((L, Tp, d), np.float16); vc = np.empty((L, Tp, d), np.float16)
    assert ref.wref_kv_cross_k(st, kc.ctypes.data, kc.size) == kc.size and ref.wref_kv_cross_v(st, vc.ctypes.data, vc.size) == vc.size
    kc = kc.astype(np.float32); vc = vc.astype(np.float32)
    n_vocab = ref.whisper_n_vocab(ctx)
    ref.whisper_get_logits.restype = C.POINTER(C.c_float)
    sot = ref.whisper_token_sot(ctx)

    def ref_decode(feed, n_past):
        t = np.asarray(feed, np.int32)
        assert ref.whisper_decode(ctx, t.ctypes.data, len(t), n_past, 4) == 0
        return np.ctypeslib.as_array(ref.whisper_get_logits(ctx), shape=(len(t) * n_vocab,))[-n_vocab:].copy()

    def rms(a, b):
        return float(np.sqrt(((a - b) ** 2).mean()) / b.std())

    toks = [sot, 100, 200]
    batched = ref_decode(toks, 0)                                # the reference, three tokens in one call
    dec = rn.DecoderOracle(path)
    for i, tk in enumerate(toks):                                # the same tokens one by one: reference and restatement
        want = ref_decode([tk], i)
        got = dec.step([tk], i, kc, vc)
        assert rms(got, want) < tol, (i, rms(got, want))
    assert rms(batched, want) > 3 * rms(got, want)               # the reference's own batch-vs-sequential gap is the larger one
    assert rms(rn.DecoderOracle(path).step(toks, 0, kc, vc), want) < tol      # the restatement does not care how the tokens are fed
    n_past = len(toks)
    for step in range(2):                                        # two more greedy steps
        nxt = int(want.argmax())
        want = ref_decode([nxt], n_past); got = dec.step([nxt], n_past, kc, vc); n_past += 1
        assert rms(got, want) < tol, (step, rms(got, want))
        srt = np.sort(want)
        assert int(got.argmax()) == int(want.argmax()) or srt[-1] - srt[-2] < 10 * tol * want.std()
    ref.whisper_free(ctx)


@pytest.mark.parametrize("wtype,tol_enc,tol_kv", [(F16, 1e-3, 1e-4), (Q5_0, 1e-2, 1e-4)])     # measured: 2.2e-4 / 3.1e-3 and 7e-6
def test_encoder_restatement_vs_reference(ref, tmp_path, wtype, tol_enc, tol_kv):
    """oracle/ref_numpy.EncoderOracle (conv stem, encoder, cross K/V of src/whisper.cpp:1982-2354 in NumPy with the CPU backend's rounding
    points) against the reference's own tensors on the synthetic 2-layer model.  F16 weights: the difference is accumulation order / width
    (f64 here, f32 and F16 P.V there).  Q5_0: additionally every row's Q8_0 activation blocks can round differently once the inputs differ
    in the last bit, the same ~1e-2 noise floor the GPU parity tests allow (tests/test_e2e_gpu.py TOL)."""
    import importlib.util
    from wbtest import ROOT
    spec = importlib.util.spec_from_file_location("wb_synth", os.path.join(ROOT, "whisper.cpp_b200", "synth.py"))
    synth = importlib.util.module_from_spec(spec); spec.loader.exec_module(synth)
    path = str(tmp_path / "m.bin")
    synth.write_model(path, "test-2l.en", wtype, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    bind_whisper_api(ref)
    cp = ref.whisper_context_default_params(); cp.use_gpu = False
    ctx = ref.whisper_init_from_file_with_params(path.encode(), cp)
    assert ctx
    pcm = synth.synth_audio(seed=5, seconds=4.0)
    assert ref.whisper_pcm_to_mel(ctx, pcm.ctypes.data, len(pcm), 4) == 0
    assert ref.whisper_encode(ctx, 0, 4) == 0
    vp = C.c_void_p
    ref.wref_ctx_state.restype = vp; ref.wref_ctx_state.argtypes = [vp]
    st = ref.wref_ctx_state(ctx)
    ref.wref_mel_n_len.argtypes = [vp]; ref.wref_mel_n_mel.argtypes = [vp]; ref.wref_mel_copy.argtypes = [vp, vp, C.c_int64]
    n_len, n_mel = ref.wref_mel_n_len(st), ref.wref_mel_n_mel(st)
    mel = np.empty((n_mel, n_len), np.float32)
    assert ref.wref_mel_copy(st, mel.ctypes.data, mel.size) == 0
    L, d, T, Tp = 2, 384, 1500, 1536
    for nme in ("wref_embd_conv", "wref_embd_enc", "wref_kv_cross_k", "wref_kv_cross_v"):
        getattr(ref, nme).restype = C.c_int64; getattr(ref, nme).argtypes = [vp, vp, C.c_int64]
    conv = np.empty((d, T), np.float32); enc = np.empty((T, d), np.float32)
    assert ref.wref_embd_conv(st, conv.ctypes.data, conv.size) == conv.size and ref.wref_embd_enc(st, enc.ctypes.data, enc.size) == enc.size
    kc = np.empty((L, Tp, d), np.float16); vc = np.empty((L, Tp, d), np.float16)
    assert ref.wref_kv_cross_k(st, kc.ctypes.data, kc.size) == kc.size and ref.wref_kv_cross_v(st, vc.ctypes.data, vc.size) == vc.size
    ref.whisper_free(ctx)

    def rms(a, b):
        return float(np.sqrt(((np.asarray(a, np.float64) - b) ** 2).mean()) / np.sqrt((np.asarray(b, np.float64) ** 2).mean()))

    E = rn.EncoderOracle(path)
    my_conv = E.conv(mel[:, :2 * T])
    e_conv = rms(my_conv, conv)
    my_enc = E.encode(conv)                                       # fed with the reference's conv output: errors do not compound
    e_enc = rms(my_enc, enc)
    my_k, my_v = E.cross(enc)
    e_k, e_v = rms(my_k, kc[:, :T].astype(np.float32)), rms(my_v, vc[:, :T].astype(np.float32))
    print("encoder restatement (%d): conv %.2e  enc %.2e  cross K %.2e  V %.2e" % (wtype, e_conv, e_enc, e_k, e_v))
    assert e_conv < 1e-4                                          # F16 x F16 products, f32 vs f64 sums (measured 7e-6)
    assert e_enc < tol_enc
    assert e_k < tol_kv and e_v < tol_kv
    assert np.abs(kc[:, T:].astype(np.float32)).max() == 0 and np.abs(vc[:, T:].astype(np.float32)).max() == 0      # the 36 padded keys
