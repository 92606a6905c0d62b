"""GPU: checkpoints in ggml formats that have no device kernels here (Q5_1, Q4_1, Q6_K, Q3_K, Q2_K, BF16) -- expanded to F16 on the host at load
time (csrc/wb_dequant_host.cpp, pinned against ggml's to_float by tests/test_dequant_cpu.py) and run by the F16 kernels -- against the
reference CPU build on the same file.  The reference multiplies these blocks with int8 activation blocks (Q8_1 / Q8_K), so its own
outputs carry the same ~1e-2 activation-quantisation noise as for Q5_0 / Q4_K; the tolerances are those of tests/test_e2e_gpu.py for the
format of equal bit width.  (Not run on a GPU in round 1: the GPU budget was spent; the F16 device path itself is covered there.)"""
import os
import numpy as np
import pytest

os.environ["WB200_DEBUG_TAPS"] = "1"
from wbtest import DATA_DIR, data_file, read_wav_f32, ref_quantize
from e2e_util import Side, synth, taps, rms_err

pytestmark = pytest.mark.gpu

#                 cfg,               enc rms, kv rms, logits rms (of std), argmax margin (std)
CASES = {synth.Q5_1: ("test-2l.en",     3e-2, 3.5e-2, 5e-2, 0.3), synth.Q4_1: ("test-2l.en",     4e-2, 5e-2, 7e-2, 0.4),
         synth.Q6_K: ("test-2l-512.en", 3e-2, 3.5e-2, 5e-2, 0.3), synth.Q3_K: ("test-2l-512.en", 8e-2, 1e-1, 1.2e-1, 0.6),
         synth.Q2_K: ("test-2l-512.en", 1.5e-1, 1.8e-1, 2.2e-1, 1.0),
         synth.BF16: ("test-2l.en",     1.5e-2, 2e-2, 3e-2, 0.2)}        # the reference rounds activations to bf16 (8 mantissa bits)


@pytest.mark.parametrize("wt", [synth.Q5_1, synth.Q6_K, synth.Q4_1, synth.Q3_K, synth.Q2_K, synth.BF16])
def test_host_expanded_formats_match_reference(lib, ref, tmp_path, wt):
    cfg, e_enc, e_kv, e_log, margin = CASES[wt]
    path = str(tmp_path / "m.bin")
    synth.write_model(path, cfg, wt, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"), quantizer=lambda t, w: ref_quantize(ref, t, w))
    pcm = read_wav_f32(os.path.join(DATA_DIR, "jfk.wav"))
    A = Side(lib, path, False); B = Side(ref, path, True)
    try:
        assert A.L.whisper_model_ftype(A.ctx) == B.L.whisper_model_ftype(B.ctx) == synth.FTYPE_OF[wt]
        A.pcm_to_mel(pcm); B.pcm_to_mel(pcm)
        A.encode(0); B.encode(0)
        ta, tb = taps(A), taps(B)
        assert rms_err(ta["enc"], tb["enc"]) < e_enc, rms_err(ta["enc"], tb["enc"])
        assert rms_err(ta["kc"], tb["kc"]) < e_kv and rms_err(ta["kv"], tb["kv"]) < e_kv
        sot = A.L.whisper_token_sot(A.ctx)
        toks = [sot]; n_past = 0
        for step in range(8):
            feed = toks if step == 0 else toks[-1:]
            la = A.decode(feed, n_past); lb = B.decode(feed, n_past)
            n_past += len(feed)
            assert np.isfinite(la).all()
            err = rms_err(la - lb.mean(), lb - lb.mean())
            assert err < e_log, (step, err)
            srt = np.sort(lb)
            if (srt[-1] - srt[-2]) / lb.std() > margin:
                assert int(la.argmax()) == int(lb.argmax()), step
            toks.append(int(lb.argmax()))
    finally:
        A.free(); B.free()


@pytest.mark.parametrize("wt", [synth.Q4_K, synth.Q5_K])
def test_kquants_expanded_to_f16_opt_in(lib, ref, tmp_path, monkeypatch, wt):
    """WB200_KQUANT_AS_F16=1: Q4_K / Q5_K files through the persistent decode kernel as F16 matrices (default: kernel chain on the blocks)"""
    monkeypatch.setenv("WB200_KQUANT_AS_F16", "1")
    e_enc, e_kv, e_log, margin = (4e-2, 5e-2, 7e-2, 0.4) if wt == synth.Q4_K else (3e-2, 3.5e-2, 5e-2, 0.3)     # tests/test_e2e_gpu.py TOL
    path = str(tmp_path / "m.bin")
    synth.write_model(path, "test-2l-512.en", wt, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"), quantizer=lambda t, w: ref_quantize(ref, t, w))
    pcm = read_wav_f32(os.path.join(DATA_DIR, "jfk.wav"))
    A = Side(lib, path, False); B = Side(ref, path, True)
    try:
        A.pcm_to_mel(pcm); B.pcm_to_mel(pcm)
        A.encode(0); B.encode(0)
        ta, tb = taps(A), taps(B)
        assert rms_err(ta["enc"], tb["enc"]) < e_enc
        sot = A.L.whisper_token_sot(A.ctx)
        toks = [sot]; n_past = 0
        for step in range(6):
            feed = toks if step == 0 else toks[-1:]
            la = A.decode(feed, n_past); lb = B.decode(feed, n_past)
            n_past += len(feed)
            assert rms_err(la - lb.mean(), lb - lb.mean()) < e_log, step
            toks.append(int(lb.argmax()))
    finally:
        A.free(); B.free()
