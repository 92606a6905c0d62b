"""CPU tests of the synthetic-model tooling (whisper.cpp_b200/synth.py): the NumPy block quantisers are bit-identical
to ggml's reference quantisers, the mel filterbank equals the one shipped inside the reference's own model files, and
the files it writes load in the UNMODIFIED reference (loader/format parity, src/whisper.cpp:1485-1962)."""
import importlib.util
import os
import ctypes as C
import numpy as np
import pytest

from wbtest import ROOT, data_file, Q4_0, Q5_0, Q8_0, F16, ref_quantize, bind_whisper_api, parse_model_header

spec = importlib.util.spec_from_file_location("wb_synth", os.path.join(ROOT, "whisper.cpp_b200", "synth.py"))
synth = importlib.util.module_from_spec(spec); spec.loader.exec_module(synth)


@pytest.mark.parametrize("wtype", [Q4_0, Q5_0, Q8_0])
def test_numpy_quantisers_bit_exact_vs_ggml(ref, wtype):
    rng = np.random.default_rng(wtype)
    w = (rng.standard_normal((64, 1280)) * 0.02).astype(np.float32)
    w[0, :32] = 0.0
    w[1, 5] = 0.5
    assert synth.quantize(wtype, w) == ref_quantize(ref, wtype, w)


@pytest.mark.parametrize("stub,n_mels", [("for-tests-ggml-tiny.en.bin", 80)])
def test_mel_filterbank_matches_reference_model_files(stub, n_mels):
    _, filt = parse_model_header(data_file(stub))
    mine = synth.mel_filters(n_mels)
    assert mine.shape == filt.shape
    assert np.abs(mine - filt).max() < 1e-6


@pytest.mark.parametrize("wtype", [F16, Q5_0])
def test_written_model_loads_in_reference(ref, tmp_path, wtype):
    bind_whisper_api(ref)
    path = str(tmp_path / "m.bin")
    synth.write_model(path, "test-2l.en", wtype, seed=1, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    cp = ref.whisper_context_default_params(); cp.use_gpu = False
    ctx = ref.whisper_init_from_file_with_params(path.encode(), cp)
    assert ctx
    assert ref.whisper_model_n_audio_layer(ctx) == 2 and ref.whisper_model_n_text_state(ctx) == 384
    assert ref.whisper_model_ftype(ctx) == synth.FTYPE_OF[wtype]
    assert ref.whisper_token_to_str(ctx, 220) == b" "
    ref.whisper_free(ctx)


@pytest.mark.parametrize("wtype", [synth.Q5_1, synth.Q6_K, synth.Q4_1, synth.Q2_K, synth.Q3_K, synth.BF16])
def test_host_expanded_formats_load_in_reference_and_parse_here(lib, ref, tmp_path, wtype):
    """files in the formats this engine expands to F16 at load time (csrc/wb_dequant_host.cpp): written with ggml's own quantisers, they load
    in the reference, and this library's header parser accepts the ftype (the weight upload itself needs a GPU: tests/test_wider_formats_gpu.py)"""
    from wbtest import ref_quantize
    bind_whisper_api(ref); bind_whisper_api(lib)
    path = str(tmp_path / "m.bin")
    cfg = "test-2l-512.en" if wtype in (synth.Q2_K, synth.Q3_K, synth.Q6_K) else "test-2l.en"          # K-quants need rows of 256
    synth.write_model(path, cfg, wtype, seed=1, vocab_from=data_file("for-tests-ggml-tiny.en.bin"), quantizer=lambda t, w: ref_quantize(ref, t, w))
    cp = ref.whisper_context_default_params(); cp.use_gpu = False
    ctx = ref.whisper_init_from_file_with_params(path.encode(), cp)
    assert ctx
    assert ref.whisper_model_ftype(ctx) == synth.FTYPE_OF[wtype]
    ref.whisper_free(ctx)
    lib.wb200_dbg_vocab_context.restype = C.c_void_p; lib.wb200_dbg_vocab_context.argtypes = [C.c_char_p]
    mine = lib.wb200_dbg_vocab_context(path.encode())
    assert mine, lib.wb200_last_error()
    assert lib.whisper_model_ftype(mine) == synth.FTYPE_OF[wtype] and lib.whisper_model_n_text_layer(mine) == 2


def test_simple_q4_k_writer_is_valid_q4_k(ref):
    """synth.quantize_q4_k_simple (the multi-GB benchmark model of BASELINE config 3) writes super-blocks the reference's
    dequantize_row_q4_K reads back close to the input; it is NOT ggml's quantiser (parity tests use ggml_quantize_chunk)"""
    from wbtest import ref_dequantize, Q4_K
    rng = np.random.default_rng(3)
    w = (rng.standard_normal((6, 1024)) * 0.02).astype(np.float32)
    w[1, :300] = 0.0
    raw = synth.quantize(Q4_K, w)
    assert len(raw) == 6 * 4 * 144
    deq = ref_dequantize(ref, Q4_K, raw, 6, 1024)
    assert np.sqrt(((deq - w) ** 2).mean()) / w.std() < 0.12
    assert np.abs(deq[1, :256]).max() < 1e-6
