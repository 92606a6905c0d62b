"""CPU: tokenizer, special tokens, token strings, language tables and model-shape getters of libwhisper_b200.so against the
reference on the weight-less stubs (real vocabularies), through a vocabulary-only context (wb200_dbg_vocab_context: no CUDA)."""
import ctypes as C
import os
import pytest

from wbtest import data_file, bind_whisper_api

vp = C.c_void_p
TEXTS = ["", " ", "hello world", " Hello, World!", "And so my fellow Americans, ask not what your country can do for you.",
         "it's 12:45pm -- don't", "  multiple   spaces\ttab\nnewline ", "naïve café 東京 ☃", "1234567890 3.14159", "[_BEG_] <|endoftext|>"]


@pytest.mark.parametrize("stub", ["for-tests-ggml-tiny.en.bin", "for-tests-ggml-tiny.bin", "for-tests-ggml-large.bin"])
def test_vocabulary_and_tokenizer_match_reference(lib, ref, stub):
    L = bind_whisper_api(lib); R = bind_whisper_api(ref)
    path = data_file(stub).encode()
    cp = R.whisper_context_default_params(); cp.use_gpu = False
    rctx = R.whisper_init_from_file_with_params(path, cp)
    assert rctx
    L.wb200_dbg_vocab_context.restype = vp; L.wb200_dbg_vocab_context.argtypes = [C.c_char_p]
    lctx = L.wb200_dbg_vocab_context(path)
    assert lctx
    for name in ("whisper_n_vocab", "whisper_n_text_ctx", "whisper_n_audio_ctx", "whisper_is_multilingual", "whisper_model_n_vocab", "whisper_model_n_audio_ctx",
                 "whisper_model_n_audio_state", "whisper_model_n_audio_head", "whisper_model_n_audio_layer", "whisper_model_n_text_ctx", "whisper_model_n_text_state",
                 "whisper_model_n_text_head", "whisper_model_n_text_layer", "whisper_model_n_mels", "whisper_model_ftype", "whisper_model_type",
                 "whisper_token_eot", "whisper_token_sot", "whisper_token_solm", "whisper_token_prev", "whisper_token_nosp", "whisper_token_not", "whisper_token_beg",
                 "whisper_token_translate", "whisper_token_transcribe"):
        for lib_ in (L, R):
            getattr(lib_, name).argtypes = [vp]; getattr(lib_, name).restype = C.c_int
        assert getattr(L, name)(lctx) == getattr(R, name)(rctx), name
    for lib_ in (L, R):
        lib_.whisper_token_lang.argtypes = [vp, C.c_int]; lib_.whisper_token_to_str.argtypes = [vp, C.c_int]; lib_.whisper_token_to_str.restype = C.c_char_p
        lib_.whisper_tokenize.argtypes = [vp, C.c_char_p, vp, C.c_int]; lib_.whisper_token_count.argtypes = [vp, C.c_char_p]
        lib_.whisper_model_type_readable.argtypes = [vp]; lib_.whisper_model_type_readable.restype = C.c_char_p
        lib_.whisper_lang_id.argtypes = [C.c_char_p]; lib_.whisper_lang_str.argtypes = [C.c_int]; lib_.whisper_lang_str.restype = C.c_char_p
        lib_.whisper_lang_str_full.argtypes = [C.c_int]; lib_.whisper_lang_str_full.restype = C.c_char_p
    assert L.whisper_model_type_readable(lctx) == R.whisper_model_type_readable(rctx)
    n_vocab = R.whisper_n_vocab(rctx)
    for i in list(range(0, n_vocab, 97)) + list(range(n_vocab - 1700, n_vocab)):
        assert L.whisper_token_to_str(lctx, i) == R.whisper_token_to_str(rctx, i), i
    for lid in range(0, R.whisper_lang_max_id() + 1):
        assert L.whisper_lang_str(lid) == R.whisper_lang_str(lid) and L.whisper_lang_str_full(lid) == R.whisper_lang_str_full(lid)
        assert L.whisper_lang_id(R.whisper_lang_str(lid)) == lid
        assert L.whisper_token_lang(lctx, lid) == R.whisper_token_lang(rctx, lid)
    assert L.whisper_lang_max_id() == R.whisper_lang_max_id()
    for text in TEXTS:
        t = text.encode("utf-8")
        a = (C.c_int * 256)(); b = (C.c_int * 256)()
        na = L.whisper_tokenize(lctx, t, a, 256); nb = R.whisper_tokenize(rctx, t, b, 256)
        assert na == nb and list(a[:max(na, 0)]) == list(b[:max(nb, 0)]), text
        assert L.whisper_token_count(lctx, t) == R.whisper_token_count(rctx, t), text
        assert L.whisper_tokenize(lctx, t, a, 1) == R.whisper_tokenize(rctx, t, b, 1), text      # too-small buffer: -n
    R.whisper_free(rctx)


def test_header_parser_rejects_bad_files(lib, tmp_path):
    """loader error paths that need no device (src/whisper.cpp:1497-1500, 1589-1600): bad magic, truncated header / vocabulary"""
    L = bind_whisper_api(lib)
    L.wb200_dbg_vocab_context.restype = vp; L.wb200_dbg_vocab_context.argtypes = [C.c_char_p]
    good = open(data_file("for-tests-ggml-tiny.en.bin"), "rb").read()
    cases = {"magic.bin": b"\x00\x01\x02\x03" + good[4:], "short_header.bin": good[:30], "short_vocab.bin": good[:4 + 44 + 8 + 80 * 201 * 4 + 4 + 1000],
             "empty.bin": b""}
    for name, blob in cases.items():
        p = tmp_path / name
        p.write_bytes(blob)
        assert not L.wb200_dbg_vocab_context(str(p).encode()), name
    assert not L.wb200_dbg_vocab_context(b"/nonexistent/model.bin")
    ok = tmp_path / "ok.bin"; ok.write_bytes(good)
    assert L.wb200_dbg_vocab_context(str(ok).encode())
