"""Shared helpers for the tests: library loading, ctypes mirrors of the ABI structs, numpy (de)quantisers.

The reference library (oracle/_ref) is only ever used as a CHECKER here.
"""
import ctypes as C
import os
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.environ.get("WB200_LIB") or os.path.join(ROOT, "whisper.cpp_b200", "libwhisper_b200.so")      # WB200_LIB: instrumented / A-B builds (scripts/sanitize_host.sh)
REF_PATH = os.path.join(ROOT, "oracle", "_ref", "libwhisper_ref.so")

# ggml_type ids (ggml/include/ggml.h:390-405)
F32, F16, Q4_0, Q5_0, Q8_0, Q4_K, Q5_K = 0, 1, 2, 6, 8, 12, 13
BLOCK_BYTES = {Q4_0: (32, 18), Q5_0: (32, 22), Q8_0: (32, 34), Q4_K: (256, 144), Q5_K: (256, 176)}


def load_ref():
    if not os.path.exists(REF_PATH):
        import pytest
        pytest.skip("oracle/_ref/libwhisper_ref.so not built (run __graft_entry__.build() where /root/reference exists)")
    L = C.CDLL(REF_PATH)
    L.wref_quantize.restype = C.c_int64
    L.wref_quantize.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]
    L.wref_row_size.restype = C.c_int64
    L.wref_row_size.argtypes = [C.c_int, C.c_int64]
    L.wref_dequantize.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
    return L


def load_lib():
    L = C.CDLL(LIB_PATH)
    L.wb200_last_error.restype = C.c_char_p
    return L


def ref_quantize(ref, wtype, w):
    """w: float32 [rows][k] -> bytes in the ggml file layout (ggml_quantize_chunk, ggml-quants.c)"""
    w = np.ascontiguousarray(w, dtype=np.float32)
    rows, k = w.shape
    if wtype == F16:
        return w.astype(np.float16).tobytes()
    nbytes = ref.wref_row_size(wtype, k) * rows
    out = np.empty(nbytes, dtype=np.uint8)
    got = ref.wref_quantize(wtype, w.ctypes.data, out.ctypes.data, rows, k)
    assert got == nbytes
    return out.tobytes()


def ref_dequantize(ref, wtype, raw, rows, k):
    if wtype == F16:
        return np.frombuffer(raw, dtype=np.float16).astype(np.float32).reshape(rows, k)
    out = np.empty(rows * k, dtype=np.float32)
    buf = np.frombuffer(raw, dtype=np.uint8)
    ref.wref_dequantize(wtype, buf.ctypes.data, out.ctypes.data, rows * k)
    return out.reshape(rows, k)


def gelu_ref_f16(x):
    """GELU with the reference CPU semantics (f16 table): ggml/src/ggml-cpu/vec.h:988-1001"""
    x = np.asarray(x, dtype=np.float32)
    xh = x.astype(np.float16).astype(np.float32)
    g = 0.5 * xh * (1.0 + np.tanh(np.float32(0.79788456080286535587989211986876) * xh * (1.0 + np.float32(0.044715) * xh * xh)))
    g = g.astype(np.float16).astype(np.float32)
    return np.where(x <= -10, 0.0, np.where(x >= 10, x, g)).astype(np.float32)


import importlib.util as _ilu
_spec = _ilu.spec_from_file_location("wb200_api", os.path.join(ROOT, "whisper.cpp_b200", "api.py"))
_api = _ilu.module_from_spec(_spec); _spec.loader.exec_module(_api)
Aheads, ContextParams, TokenData, VadParams, Greedy, BeamSearch, FullParams, bind_whisper_api = (
    _api.Aheads, _api.ContextParams, _api.TokenData, _api.VadParams, _api.Greedy, _api.BeamSearch, _api.FullParams, _api.bind_whisper_api)


def read_wav_f32(path):
    import wave
    with wave.open(path, "rb") as w:
        assert w.getframerate() == 16000 and w.getsampwidth() == 2
        data = np.frombuffer(w.readframes(w.getnframes()), dtype=np.int16)
        if w.getnchannels() == 2:
            data = data.reshape(-1, 2).mean(axis=1)
    return (data.astype(np.float32) / 32768.0).astype(np.float32)


DATA_DIR = os.path.join(ROOT, "oracle", "_ref", "data")
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def data_file(name):
    """path of a fixture of the reference's own tests: the copy kept in the repository (tests/golden/<name>.xz, unpacked into the
    temp directory; a file already there is reused only if its bytes are the unpacked ones) when there is one, otherwise
    oracle/_ref/data/<name> as build() copied it"""
    packed = os.path.join(GOLDEN_DIR, name + ".xz")
    if not os.path.exists(packed):
        return os.path.join(DATA_DIR, name)
    import lzma
    import tempfile
    with open(packed, "rb") as f:
        data = lzma.decompress(f.read())
    out_dir = os.path.join(tempfile.gettempdir(), "wb200-fixtures-%d" % os.getuid())
    out = os.path.join(out_dir, name)
    if os.path.exists(out):
        with open(out, "rb") as f:
            if f.read() == data:
                return out
    os.makedirs(out_dir, exist_ok=True)
    tmp = "%s.tmp.%d" % (out, os.getpid())
    with open(tmp, "wb") as g:
        g.write(data)
    os.replace(tmp, out)
    return out


def parse_model_header(path):
    """hparams + mel filters of a legacy ggml model file (src/whisper.cpp:1496-1586)"""
    import struct
    with open(path, "rb") as f:
        magic, = struct.unpack("<I", f.read(4))
        assert magic == 0x67676d6c
        hp = struct.unpack("<11i", f.read(44))
        n_mel, n_fft = struct.unpack("<2i", f.read(8))
        filt = np.frombuffer(f.read(n_mel * n_fft * 4), dtype=np.float32).reshape(n_mel, n_fft).copy()
    return hp, filt
