"""CPU tests of the drop-in boundary: libwhisper_b200.so loads without a GPU, exports every symbol include/whisper_b200.h
declares (and exactly the whisper_* set the reference library exports), its by-value structs have the reference's sizes,
pure-host entry points behave like the reference, and the product path fails LOUDLY when no CUDA device exists."""
import ctypes as C
import os
import re
import subprocess

import pytest

from wbtest import ROOT, LIB_PATH, REF_PATH, DATA_DIR, data_file, bind_whisper_api, ContextParams, FullParams, TokenData, load_lib


def _exported(path):
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    return {l.split()[-1] for l in out.splitlines() if " T " in l}


def test_header_symbols_all_exported():
    hdr = open(os.path.join(ROOT, "include", "whisper_b200.h")).read()
    declared = set(re.findall(r"WB_EXPORT[^;(]*?\b(whisper_\w+|wb200_\w+)\s*\(", hdr))
    assert len(declared) > 130
    missing = declared - _exported(LIB_PATH)
    assert not missing, missing


def test_same_whisper_symbols_as_reference():
    if not os.path.exists(REF_PATH):
        pytest.skip("reference library not built")
    mine = {s for s in _exported(LIB_PATH) if s.startswith("whisper_")}
    theirs = {s for s in _exported(REF_PATH) if s.startswith("whisper_")}
    assert mine == theirs


def test_nothing_else_is_exported():
    """linker version script (whisper.cpp_b200/exports.map): no libstdc++ template instantiations or CUDA runtime symbols leak out"""
    out = subprocess.run(["nm", "-D", "--defined-only", LIB_PATH], capture_output=True, text=True, check=True).stdout
    names = [l.split()[-1] for l in out.splitlines() if l.strip()]
    stray = [n for n in names if not (n.startswith("whisper_") or n.startswith("wb200_"))]
    assert not stray, stray[:10]


def test_struct_sizes_match_reference(ref):
    assert C.sizeof(FullParams) == ref.wref_sizeof_full_params() == 304
    assert C.sizeof(ContextParams) == ref.wref_sizeof_context_params() == 48
    assert C.sizeof(TokenData) == ref.wref_sizeof_token_data() == 56


def test_default_params_equal_reference(ref):
    L = bind_whisper_api(load_lib()); R = bind_whisper_api(ref)
    for strategy in (0, 1):
        a = L.whisper_full_default_params(strategy); b = R.whisper_full_default_params(strategy)
        for name, _ in FullParams._fields_:
            va, vb = getattr(a, name), getattr(b, name)
            if name == "n_threads":
                continue
            if name == "prompt_tokens":
                assert not va and not vb      # NULL pointers on both sides
                continue
            if name in ("greedy", "beam_search", "vad_params"):
                for sub, _ in type(va)._fields_:
                    assert getattr(va, sub) == getattr(vb, sub), (name, sub)
            else:
                assert va == vb, name
    a = L.whisper_context_default_params(); b = R.whisper_context_default_params()
    for name in ("use_gpu", "flash_attn", "gpu_device", "dtw_token_timestamps", "dtw_aheads_preset", "dtw_n_top", "dtw_mem_size"):
        assert getattr(a, name) == getattr(b, name), name


def test_language_table_equals_reference(ref):
    L = bind_whisper_api(load_lib()); R = bind_whisper_api(ref)
    assert L.whisper_lang_max_id() == R.whisper_lang_max_id() == 99
    for i in range(100):
        assert L.whisper_lang_str(i) == R.whisper_lang_str(i)
        assert L.whisper_lang_str_full(i) == R.whisper_lang_str_full(i)
        assert L.whisper_lang_id(R.whisper_lang_str(i)) == i
        assert L.whisper_lang_id(R.whisper_lang_str_full(i)) == i
    assert L.whisper_lang_id(b"klingon") == -1


def test_no_cpu_fallback_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L = bind_whisper_api(load_lib())
    cp = L.whisper_context_default_params()
    ctx = L.whisper_init_from_file_with_params(data_file("for-tests-ggml-tiny.en.bin").encode(), cp)
    assert not ctx
    assert b"no CUDA device" in L.wb200_last_error() or b"CPU fallback" in L.wb200_last_error()
    cp.use_gpu = False
    assert not L.whisper_init_from_file_with_params(data_file("for-tests-ggml-tiny.en.bin").encode(), cp)


C_PROGRAM = r"""
#include "whisper_b200.h"
#include <stdio.h>
#include <string.h>
/* a C99 client of the header, as tests/test-c.c of the reference is for whisper.h: structs by value, callbacks, enums */
static void on_segment(struct whisper_context * ctx, struct whisper_state * st, int n_new, void * ud) { (void) ctx; (void) st; (void) n_new; (void) ud; }
int main(void) {
    struct whisper_context_params cp = whisper_context_default_params();
    struct whisper_full_params fp = whisper_full_default_params(WHISPER_SAMPLING_BEAM_SEARCH);
    struct whisper_vad_params vp = whisper_vad_default_params();
    struct whisper_vad_context_params vcp = whisper_vad_default_context_params();
    fp.new_segment_callback = on_segment;
    printf("%zu %zu %zu %zu %zu\n", sizeof(cp), sizeof(fp), sizeof(whisper_token_data), sizeof(vp), sizeof(vcp));
    printf("%d %d %d %.2f %d %d\n", (int) cp.use_gpu, (int) cp.flash_attn, fp.beam_search.beam_size, (double) fp.entropy_thold, fp.greedy.best_of, vp.speech_pad_ms);
    printf("%s %d %s\n", whisper_lang_str(whisper_lang_id("de")), whisper_lang_max_id(), whisper_version());
    /* no GPU here: init must fail cleanly, not crash */
    cp.use_gpu = 0;
    printf("%d\n", whisper_init_from_file_with_params("/nonexistent.bin", cp) == NULL);
    return 0;
}
"""


def test_header_is_valid_c_and_links(tmp_path, ref):
    """the reference keeps tests/test-c.c to guarantee that whisper.h stays C; same for include/whisper_b200.h, plus a link + run"""
    src = tmp_path / "client.c"
    src.write_text(C_PROGRAM)
    exe = str(tmp_path / "client")
    inc = os.path.join(ROOT, "include")
    libdir = os.path.dirname(LIB_PATH)
    cmd = ["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", inc, str(src), "-o", exe, "-L", libdir, "-lwhisper_b200", "-Wl,-rpath," + libdir]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.strip().splitlines()
    assert lines[0].split()[:3] == ["48", "304", "56"], lines[0]            # the reference's struct sizes (test_struct_sizes_match_reference)
    rp = bind_whisper_api(ref).whisper_full_default_params(1)
    assert lines[1] == "1 1 %d %.2f %d 30" % (rp.beam_search.beam_size, rp.entropy_thold, rp.greedy.best_of), lines[1]
    assert lines[2].split()[0] == "de" and lines[2].split()[1] == "99"
    assert lines[3] == "1"


def test_unmodified_reference_cli_links_against_this_library(tmp_path):
    """oracle/_ref/whisper-cli-b200 = the reference's examples/cli/cli.cpp (+ common*.cpp, grammar-parser.cpp), compiled from the reference tree
    without a change and linked against libwhisper_b200.so: every whisper_* symbol it imports binds to this library, and on a box without
    a GPU it stops with the loud no-CPU-fallback error (exit code 3 of cli.cpp), not with a transcript."""
    exe = os.path.join(ROOT, "oracle", "_ref", "whisper-cli-b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/whisper-cli-b200 not built (make -C oracle cli)")
    env = dict(os.environ, LD_DEBUG="bindings")
    r = subprocess.run([exe, "--help"], capture_output=True, text=True, env=env, timeout=120)
    bound = re.findall(r"binding file \S*whisper-cli-b200 \[0\] to (\S+) \[0\]: normal symbol `(whisper_\w+)'", r.stderr + r.stdout)
    assert bound, "no whisper_* bindings seen"
    assert all(lib.endswith("libwhisper_b200.so") for lib, _ in bound), sorted({lib for lib, _ in bound})
    model = data_file("for-tests-ggml-tiny.en.bin"); wav = os.path.join(DATA_DIR, "jfk.wav")
    r = subprocess.run([exe, "-m", model, "-f", wav], capture_output=True, text=True, timeout=120)
    import ctypes
    try:
        ctypes.CDLL("libcuda.so.1"); has_driver = True
    except OSError:
        has_driver = False
    if not has_driver:
        assert r.returncode == 3 and "no CPU fallback" in (r.stderr + r.stdout), (r.returncode, r.stderr[-400:])


def test_vad_init_fails_loudly_without_cuda(tmp_path):
    """whisper_vad_init_* has no CPU path either"""
    import ctypes
    try:
        ctypes.CDLL("libcuda.so.1")
        pytest.skip("a CUDA driver is present")
    except OSError:
        pass
    lib = load_lib()
    silero = os.path.join(DATA_DIR, "for-tests-silero-v6.2.0-ggml.bin")
    if not os.path.exists(silero):
        pytest.skip("silero fixture missing")

    class VadCtxParams(C.Structure):
        _fields_ = [("n_threads", C.c_int), ("use_gpu", C.c_bool), ("gpu_device", C.c_int)]
    lib.whisper_vad_default_context_params.restype = VadCtxParams
    lib.whisper_vad_init_from_file_with_params.restype = C.c_void_p
    lib.whisper_vad_init_from_file_with_params.argtypes = [C.c_char_p, VadCtxParams]
    lib.wb200_last_error.restype = C.c_char_p
    assert not lib.whisper_vad_init_from_file_with_params(silero.encode(), lib.whisper_vad_default_context_params())
    assert b"no CPU fallback" in lib.wb200_last_error()
