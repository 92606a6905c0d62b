"""CPU: plumbing of the ggml backend plugin (whisper.cpp_b200/libggml-b200.so) without a GPU.  With WB200_PLUGIN_DRY=1 the plugin registers its
device, hands out buffers, finds the host's model file and parses whisper.cpp's four graphs (conv / encoder / cross / decoder), but
computes nothing (logits = 0): the reference's unmodified whisper-cli + libwhisper must load it through GGML_BACKEND_PATH, route every
graph to it and run to completion.  The arithmetic is tested on the GPU (tests/test_zz_ggml_backend_plugin_gpu.py)."""
import ctypes as C
import os
import subprocess
import pytest

from wbtest import ROOT, DATA_DIR, data_file, F16
from e2e_util import synth

CLI = os.path.join(ROOT, "oracle", "_ref", "whisper-cli-ref")
PLUGIN = os.path.join(ROOT, "whisper.cpp_b200", "libggml-b200.so")


def test_plugin_exports_the_ggml_entry_point():
    if not os.path.exists(PLUGIN):
        pytest.skip("libggml-b200.so not built (needs the reference tree: make -C whisper.cpp_b200)")
    out = subprocess.run(["nm", "-D", "--defined-only", PLUGIN], capture_output=True, text=True).stdout
    names = {l.split()[-1] for l in out.splitlines() if l.strip()}
    assert {"ggml_backend_init", "ggml_backend_score"} <= names
    assert not any(n.startswith("whisper_") for n in names)            # nothing that could shadow the host's own libwhisper


def test_reference_cli_routes_all_four_graphs_to_the_plugin(tmp_path):
    if not (os.path.exists(CLI) and os.path.exists(PLUGIN)):
        pytest.skip("oracle/_ref/whisper-cli-ref or libggml-b200.so not built")
    model = str(tmp_path / "m.bin")
    synth.write_model(model, "test-2l.en", F16, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    env = dict(os.environ, GGML_BACKEND_PATH=PLUGIN, WB200_PLUGIN_DRY="1", WB200_PLUGIN_VERBOSE="1")
    r = subprocess.run([CLI, "-m", model, "-f", os.path.join(DATA_DIR, "jfk.wav"), "-bs", "1", "-bo", "1", "-nf", "-np", "-t", "2"],
                       capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-1500:]
    assert "loaded B200 backend" in r.stderr
    assert "model file of the host: " + model in r.stderr               # found among the host's open descriptors during the weight upload
    assert "none of whisper.cpp's four" not in r.stderr
    assert "-->" in r.stdout                                            # a segment was printed: the decode loop ran on the plugin's (zero) logits


def test_reference_bench_program_routes_its_graphs_to_the_plugin(tmp_path):
    """examples/bench/bench.cpp of the reference (whisper_set_mel(NULL), whisper_encode, 256-token prompts, single-token steps, batches of 5
    through whisper_decode): other decoder-graph shapes than whisper_full's; dry run, the run counts of whisper_print_timings must be complete"""
    import re
    exe = os.path.join(ROOT, "oracle", "_ref", "whisper-bench-ref")
    if not (os.path.exists(exe) and os.path.exists(PLUGIN)):
        pytest.skip("oracle/_ref/whisper-bench-ref or libggml-b200.so not built")
    model = str(tmp_path / "m.bin")
    synth.write_model(model, "test-2l.en", F16, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    env = dict(os.environ, GGML_BACKEND_PATH=PLUGIN, WB200_PLUGIN_DRY="1", WB200_PLUGIN_VERBOSE="1")
    r = subprocess.run([exe, "-m", model, "-t", "2"], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-1500:]
    out = r.stderr + r.stdout
    assert "loaded B200 backend" in out and "none of whisper.cpp's four" not in out
    runs = {k: int(v) for k, v in re.findall(r"(\w+) time =\s*[\d.]+ ms /\s*(\d+) runs", out)}
    assert {k: runs.get(k) for k in ("encode", "decode", "batchd", "prompt")} == {"encode": 1, "decode": 256, "batchd": 320, "prompt": 4096}, runs
