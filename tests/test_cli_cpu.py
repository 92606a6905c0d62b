"""CPU: validates the CLI-vs-API harness (tests/cli_util.py) on the reference pair -- the reference's whisper-cli linked against the reference
library must write exactly what the reference's C ABI returns for the mirrored parameters -- so that the GPU test of the same harness on
libwhisper_b200.so (tests/test_zz_reference_cli_gpu.py) checks the engine, not the harness."""
import os
import pytest

from wbtest import ROOT, data_file, F16
from e2e_util import synth
from cli_util import check_cli_against_api, SILERO

CLI_REF = os.path.join(ROOT, "oracle", "_ref", "whisper-cli-ref")


@pytest.mark.parametrize("vad", [False, True])
def test_reference_cli_equals_reference_api(ref, tmp_path, vad):
    if not os.path.exists(CLI_REF):
        pytest.skip("oracle/_ref/whisper-cli-ref not built (make -C oracle cli)")
    if vad and not os.path.exists(SILERO):
        pytest.skip("silero fixture missing")
    path = str(tmp_path / "m.bin")
    synth.write_model(path, "test-2l.en", F16, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    got = check_cli_against_api(CLI_REF, ref, True, path, tmp_path, vad)
    assert sum(len(c["tokens"]) for c in got) > 50


def test_reference_bench_harness_on_reference(tmp_path):
    """the parser / expectations used for whisper-bench on the engine (GPU test), validated here on the reference's own build"""
    from cli_util import run_reference_bench
    exe = os.path.join(ROOT, "oracle", "_ref", "whisper-bench-ref")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/whisper-bench-ref not built (make -C oracle cli)")
    path = str(tmp_path / "m.bin")
    synth.write_model(path, (51864, 1500, 384, 6, 1, 448, 384, 6, 1, 80), F16, seed=3, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    t = run_reference_bench(exe, path)
    print("reference whisper-bench on a 1-layer synthetic model:", {k: round(v[2], 2) for k, v in t.items()})


def test_reference_vad_example_prints_the_golden_segments():
    from cli_util import run_reference_vad_example
    import numpy as np
    exe = os.path.join(ROOT, "oracle", "_ref", "vad-segments-ref")
    if not os.path.exists(exe) or not os.path.exists(SILERO):
        pytest.skip("oracle/_ref/vad-segments-ref or the silero fixture missing")
    g = np.load(os.path.join(ROOT, "tests", "golden", "vad_r01.npz"))
    assert run_reference_vad_example(exe) == list(zip(g["seg_t0"].astype(float).tolist(), g["seg_t1"].astype(float).tolist()))


def test_reference_server_harness_on_reference(ref, tmp_path):
    """examples/server/server.cpp on the reference library answers /inference with what the reference's C ABI gives for the mirrored
    parameters: validates tests/cli_util.check_server_against_api before it is pointed at libwhisper_b200.so on the GPU"""
    from cli_util import check_server_against_api
    exe = os.path.join(ROOT, "oracle", "_ref", "whisper-server-ref")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/whisper-server-ref not built (make -C oracle cli)")
    pytest.importorskip("requests")
    path = str(tmp_path / "m.bin")
    synth.write_model(path, "test-2l.en", F16, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    out = check_server_against_api(exe, ref, True, path)
    assert len(out["verbose_json"]["segments"]) >= 2                  # the 60-character wrap produced several segments
