"""GPU: the reference's UNMODIFIED whisper-cli (examples/cli/cli.cpp, compiled from the reference tree into oracle/_ref/whisper-cli-b200 and
linked against libwhisper_b200.so) transcribes on this engine, and what it writes (-ojf: full JSON with token ids and probabilities) is what the
same parameters give through the C ABI directly.  With --vad it goes through params.vad with the Silero weights of the reference's tests.
The harness itself is validated on the CPU with the reference pair (tests/test_cli_cpu.py).
(Written after the GPU budget of round 1 was spent: not yet run on a GPU.)"""
import os
import pytest

from wbtest import ROOT, data_file, F16, Q5_0
from e2e_util import synth
from cli_util import check_cli_against_api, SILERO

pytestmark = pytest.mark.gpu
CLI = os.path.join(ROOT, "oracle", "_ref", "whisper-cli-b200")


@pytest.mark.parametrize("wt,vad", [(F16, False), (Q5_0, False), (F16, True)])
def test_reference_cli_runs_on_this_engine(lib, tmp_path, wt, vad):
    if not os.path.exists(CLI):
        pytest.skip("oracle/_ref/whisper-cli-b200 not built")
    if vad and not os.path.exists(SILERO):
        pytest.skip("silero fixture missing")
    path = str(tmp_path / "m.bin")
    synth.write_model(path, "test-2l.en", wt, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    check_cli_against_api(CLI, lib, False, path, tmp_path, vad)


def test_reference_bench_program_runs_on_this_engine(lib, tmp_path):
    """examples/bench/bench.cpp of the reference, unmodified, linked against libwhisper_b200.so: whisper_set_mel(NULL, 0), whisper_encode,
    256-token prompts, 256 single-token steps, 64 batches of 5 through whisper_decode, then whisper_print_timings with the expected run counts"""
    from cli_util import run_reference_bench
    exe = os.path.join(ROOT, "oracle", "_ref", "whisper-bench-b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/whisper-bench-b200 not built")
    path = str(tmp_path / "m.bin")
    synth.write_model(path, "test-2l.en", Q5_0, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    t = run_reference_bench(exe, path)
    print("whisper-bench on the engine (test-2l.en Q5_0):", {k: round(v[2], 3) for k, v in t.items()})


def test_reference_vad_example_runs_on_this_engine():
    """examples/vad-speech-segments/speech.cpp of the reference, unmodified, on libwhisper_b200.so: prints the reference's known answer"""
    import numpy as np
    from cli_util import run_reference_vad_example
    exe = os.path.join(ROOT, "oracle", "_ref", "vad-segments-b200")
    if not os.path.exists(exe) or not os.path.exists(SILERO):
        pytest.skip("oracle/_ref/vad-segments-b200 or the silero fixture missing")
    g = np.load(os.path.join(ROOT, "tests", "golden", "vad_r01.npz"))
    assert run_reference_vad_example(exe) == list(zip(g["seg_t0"].astype(float).tolist(), g["seg_t1"].astype(float).tolist()))


def test_reference_server_runs_on_this_engine(lib, tmp_path):
    """examples/server/server.cpp of the reference, unmodified, linked against libwhisper_b200.so: HTTP /inference (json and verbose_json)
    answers with what the C ABI returns directly"""
    from cli_util import check_server_against_api
    exe = os.path.join(ROOT, "oracle", "_ref", "whisper-server-b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/whisper-server-b200 not built")
    pytest.importorskip("requests")
    path = str(tmp_path / "m.bin")
    synth.write_model(path, "test-2l.en", Q5_0, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    check_server_against_api(exe, lib, False, path)
