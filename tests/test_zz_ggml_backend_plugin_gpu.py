"""GPU: the ggml backend PLUGIN (whisper.cpp_b200/libggml-b200.so, plugin/ggml_b200_backend.cpp; SURVEY.md section 8(f) rank 2).

The reference's own whisper-cli AND the reference's own libwhisper (oracle/_ref/whisper-cli-ref: unmodified sources, compiled from the
reference tree) load the plugin through GGML_BACKEND_PATH (ggml_backend_load_all, reference ggml/src/ggml-backend-reg.cpp:562-591).
All host logic is then the reference's; conv / encoder / cross / decoder graphs run on this engine.  The transcript must be the one the
same program produces on its CPU backend (-ng):
  * conditioned model (synth.conditioned: peaked logits, see tests/test_exact_tokens_gpu.py): token ids and segment times identical;
  * plain random weights: identical up to the first near-tie, and a common prefix of at least 8 tokens.
Also checked: the plugin really computed (graphs per kind counted through its log), and a run with -ng never touches it."""
import json
import os
import re
import subprocess
import pytest

from wbtest import ROOT, DATA_DIR, data_file, F16, Q5_0
from e2e_util import synth

pytestmark = pytest.mark.gpu
CLI = os.path.join(ROOT, "oracle", "_ref", "whisper-cli-ref")
PLUGIN = os.path.join(ROOT, "whisper.cpp_b200", "libggml-b200.so")
STUB = data_file("for-tests-ggml-tiny.en.bin")


CLI_DIRECT = os.path.join(ROOT, "oracle", "_ref", "whisper-cli-b200")     # the same CLI sources linked against libwhisper_b200.so (whisper.h boundary)


def _run(model, tmp_path, tag, plugin, extra=(), cli=CLI):
    out = str(tmp_path / ("cli_" + tag))
    env = dict(os.environ)
    env.pop("GGML_BACKEND_PATH", None)
    cmd = [cli, "-m", model, "-f", os.path.join(DATA_DIR, "jfk.wav"), "-bs", "1", "-bo", "1", "-nf", "-np", "-ojf", "-of", out, "-t", "4"] + list(extra)
    if plugin:
        env["GGML_BACKEND_PATH"] = PLUGIN
        env["WB200_PLUGIN_VERBOSE"] = "1"
    elif cli == CLI:
        cmd.append("-ng")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, (r.returncode, r.stderr[-1500:])
    doc = json.loads(open(out + ".json", encoding="utf-8", errors="replace").read(), strict=False)
    segs = [((c["offsets"]["from"], c["offsets"]["to"]), [t["id"] for t in c["tokens"]], [t["p"] for t in c["tokens"]]) for c in doc["transcription"]]
    return segs, r.stderr


@pytest.mark.parametrize("wt,seed,conditioned", [(F16, 3, True), (Q5_0, 0, True), (F16, 7, False), (Q5_0, 7, False)])
def test_reference_cli_on_the_plugin_matches_its_cpu_run(tmp_path, wt, seed, conditioned):
    if not (os.path.exists(CLI) and os.path.exists(PLUGIN)):
        pytest.skip("oracle/_ref/whisper-cli-ref or libggml-b200.so not built (make -C oracle; make -C whisper.cpp_b200 where the reference tree is present)")
    model = str(tmp_path / "m.bin")
    if conditioned:
        synth.write_model(model, "test-3l.en", wt, seed=seed, vocab_from=STUB, scale=lambda n: synth.conditioned(n, 1e-3 if wt == F16 else 0.0, 100.0))
    else:
        synth.write_model(model, "test-2l.en", wt, seed=seed, vocab_from=STUB)
    cpu, err_cpu = _run(model, tmp_path, "cpu", False)
    gpu, err_gpu = _run(model, tmp_path, "b200", True)
    assert "ggml-b200" not in err_cpu
    assert "loaded B200 backend" in err_gpu and "engine context ready" in err_gpu and "engine state 1" in err_gpu, err_gpu[-1500:]
    tc = [t for s in cpu for t in s[1]]; tg = [t for s in gpu for t in s[1]]
    common = 0
    while common < min(len(tc), len(tg)) and tc[common] == tg[common]:
        common += 1
    print("plugin run: %d tokens, CPU run: %d tokens, common prefix %d, %d / %d segments" % (len(tg), len(tc), common, len(gpu), len(cpu)))
    assert len(tg) > 8
    if conditioned and wt != F16:
        assert common >= 50, (common, len(tc), len(tg))                                     # int8 activation roundings: identical until the reference's own first near-tie (tests/test_exact_tokens_gpu.py)
    elif conditioned:
        assert tg == tc, (common, len(tc), len(tg))
        assert [s[0] for s in gpu] == [s[0] for s in cpu]                                   # segment times
        pc = [p for s in cpu for p in s[2]]; pg = [p for s in gpu for p in s[2]]
        assert max(abs(a - b) for a, b in zip(pc, pg)) < 5e-2
    else:
        assert common >= 8, (common, tc[:12], tg[:12])
    if os.path.exists(CLI_DIRECT):
        # the same kernels behind the OTHER boundary (whisper.h): host logic of this repository instead of the reference's, mel from the device
        # kernels instead of the reference's CPU code (<= 2e-3 apart) -- the transcripts agree up to the first near-tie
        direct, _ = _run(model, tmp_path, "direct", False, cli=CLI_DIRECT)
        td = [t for s in direct for t in s[1]]
        cd = 0
        while cd < min(len(td), len(tg)) and td[cd] == tg[cd]:
            cd += 1
        print("engine through whisper.h: %d tokens, common prefix with the plugin run %d" % (len(td), cd))
        assert cd >= 8
        if conditioned and wt == F16:
            assert td == tg


def test_two_host_states_get_two_engine_states(tmp_path):
    """whisper-cli -p 2 = whisper_full_parallel of the reference: two host states, each with its own kv_cross / kv_self tensors, decode
    concurrently; the plugin keeps one engine state per host state (keyed by the kv_cross tensor) and the result is the one of the same
    split on the CPU backend."""
    if not (os.path.exists(CLI) and os.path.exists(PLUGIN)):
        pytest.skip("oracle/_ref/whisper-cli-ref or libggml-b200.so not built")
    model = str(tmp_path / "m.bin")
    synth.write_model(model, "test-3l.en", F16, seed=3, vocab_from=STUB, scale=lambda n: synth.conditioned(n, 1e-3, 100.0))
    cpu, _ = _run(model, tmp_path, "cpu2", False, extra=("-p", "2"))
    gpu, err = _run(model, tmp_path, "b2002", True, extra=("-p", "2"))
    assert "engine state 2" in err, err[-1500:]
    tc = [t for s in cpu for t in s[1]]; tg = [t for s in gpu for t in s[1]]
    print("-p 2: plugin %d tokens in %d segments, CPU %d tokens in %d segments" % (len(tg), len(gpu), len(tc), len(cpu)))
    assert tg == tc and [s[0] for s in gpu] == [s[0] for s in cpu]
