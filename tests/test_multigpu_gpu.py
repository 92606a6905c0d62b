"""GPU (needs >= 2 GPUs, skipped otherwise): in-library multi-GPU.  With WB200_DEVICES=all a context keeps a replica of the weights on
every GPU, whisper_init_state places states on the least-loaded GPU, and whisper_full_parallel / concurrent whisper_full_with_state
callers spread over the box -- with results identical to the single-GPU run (chunks are independent; no data crosses GPUs)."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np
import pytest

from wbtest import data_file, Q5_0
from e2e_util import Side, synth

pytestmark = pytest.mark.gpu
vp = C.c_void_p


def _n_gpus():
    try:
        return len(subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout.strip().splitlines())
    except Exception:  # noqa: BLE001
        return 0


@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs (run under gpurun --gpus 2)")
def test_states_spread_over_gpus_and_results_match_single_gpu(lib, tmp_path):
    path = str(tmp_path / "m.bin")
    synth.write_model(path, "test-2l.en", Q5_0, seed=5, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    chunks = [synth.synth_audio(seed=70 + i, seconds=s) for i, s in enumerate((30.0, 12.0, 25.0, 7.0, 30.0, 18.0))]

    def run(multi):
        if multi:
            os.environ["WB200_DEVICES"] = "all"
        else:
            os.environ.pop("WB200_DEVICES", None)
        A = Side(lib, path, False); L = A.L
        L.wb200_n_devices.argtypes = [vp]; L.wb200_state_device.argtypes = [vp]
        try:
            fp = L.whisper_full_default_params(0); fp.print_progress = False; fp.temperature_inc = 0.0; fp.greedy.best_of = 1
            states = [L.whisper_init_state(A.ctx) for _ in chunks]
            assert all(states), L.wb200_last_error()
            devs = [L.wb200_state_device(s) for s in states]
            rcs = [None] * len(chunks)

            def work(i):
                rcs[i] = L.whisper_full_with_state(A.ctx, states[i], fp, chunks[i].ctypes.data_as(vp), len(chunks[i]))
            th = [threading.Thread(target=work, args=(i,)) for i in range(len(chunks))]
            for t in th: t.start()
            for t in th: t.join()
            assert rcs == [0] * len(chunks), (rcs, L.wb200_last_error())
            toks = [[[L.whisper_full_get_token_id_from_state(st, s, j) for j in range(L.whisper_full_n_tokens_from_state(st, s))]
                     for s in range(L.whisper_full_n_segments_from_state(st))] for st in states]
            # whisper_full_parallel on one long buffer: its states are spread the same way
            buf = np.ascontiguousarray(np.concatenate([chunks[0], chunks[4]]))
            assert L.whisper_full_parallel(A.ctx, fp, buf.ctypes.data_as(vp), len(buf), 2) == 0
            par = [[L.whisper_full_get_token_id(A.ctx, s, j) for j in range(L.whisper_full_n_tokens(A.ctx, s))] for s in range(L.whisper_full_n_segments(A.ctx))]
            nd = L.wb200_n_devices(A.ctx)
            for st in states: L.whisper_free_state(st)
            return nd, devs, toks, par
        finally:
            A.free(); os.environ.pop("WB200_DEVICES", None)
    nd1, devs1, toks1, par1 = run(False)
    nd2, devs2, toks2, par2 = run(True)
    assert nd1 == 1 and set(devs1) == {0}
    assert nd2 >= 2 and len(set(devs2)) >= 2, (nd2, devs2)
    assert toks2 == toks1 and par2 == par1
    assert sum(len(t) for c in toks1 for t in c) > 50
