"""tiny driver for compute-sanitizer runs: one encode + one decode step of the synthetic 2-layer model"""
import os, sys, tempfile
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from wbtest import data_file, Q5_0, load_lib
from e2e_util import Side, synth

wt = int(os.environ.get("WT", Q5_0))
path = os.path.join(tempfile.gettempdir(), "mk-smoke-%d.bin" % wt)
synth.write_model(path, "test-2l.en", wt, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
A = Side(load_lib(), path, False)
A.pcm_to_mel(synth.synth_audio(seed=1, seconds=2.0))
A.encode(0)
print("encode ok", flush=True)
sot = A.L.whisper_token_sot(A.ctx)
lg = A.decode([sot], 0)
print("decode ok", float(lg.std()), flush=True)
lg = A.decode([int(lg.argmax())], 1)
print("decode 2 ok", float(lg.std()), flush=True)
A.free()
