"""diagnostic: determinism of whisper_full / whisper_full_parallel with the persistent decode kernel"""
import ctypes as C, os, sys, tempfile
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from wbtest import data_file, Q5_0, load_lib
from e2e_util import Side, synth

path = os.path.join(tempfile.gettempdir(), "mk-par.bin")
synth.write_model(path, "test-2l.en", Q5_0, seed=3, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
pcm = synth.synth_audio(seed=9, seconds=60.0)
A = Side(load_lib(), path, False); L = A.L
fp = L.whisper_full_default_params(0); fp.print_progress = False; fp.temperature_inc = 0.0; fp.greedy.best_of = 1

def toks():
    return [[L.whisper_full_get_token_id(A.ctx, i, j) for j in range(L.whisper_full_n_tokens(A.ctx, i))] for i in range(L.whisper_full_n_segments(A.ctx))]

def run_par():
    assert L.whisper_full_parallel(A.ctx, fp, pcm.ctypes.data_as(C.c_void_p), len(pcm), 2) == 0, L.wb200_last_error()
    return toks()

def run_seq():
    half = len(pcm) // 2; out = []
    for sl in (pcm[:half], pcm[half:]):
        sl = np.ascontiguousarray(sl)
        assert L.whisper_full(A.ctx, fp, sl.ctypes.data_as(C.c_void_p), len(sl)) == 0
        out += toks()
    return out

def first_diff(a, b):
    fa = [t for s in a for t in s]; fb = [t for s in b for t in s]
    for i, (x, y) in enumerate(zip(fa, fb)):
        if x != y: return i, len(fa), len(fb)
    return (None if len(fa) == len(fb) else min(len(fa), len(fb))), len(fa), len(fb)

s1 = run_seq(); s2 = run_seq(); p1 = run_par(); p2 = run_par(); s3 = run_seq()
print("seq1 vs seq2", first_diff(s1, s2)); print("par1 vs par2", first_diff(p1, p2)); print("seq1 vs par1", first_diff(s1, p1)); print("seq1 vs seq3", first_diff(s1, s3))
print("segments", len(s1), len(p1))
A.free()
