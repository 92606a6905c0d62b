"""CPU: how far the reference is from ITSELF -- the noise floor every parity tolerance in this repository is stated against.

The unmodified reference CPU build gives different numbers for the same model and audio when only `n_threads` changes:
  * its flash attention accumulates P.V in F16 (ggml-cpu/ops.cpp:8585-8600) and, for a single query row over >= 512 keys (every decode
    step's cross-attention: 1536 keys), cuts the keys into one chunk PER THREAD (ops.cpp:9122-9157) -- the rounding of a 1536-term F16
    running sum depends on where the chunks end;
  * encoder output and cross K/V therefore move with the thread count as well, more so for quantised weights, whose activations are
    re-quantised to int8 blocks in front of every matrix (a rounding flip is a 1/127 step of the block maximum).
This test measures that self-distance (1 thread vs 4 threads) on the synthetic 2-layer model and asserts it is what DESIGN.md quotes:
logits 2e-2 .. 8e-2 of their standard deviation, i.e. as large as or larger than the distance between this engine and the 4-thread
reference (tests/test_e2e_gpu.py: 2e-3 F16, 1.4e-2 Q5_0 measured on B200).  "Identical to the reference" can therefore only mean
"within the reference's own reproducibility", except where the arithmetic is integer or thread-independent (tokenizer, filters,
samplers, KV bookkeeping, seek loop: pinned exactly elsewhere), or on a conditioned model (tests/test_exact_tokens_gpu.py).
"""
import ctypes as C
import os

import numpy as np
import pytest

from wbtest import data_file, F16, Q5_0
from e2e_util import Side, synth, taps, rms_err

vp = C.c_void_p


def _logits_and_taps(ref, path, nth, pcm, steps=6):
    B = Side(ref, path, True)
    L = B.L
    try:
        assert L.whisper_pcm_to_mel(B.ctx, pcm.ctypes.data_as(vp), len(pcm), nth) == 0
        assert L.whisper_encode(B.ctx, 0, nth) == 0
        t = taps(B)
        toks = [L.whisper_token_sot(B.ctx)]; out = []
        rng = np.random.default_rng(5)
        for s in range(steps):
            a = np.asarray(toks[-1:], np.int32)
            assert L.whisper_decode(B.ctx, a.ctypes.data_as(vp), 1, s, nth) == 0
            out.append(np.ctypeslib.as_array(L.whisper_get_logits(B.ctx), shape=(B.n_vocab,)).copy())
            toks.append(int(rng.integers(300, 20000)))
        return t, out
    finally:
        B.free()


@pytest.mark.parametrize("wt,enc_lo,log_lo", [(F16, 5e-5, 1e-2), (Q5_0, 1e-3, 1e-2)])
def test_reference_differs_from_itself_across_thread_counts(ref, tmp_path, wt, enc_lo, log_lo):
    path = str(tmp_path / "m.bin")
    synth.write_model(path, "test-2l.en", wt, seed=7, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    pcm = synth.synth_audio(seed=512, seconds=30.0)
    t1, l1 = _logits_and_taps(ref, path, 1, pcm)
    t4, l4 = _logits_and_taps(ref, path, 4, pcm)
    t4b, l4b = _logits_and_taps(ref, path, 4, pcm)
    e_enc = rms_err(t1["enc"], t4["enc"]); e_kv = rms_err(t1["kv"], t4["kv"])
    e_log = [float(np.sqrt(((a - b) ** 2).mean()) / b.std()) for a, b in zip(l1, l4)]
    print("reference vs itself (1 vs 4 threads), type %d: encoder output %.2e, cross V %.2e, logits %.2e .. %.2e of std" % (wt, e_enc, e_kv, min(e_log), max(e_log)))
    # same thread count: bit-reproducible
    assert all(np.array_equal(a, b) for a, b in zip(l4, l4b)) and np.array_equal(t4["enc"], t4b["enc"])
    # different thread count: a different answer, of the size DESIGN.md section 2 quotes
    assert e_enc > enc_lo and max(e_log) > log_lo, (e_enc, e_log)
    assert max(e_log) < 0.2                              # ... but still the same model
