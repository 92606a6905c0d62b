"""Golden data of __graft_entry__.smoke(): the reference's logits for the smoke model and audio, so that smoke() needs no reference build.

The reference CPU library (oracle/_ref) runs the same three decode steps smoke() runs: SOT, then twice its own argmax token.  Stored:
the three fed tokens, the standard deviation of each step's full logit vector, and the logits at a fixed, seeded sample of the
vocabulary (the full vectors would be 600 KB).

Run where the reference tree exists (after `make -C oracle`):   python tests/golden/make_smoke_golden.py
"""
import ctypes as C
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from __graft_entry__ import SMOKE_SAMPLE, load_pkg, smoke_inputs  # noqa: E402


def main():
    pkg = load_pkg()
    model, pcm = smoke_inputs(tempfile.mkdtemp())
    R = pkg.bind_whisper_api(C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libwhisper_ref.so")))
    cp = R.whisper_context_default_params(); cp.use_gpu = False
    ctx = R.whisper_init_from_file_with_params(model.encode(), cp)
    assert ctx
    assert R.whisper_pcm_to_mel(ctx, pcm.ctypes.data_as(C.c_void_p), len(pcm), 4) == 0
    assert R.whisper_encode(ctx, 0, 4) == 0
    n_vocab = R.whisper_n_vocab(ctx)
    idx = np.sort(np.random.default_rng(0).choice(n_vocab, SMOKE_SAMPLE, replace=False))
    tokens, std, sampled = [R.whisper_token_sot(ctx)], [], []
    for i in range(3):
        t = np.array([tokens[-1]], np.int32)
        assert R.whisper_decode(ctx, t.ctypes.data_as(C.c_void_p), 1, i, 4) == 0
        logits = np.ctypeslib.as_array(R.whisper_get_logits(ctx), shape=(n_vocab,)).copy()
        std.append(logits.std()); sampled.append(logits[idx])
        if i < 2:
            tokens.append(int(logits.argmax()))
    R.whisper_free(ctx)
    out = os.path.join(ROOT, "tests", "golden", "smoke_ref.npz")
    np.savez_compressed(out, tokens=np.array(tokens, np.int32), index=idx.astype(np.int32), logits=np.array(sampled, np.float32),
                        std=np.array(std, np.float64), n_vocab=np.int32(n_vocab))
    print("wrote", out, "tokens", tokens)


if __name__ == "__main__":
    main()
