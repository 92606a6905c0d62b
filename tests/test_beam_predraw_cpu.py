"""CPU: beam search with the uniforms of the categorical draws taken from each decoder's mt19937 BEFORE the decode is submitted (what lets
the draws run on the device, csrc/wb_full.cpp) must consume the generators exactly like the reference's order "decode, then draw" does.

On an engine-less test context (wb200_dbg_scripted_context: decodes leave zero logits, so after the logits filter the distribution is
uniform over the allowed tokens and every draw depends on the generator state) whisper_full is run twice, with the pre-drawn path
(the decode ignores the device request, the host sampler uses the pre-drawn uniforms: sample_token_topk_u) and with WB200_HOST_BEAM=1
(draws made at sampling time: sample_token_topk, pinned to the reference bit for bit in test_sampler_cpu).  Both must give the same
segments and tokens -- through window changes, completed / failed decoders and temperature fallback attempts (where the pre-drawn path is
off and the generators simply continue)."""
import ctypes as C
import os
import numpy as np
import pytest

from wbtest import data_file, F16, TokenData, bind_whisper_api
from e2e_util import synth

vp = C.c_void_p


def _collect(L, ctx):
    L.whisper_full_get_segment_t0.restype = C.c_int64; L.whisper_full_get_segment_t1.restype = C.c_int64
    L.whisper_full_get_token_data.restype = TokenData; L.whisper_full_get_token_data.argtypes = [vp, C.c_int, C.c_int]
    out = []
    for i in range(L.whisper_full_n_segments(ctx)):
        toks = [L.whisper_full_get_token_data(ctx, i, j) for j in range(L.whisper_full_n_tokens(ctx, i))]
        out.append((L.whisper_full_get_segment_t0(ctx, i), L.whisper_full_get_segment_t1(ctx, i), [(t.id, t.tid, t.p, t.plog, t.pt, t.ptsum) for t in toks]))
    return out


@pytest.mark.parametrize("beam,temp_inc,seconds", [(5, 0.0, 40.0), (3, 0.2, 65.0), (8, 0.0, 12.0)])
def test_predrawn_uniforms_consume_the_generators_like_the_reference_order(lib, tmp_path, beam, temp_inc, seconds):
    if not hasattr(lib, "wb200_dbg_scripted_context"):
        pytest.skip("library predates wb200_dbg_scripted_context")
    L = bind_whisper_api(lib)
    L.wb200_dbg_scripted_context.restype = vp; L.wb200_dbg_scripted_context.argtypes = [C.c_char_p]
    path = str(tmp_path / "m.bin")
    synth.write_model(path, (51864, 1500, 384, 6, 1, 448, 384, 6, 3, 80), F16, seed=5, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    pcm = (np.random.default_rng(3).standard_normal(int(seconds * 16000)) * 0.01).astype(np.float32)
    results = []
    for host_beam in (False, True):
        if host_beam:
            os.environ["WB200_HOST_BEAM"] = "1"
        else:
            os.environ.pop("WB200_HOST_BEAM", None)
        try:
            ctx = L.wb200_dbg_scripted_context(path.encode())
            assert ctx
            fp = L.whisper_full_default_params(1)
            fp.print_progress = False; fp.n_threads = 2
            fp.beam_search.beam_size = beam; fp.greedy.best_of = 2
            fp.temperature_inc = temp_inc
            fp.no_timestamps = True                  # (with timestamps on, the uniform distribution puts all mass on timestamp tokens and a window ends after two)
            fp.max_tokens = 24                       # uniform draws hardly ever produce EOT on their own: bound the windows
            fp.entropy_thold = 8.0 if temp_inc > 0 else fp.entropy_thold      # with fallback: every window fails the entropy check at T = 0 and is retried at T > 0
            assert L.whisper_full(ctx, fp, pcm.ctypes.data_as(vp), len(pcm)) == 0
            results.append(_collect(L, ctx))
            L.whisper_free(ctx)
        finally:
            os.environ.pop("WB200_HOST_BEAM", None)
    a, b = results
    n_tok = sum(len(s[2]) for s in b)
    print("beam %d, temperature_inc %.1f: %d segments, %d tokens" % (beam, temp_inc, len(b), n_tok))
    assert n_tok > 20 and len({t[0] for s in b for t in s[2]}) > 10          # random draws: many distinct tokens
    assert len(a) == len(b)
    for sa, sb in zip(a, b):
        assert sa[:2] == sb[:2]
        assert sa[2] == sb[2]
