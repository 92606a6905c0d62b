"""CPU: the complete whisper_full control flow of libwhisper_b200.so against the reference, with the model taken out of the equation.

Both libraries run whisper_full / whisper_full_parallel with the SAME logits_filter_callback, which overwrites every logit with a value
scripted from the decoder's token history (the callback runs before the timestamp rules, src/whisper.cpp:6246-6249, so all later
filtering, sampling and bookkeeping still happens inside the libraries).  The reference runs its real CPU graphs on a synthetic 1-layer
model; the product runs on an engine-less test context (wb200_dbg_scripted_context) whose decodes return zeros.  Everything downstream of
the logits -- seek loop, prompt / context carry-over, temperature fallback with std::mt19937 draws, beam search, timestamp pairing,
segment emission, max_tokens / single_segment, token-level timestamps + max_len wrapping, grammar, callbacks, whisper_full_parallel --
must then agree EXACTLY: same segments, times, text, and per token id / tid / p / plog / pt / ptsum / t0 / t1 / vlen."""
import ctypes as C
import os
import zlib
import numpy as np
import pytest

from wbtest import DATA_DIR, data_file, F16, TokenData, bind_whisper_api
from e2e_util import synth
from test_grammar_cpu import build as build_grammar, lit, ALT, REF, CHAR, RNG
from test_vad_cpu import SILERO
from wbtest import read_wav_f32

vp = C.c_void_p
LOGITS_CB = C.CFUNCTYPE(None, vp, vp, C.POINTER(TokenData), C.c_int, C.POINTER(C.c_float), vp)
SEG_CB = C.CFUNCTYPE(None, vp, vp, C.c_int, vp)
PROG_CB = C.CFUNCTYPE(None, vp, vp, C.c_int, vp)
ENC_CB = C.CFUNCTYPE(C.c_bool, vp, vp, vp)
LOG_CB = C.CFUNCTYPE(None, C.c_int, C.c_char_p, vp)
_quiet = LOG_CB(lambda level, text, ud: None)


class Script:
    """deterministic logits from (token history, number of segments emitted so far, scenario seed)"""

    def __init__(self, L, ctx, seed, style, timestamps=True, use_segments=True):
        self.L, self.seed, self.style, self.timestamps, self.use_segments = L, seed, style, timestamps, use_segments
        self.V = L.whisper_n_vocab(ctx)
        self.beg, self.eot = L.whisper_token_beg(ctx), L.whisper_token_eot(ctx)
        self._calls = []                                  # list.append is atomic: callbacks can arrive from several member threads
        self.batches = []                                  # crc of (tokens, positions, sequence ids, logits flags) fed to the decoder before each filtered step
        self.tap = getattr(L, "wref_last_batch", None) or getattr(L, "wb200_dbg_last_batch", None)
        self.tap_att = getattr(L, "wref_last_attended", None) or getattr(L, "wb200_dbg_last_attended", None)
        if self.tap_att is not None:
            self.tap_att.argtypes = [vp, vp, C.c_int]
            self._ta = np.empty(2048, np.uint64)
        if self.tap is not None:
            self.tap.argtypes = [vp, vp, vp, vp, vp, C.c_int]
            self._tb = [np.empty(2048, np.int32) for _ in range(3)] + [np.empty(2048, np.int8)]
        L.whisper_full_n_segments_from_state.argtypes = [vp]
        self.cb = LOGITS_CB(self._cb)

    @property
    def calls(self):
        return len(self._calls)

    def _cb(self, ctx, st, toks, n, logits, ud):
        self._calls.append(None)
        ids = np.fromiter((toks[i].id for i in range(n)), np.int32, n)
        if self.tap is not None:
            tb = [np.empty(512, np.int32) for _ in range(3)] + [np.empty(512, np.int8)]
            nb = self.tap(st, tb[0].ctypes.data, tb[1].ctypes.data, tb[2].ctypes.data, tb[3].ctypes.data, 512)
            ta = np.empty(512, np.uint64)
            na = self.tap_att(st, ta.ctypes.data, 512) if self.tap_att is not None else 0
            self.batches.append((nb, zlib.crc32(b"".join(a[:max(nb, 0)].tobytes() for a in tb)), na, zlib.crc32(ta[:max(na, 0)].tobytes()) if na > 0 else 0))
        nseg = self.L.whisper_full_n_segments_from_state(st) if self.use_segments else 0
        rng = np.random.default_rng((zlib.crc32(ids.tobytes()) ^ self.seed ^ (nseg * 7919)) & 0xFFFFFFFF)
        V, beg, eot = self.V, self.beg, self.eot
        x = rng.standard_normal(V).astype(np.float32)
        x[beg:] -= 10.0                                                        # timestamps only when the script calls for one
        ts = ids[ids >= beg]
        last_ts = int(ts[-1] - beg) if len(ts) else 0
        since = n - (int(np.nonzero(ids >= beg)[0][-1]) + 1) if len(ts) else n
        peak = {"peaked": 14.0, "medium": 10.5, "flat": 8.5}[self.style]
        x[int(rng.integers(300, 20000))] += peak                               # the word this history "wants"
        if self.style != "peaked":
            x[rng.integers(300, 20000, 6)] += peak * 0.6
        if self.timestamps:
            if n == 0:
                x[beg + int(rng.integers(0, 12))] += 30.0                      # open the window with a timestamp near 0
            elif since >= int(rng.integers(4, 14)) or (len(ts) % 2 == 1 and since == 0):
                step = int(rng.integers(8, 90))
                x[min(beg + last_ts + step, V - 1)] += 28.0                    # close / reopen a segment a little later
        if (self.timestamps and last_ts > int(rng.integers(1250, 1480))) or n > int(rng.integers(110, 190)):
            x[eot] += 25.0
        np.ctypeslib.as_array(logits, (V,))[:] = x


def make_en_model(tmp_path):
    en = str(tmp_path / "s1.en.bin")
    synth.write_model(en, (51864, 1500, 384, 6, 1, 448, 384, 6, 1, 80), F16, seed=21, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    return en


def make_models(tmp_path):
    en = make_en_model(tmp_path); ml = str(tmp_path / "s1.multi.bin")
    synth.write_model(ml, (51865, 1500, 384, 6, 1, 448, 384, 6, 1, 80), F16, seed=22, vocab_from=os.path.join(DATA_DIR, "for-tests-ggml-tiny.bin"))
    return en, ml


def collect(L, ctx):
    L.whisper_full_get_segment_speaker_turn_next.restype = C.c_bool
    L.whisper_full_get_segment_speaker_turn_next.argtypes = [vp, C.c_int]
    for fn in ("whisper_full_get_token_t0", "whisper_full_get_token_t1"):
        getattr(L, fn).restype = C.c_int64; getattr(L, fn).argtypes = [vp, C.c_int, C.c_int]
    out = []
    for i in range(L.whisper_full_n_segments(ctx)):
        toks = []
        for j in range(L.whisper_full_n_tokens(ctx, i)):
            t = L.whisper_full_get_token_data(ctx, i, j)
            toks.append((t.id, t.tid, t.p, t.plog, t.pt, t.ptsum, t.t0, t.t1, t.t_dtw, t.vlen,
                         L.whisper_full_get_token_t0(ctx, i, j), L.whisper_full_get_token_t1(ctx, i, j)))      # mapped back through the VAD cut, if any
        out.append((L.whisper_full_get_segment_t0(ctx, i), L.whisper_full_get_segment_t1(ctx, i), L.whisper_full_get_segment_text(ctx, i),
                    bool(L.whisper_full_get_segment_speaker_turn_next(ctx, i)), toks))
    return out


SCENARIOS = [
    # name, model, seconds, style, params, extras
    ("greedy_default",      "en", 65.0, "peaked", dict(), {}),
    ("greedy_fallback",     "en", 40.0, "flat",   dict(best_of=2, logprob_thold=-2.0, temperature_inc=0.4), {}),
    ("greedy_medium_bo3",   "en", 31.0, "medium", dict(best_of=3, temperature=0.4, temperature_inc=0.3, logprob_thold=-3.5), {}),
    ("beam3",               "en", 42.0, "medium", dict(strategy=1, beam_size=3), {}),
    ("beam5_fallback",      "en", 25.0, "flat",   dict(strategy=1, beam_size=5, best_of=3, temperature_inc=0.5, logprob_thold=-2.5), {}),
    ("no_timestamps_maxtok", "en", 50.0, "peaked", dict(no_timestamps=True, max_tokens=12), {"timestamps": False}),
    ("single_segment_prompt", "en", 58.0, "peaked", dict(single_segment=True, initial_prompt=b" Hello world, previous context.", carry_initial_prompt=True), {}),
    ("prompt_tokens_ctx",   "en", 66.0, "medium", dict(n_max_text_ctx=64, prompt=[1000, 2000, 3000, 4000, 5000]), {}),
    ("token_ts_wrap",       "en", 35.0, "peaked", dict(token_timestamps=True, max_len=20, split_on_word=True), {}),
    ("token_ts_plain",      "en", 20.0, "medium", dict(token_timestamps=True, thold_pt=0.0005, thold_ptsum=0.0005), {}),
    ("multi_translate",     "ml", 33.0, "peaked", dict(language=b"de", translate=True, suppress_nst=True, suppress_blank=False), {}),
    ("offset_duration_actx", "en", 70.0, "peaked", dict(offset_ms=12000, duration_ms=37000, audio_ctx=768, max_initial_ts=0.5), {}),
    ("no_context_special",  "en", 45.0, "medium", dict(no_context=True, print_special=True, tdrz_enable=True, length_penalty=0.2, strategy=1, beam_size=2), {}),
    ("grammar",             "en", 28.0, "medium", dict(grammar=True, grammar_penalty=30.0, no_timestamps=True, max_tokens=24), {"timestamps": False}),
    ("parallel2",           "en", 64.0, "peaked", dict(n_processors=2), {"use_segments": False}),
    ("short_input",         "en", 0.05, "peaked", dict(), {}),
    ("encoder_begin_stop",  "en", 95.0, "peaked", dict(stop_at_window=3), {}),
    ("err_too_many_decoders", "en", 5.0, "peaked", dict(best_of=9, temperature=0.4), {}),            # -4
    ("err_audio_ctx",       "en", 5.0, "peaked", dict(audio_ctx=1600), {}),                        # -5
    ("suppress_regex_nst",  "en", 26.0, "medium", dict(suppress_regex=b"^ ?[a-mA-M]", suppress_nst=True, best_of=2, temperature_inc=0.5), {}),
    ("max_initial_ts_tdrz", "en", 12.0, "medium", dict(max_initial_ts=0.04, tdrz_enable=True, entropy_thold=3.5, n_max_text_ctx=0), {}),
    # params.vad on jfk.wav with the Silero weights of the reference's tests (product side: host walk of the VAD kernels' phases)
    ("vad_token_ts",        "en", "jfk", "peaked", dict(vad=True, token_timestamps=True, max_len=30), {}),
    ("vad_beam",            "en", "jfk", "medium", dict(vad=True, strategy=1, beam_size=2, samples_overlap=0.3), {}),
    ("vad_parallel2",       "en", "jfk", "peaked", dict(vad=True, n_processors=2), {"use_segments": False}),
    # two consecutive calls on the same context with no_context = false: the text context of the first carries into the second
    ("context_carry_1",     "en", 31.0, "peaked", dict(no_context=False), {}),
    ("context_carry_2",     "en", 47.0, "medium", dict(no_context=False, n_max_text_ctx=96, best_of=2, temperature_inc=0.5), {}),
]


def run_side(L, ctx, name, seconds, style, kw, extras, pcm, seed):
    kw = dict(kw)
    fp = L.whisper_full_default_params(kw.pop("strategy", 0))
    fp.print_progress = False; fp.n_threads = 1; fp.no_speech_thold = 2.0          # the model's own no-speech probability plays no role
    keep = []
    if "best_of" in kw:
        fp.greedy.best_of = kw.pop("best_of")
    if "beam_size" in kw:
        fp.beam_search.beam_size = kw.pop("beam_size")
    if "prompt" in kw:
        arr = (C.c_int32 * len(kw["prompt"]))(*kw.pop("prompt")); keep.append(arr)
        fp.prompt_tokens = arr; fp.prompt_n_tokens = len(arr)
    if kw.pop("grammar", False):
        # root ::= " " word rest ; rest ::= " " word rest | "." ; word ::= [a-z] tail ; tail ::= [a-z] tail | ()
        rules = [[(CHAR, 32), (REF, 2), (REF, 1)], [(CHAR, 32), (REF, 2), (REF, 1), (ALT, 0), (CHAR, ord("."))],
                 [(CHAR, ord("a")), (RNG, ord("z")), (REF, 3)], [(CHAR, ord("a")), (RNG, ord("z")), (REF, 3), (ALT, 0)]]
        ptrs, arrs = build_grammar(rules); keep += [ptrs, arrs]
        fp.grammar_rules = C.cast(ptrs, vp); fp.n_grammar_rules = len(rules); fp.i_start_rule = 0
    n_proc = kw.pop("n_processors", 1)
    stop_at = kw.pop("stop_at_window", 0)
    windows = [0]
    if stop_at:                                        # encoder_begin_callback returning false ends the run with what was transcribed so far
        def _begin(c, st, ud):
            windows[0] += 1
            return windows[0] < stop_at
        begin_cb = ENC_CB(_begin); keep.append(begin_cb)
        fp.encoder_begin_callback = C.cast(begin_cb, vp)
    if kw.pop("vad", False):
        fp.vad = True; fp.vad_model_path = SILERO.encode()
        fp.vad_params.samples_overlap = kw.pop("samples_overlap", 0.1)
    for k, v in kw.items():
        assert hasattr(fp, k), k
        setattr(fp, k, v)
    script = Script(L, ctx, seed, style, **extras)
    fp.logits_filter_callback = C.cast(script.cb, vp)
    events = []
    seg_cb = SEG_CB(lambda c, s, n_new, ud: events.append(("seg", n_new)))
    prog_cb = PROG_CB(lambda c, s, p, ud: events.append(("prog", p)))
    fp.new_segment_callback = C.cast(seg_cb, vp); fp.progress_callback = C.cast(prog_cb, vp)
    if n_proc > 1:
        rc = L.whisper_full_parallel(ctx, fp, pcm.ctypes.data_as(vp), len(pcm), n_proc)
    else:
        rc = L.whisper_full(ctx, fp, pcm.ctypes.data_as(vp), len(pcm))
    for fn in ("whisper_full_get_vad_segment_t0", "whisper_full_get_vad_segment_t1"):
        getattr(L, fn).restype = C.c_int64; getattr(L, fn).argtypes = [vp, C.c_int]
    L.whisper_full_n_vad_segments.argtypes = [vp]
    vad_segs = [(L.whisper_full_get_vad_segment_t0(ctx, i), L.whisper_full_get_vad_segment_t1(ctx, i)) for i in range(L.whisper_full_n_vad_segments(ctx))] if fp.vad else []
    # the run counters whisper_print_timings reports (fallbacks, sample / encode / decode / batchd / prompt runs)
    lines = []
    grab = LOG_CB(lambda level, text, ud: lines.append(text.decode("utf-8", "replace")))
    L.whisper_log_set(grab, None)
    L.whisper_print_timings(ctx); L.whisper_reset_timings(ctx)
    L.whisper_log_set(_quiet, None)
    import re
    txt = "".join(lines)
    counters = tuple(int(v) for v in re.findall(r"fallbacks =\s*(\d+) p /\s*(\d+) h", txt)[0]) + tuple(int(v) for v in re.findall(r"/\s*(\d+) runs", txt))
    assert len(counters) == 7, txt
    return rc, collect(L, ctx), events, script.calls, (L.whisper_full_lang_id(ctx), vad_segs, counters if n_proc == 1 else None), script.batches


def test_whisper_full_control_flow_identical_under_scripted_logits(lib, ref, tmp_path):
    if not hasattr(lib, "wb200_dbg_scripted_context"):
        pytest.skip("library predates wb200_dbg_scripted_context")
    L = bind_whisper_api(lib); R = bind_whisper_api(ref)
    for X in (L, R):
        X.whisper_log_set.argtypes = [LOG_CB, vp]
        if not os.environ.get("WB200_VERBOSE"):
            X.whisper_log_set(_quiet, None)
    L.wb200_dbg_scripted_context.restype = vp; L.wb200_dbg_scripted_context.argtypes = [C.c_char_p]
    paths = dict(zip(("en", "ml"), make_models(tmp_path)))
    ctxs = {}
    for key, path in paths.items():
        cp = R.whisper_context_default_params(); cp.use_gpu = False
        rctx = R.whisper_init_from_file_with_params(path.encode(), cp)
        lctx = L.wb200_dbg_scripted_context(path.encode())
        assert rctx and lctx
        ctxs[key] = (lctx, rctx)
    rng = np.random.default_rng(99)
    stats = []
    only = os.environ.get("WB200_SCENARIO")
    for idx, (name, model, seconds, style, kw, extras) in enumerate(SCENARIOS):
        if only and only != name:
            continue
        if seconds == "jfk":
            if not os.path.exists(SILERO):
                continue
            pcm = np.ascontiguousarray(read_wav_f32(os.path.join(DATA_DIR, "jfk.wav")), np.float32)
        else:
            pcm = (rng.standard_normal(int(seconds * 16000)) * 0.01).astype(np.float32)
        lctx, rctx = ctxs[model]
        a = run_side(L, lctx, name, seconds, style, kw, extras, pcm, 1000 + idx)
        b = run_side(R, rctx, name, seconds, style, kw, extras, pcm, 1000 + idx)
        n_tok = sum(len(s[4]) for s in b[1])
        stats.append((name, b[0], len(b[1]), n_tok, b[3]))
        assert a[0] == b[0], (name, "return code", a[0], b[0])
        assert len(a[1]) == len(b[1]), (name, "segments", len(a[1]), len(b[1]), [s[2] for s in a[1]][:3], [s[2] for s in b[1]][:3])
        for i, (sa, sb) in enumerate(zip(a[1], b[1])):
            assert sa[:4] == sb[:4], (name, i, sa[:4], sb[:4])
            assert len(sa[4]) == len(sb[4]), (name, i, "tokens")
            for j, (ta, tb) in enumerate(zip(sa[4], sb[4])):
                assert ta == tb, (name, i, j, ta, tb)
        assert a[4] == b[4], (name, "lang id / VAD segments", a[4], b[4])
        if kw.get("vad"):
            assert len(a[4][1]) == 4                                                    # the reference's KAT for jfk.wav (tests/test-vad.cpp)
        if kw.get("n_processors", 1) == 1:
            assert a[2] == b[2], (name, "callback events", a[2][:8], b[2][:8])
            assert a[3] == b[3], (name, "logits callback calls", a[3], b[3])
            assert len(a[5]) == len(b[5]) > 0 or a[3] == 0
            assert a[3] == 0 or (all(x[0] > 0 and x[2] == x[0] for x in a[5]) and all(y[0] > 0 and y[2] == y[0] for y in b[5]))   # both taps delivered
            for k, (x, y) in enumerate(zip(a[5], b[5])):                                # what the decoder was fed: prompt assembly, positions, beam sequence ids
                assert x == y, (name, "decoder input of filtered step", k, x, y)
    for s in stats:
        print("scripted %-22s rc=%d segments=%3d tokens=%4d logits-callback calls=%d" % s)
    if not only:
        assert sum(s[2] for s in stats) > 40 and sum(s[3] for s in stats) > 600       # the scripts did produce transcripts
        by = {s[0]: s for s in stats}
        assert by["greedy_fallback"][4] > 2 * by["greedy_fallback"][3]                 # fallback really re-decoded windows
        assert by["short_input"][2] == 0
    for lctx, rctx in ctxs.values():
        L.whisper_free(lctx); R.whisper_free(rctx)


def test_lockstep_batch_driver_equals_reference_chunk_by_chunk(lib, ref, tmp_path, monkeypatch):
    """wb200_full_batch on the engine-less context: 3 member threads rendezvous for every encode / decode while they work through 8 chunks
    of very different lengths (one too short to decode, one of three windows) with temperature fallback; every chunk must come out exactly
    as the reference's whisper_full_with_state gives it on a fresh state."""
    if not hasattr(lib, "wb200_dbg_scripted_context"):
        pytest.skip("library predates wb200_dbg_scripted_context")
    monkeypatch.setenv("WB200_BATCH_MEMBERS", "3")
    L = bind_whisper_api(lib); R = bind_whisper_api(ref)
    for X in (L, R):
        X.whisper_log_set.argtypes = [LOG_CB, vp]
        X.whisper_log_set(_quiet, None)
    L.wb200_dbg_scripted_context.restype = vp; L.wb200_dbg_scripted_context.argtypes = [C.c_char_p]
    en, _ = make_models(tmp_path)
    cp = R.whisper_context_default_params(); cp.use_gpu = False
    rctx = R.whisper_init_from_file_with_params(en.encode(), cp)
    lctx = L.wb200_dbg_scripted_context(en.encode())
    assert rctx and lctx
    rng = np.random.default_rng(7)
    lengths = [31.0, 0.04, 12.5, 64.0, 29.9, 3.0, 30.0, 8.2]
    chunks = [(rng.standard_normal(int(s * 16000)) * 0.01).astype(np.float32) for s in lengths]

    def params(X, ctx):
        fp = X.whisper_full_default_params(0)
        fp.print_progress = False; fp.n_threads = 1; fp.no_speech_thold = 2.0
        fp.greedy.best_of = 2; fp.logprob_thold = -1.2; fp.temperature_inc = 0.4
        script = Script(X, ctx, 4242, "medium", use_segments=True)
        fp.logits_filter_callback = C.cast(script.cb, vp)
        return fp, script

    # product: all chunks through the lock-step driver
    fp, script = params(L, lctx)
    n = len(chunks)
    ptrs = (C.POINTER(C.c_float) * n)(*[c.ctypes.data_as(C.POINTER(C.c_float)) for c in chunks])
    lens = (C.c_int * n)(*[len(c) for c in chunks])
    states = (vp * n)()
    L.wb200_full_batch.argtypes = [vp, type(fp), vp, vp, C.c_int, vp]
    assert L.wb200_full_batch(lctx, fp, ptrs, lens, n, states) == 0
    for fn in ("whisper_full_n_segments_from_state",):
        getattr(L, fn).argtypes = [vp]; getattr(R, fn).argtypes = [vp]
    for X in (L, R):
        X.whisper_full_n_tokens_from_state.argtypes = [vp, C.c_int]
        X.whisper_full_get_token_data_from_state.restype = TokenData
        X.whisper_full_get_token_data_from_state.argtypes = [vp, C.c_int, C.c_int]

    def collect_state(X, st):
        out = []
        for i in range(X.whisper_full_n_segments_from_state(st)):
            toks = []
            for j in range(X.whisper_full_n_tokens_from_state(st, i)):
                t = X.whisper_full_get_token_data_from_state(st, i, j)
                toks.append((t.id, t.tid, t.p, t.plog, t.pt, t.ptsum, t.t0, t.t1, t.vlen))
            out.append((X.whisper_full_get_segment_t0_from_state(st, i), X.whisper_full_get_segment_t1_from_state(st, i),
                        X.whisper_full_get_segment_text_from_state(st, i), toks))
        return out

    got = [collect_state(L, states[i]) for i in range(n)]
    # reference: one fresh state per chunk
    rfp, rscript = params(R, rctx)
    n_tok = 0
    for i, c in enumerate(chunks):
        st = R.whisper_init_state(rctx)
        assert R.whisper_full_with_state(rctx, st, rfp, c.ctypes.data_as(vp), len(c)) == 0
        want = collect_state(R, st)
        R.whisper_free_state(st)
        assert got[i] == want, (i, lengths[i], len(got[i]), len(want))
        n_tok += sum(len(s[3]) for s in want)
    assert script.calls == rscript.calls                      # the same number of decoder evaluations, fallback re-decodes included
    assert n_tok > 300 and got[1] == []
    print("lock-step batch: %d chunks, %d tokens, %d logits-callback calls" % (n, n_tok, script.calls))
    for i in range(n):
        L.whisper_free_state(states[i])
    L.whisper_free(lctx); R.whisper_free(rctx)
