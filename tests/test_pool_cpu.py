"""CPU: the rendezvous logic of the context pool (csrc/wb_state.h, Group) on the engine-less test context -- no GPU, no device work, the
transcript is scripted through logits_filter_callback exactly like tests/test_full_scripted_cpu.py.

What can go wrong here is host logic: a missed wake-up or a wrong active count is a deadlock, a mixed-up request is a wrong transcript.
Ten caller threads run whisper_full_with_state on their own states at staggered times while an eleventh thread keeps creating and freeing
states (pool growth / slot reuse), and one caller starts a nested whisper_full_with_state on another state from inside its
encoder_begin_callback (the outer state must be suspended, not waited for).  Every transcript must equal the one the same chunk gives
when it runs alone."""
import ctypes as C
import os
import threading
import time

import numpy as np
import pytest

from wbtest import F16, DATA_DIR
from e2e_util import synth
from test_full_scripted_cpu import Script, make_en_model, LOG_CB, _quiet

vp = C.c_void_p
ENC_CB = C.CFUNCTYPE(C.c_bool, vp, vp, vp)


def _tokens(L, st):
    return [[L.whisper_full_get_token_id_from_state(st, s, j) for j in range(L.whisper_full_n_tokens_from_state(st, s))]
            for s in range(L.whisper_full_n_segments_from_state(st))]


@pytest.mark.timeout(600)
def test_concurrent_callers_on_the_scripted_pool(lib, tmp_path):
    from wbtest import bind_whisper_api
    L = bind_whisper_api(lib)
    L.whisper_log_set.argtypes = [LOG_CB, vp]; L.whisper_log_set(_quiet, None)
    L.wb200_dbg_scripted_context.restype = vp; L.wb200_dbg_scripted_context.argtypes = [C.c_char_p]
    en = make_en_model(tmp_path)
    ctx = L.wb200_dbg_scripted_context(en.encode())
    assert ctx
    n = 10
    chunks = [synth.synth_audio(seed=900 + i, seconds=6.0 + 3.5 * (i % 4)) for i in range(n)]
    script = Script(L, ctx, 777, "peaked", use_segments=False)
    script.tap = None; script.tap_att = None
    fp = L.whisper_full_default_params(0); fp.print_progress = False; fp.greedy.best_of = 1; fp.temperature_inc = 0.0; fp.n_threads = 1
    fp.no_speech_thold = 2.0
    fp.logits_filter_callback = C.cast(script.cb, vp)

    # alone, one after the other
    alone = []
    st0 = L.whisper_init_state(ctx)
    for c in chunks:
        assert L.whisper_full_with_state(ctx, st0, fp, c.ctypes.data_as(vp), len(c)) == 0
        alone.append(_tokens(L, st0))
    assert sum(len(t) for a in alone for t in a) > 100

    states = [L.whisper_init_state(ctx) for _ in range(n)]
    assert all(states)
    rcs = [None] * n
    nested = {"done": 0}
    extra_state = L.whisper_init_state(ctx)

    def on_window(c, st, ud):                          # runs inside caller 3's whisper_full: a nested call on ANOTHER state of the same context
        if nested["done"] == 0:
            nested["done"] = 1
            short = chunks[0]
            assert L.whisper_full_with_state(ctx, extra_state, fp, short.ctypes.data_as(vp), len(short)) == 0
            nested["tokens"] = _tokens(L, extra_state)
        return True
    cb = ENC_CB(on_window)

    def work(i):
        time.sleep(0.002 * (i % 5))                    # staggered entry
        p = fp
        if i == 3:
            p = type(fp).from_buffer_copy(fp); p.encoder_begin_callback = C.cast(cb, vp)
        rcs[i] = L.whisper_full_with_state(ctx, states[i], p, chunks[i].ctypes.data_as(vp), len(chunks[i]))

    stop = threading.Event()

    def churn():                                       # pool growth and slot reuse while the others transcribe
        while not stop.is_set():
            tmp = [L.whisper_init_state(ctx) for _ in range(3)]
            time.sleep(0.001)
            for s in tmp: L.whisper_free_state(s)
    th = [threading.Thread(target=work, args=(i,)) for i in range(n)]
    ch = threading.Thread(target=churn)
    ch.start()
    for t in th: t.start()
    for t in th: t.join(timeout=300)
    stop.set(); ch.join(timeout=30)
    assert not any(t.is_alive() for t in th), "a caller is stuck in the rendezvous"
    assert rcs == [0] * n, rcs
    assert [_tokens(L, st) for st in states] == alone
    assert nested.get("tokens") == alone[0]
    for st in states + [extra_state, st0]: L.whisper_free_state(st)
    L.whisper_free(ctx)
