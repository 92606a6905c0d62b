"""CPU: grammar-constrained decoding (whisper_full_params.grammar_rules; the whisper_grammar_* pushdown automaton of
src/whisper.cpp:5480-5923) of libwhisper_b200.so against the reference: after accepting any prefix of tokens, the set of penalised
token ids (hence the filtered logits, log-probs, probs and the greedy pick) and the number of live parses must be identical."""
import ctypes as C
import os
import numpy as np
import pytest

from wbtest import data_file, FullParams, TokenData, bind_whisper_api

vp = C.c_void_p
END, ALT, REF, CHAR, NOT, RNG, CALT = range(7)


class Elem(C.Structure):
    _fields_ = [("type", C.c_int), ("value", C.c_uint32)]


def build(rules):
    """rules: list of element lists [(type, value), ...] WITHOUT the final END -> (array of pointers, keep-alive list)"""
    arrs = []
    for r in rules:
        a = (Elem * (len(r) + 1))(*[Elem(t, v) for t, v in r], Elem(END, 0))
        arrs.append(a)
    ptrs = (C.POINTER(Elem) * len(arrs))(*[C.cast(a, C.POINTER(Elem)) for a in arrs])
    return ptrs, arrs


def lit(s):
    return [(CHAR, ord(c)) for c in s]


GRAMMARS = {
    # root ::= " yes" | " no" | " maybe so"
    "choice": ([lit(" yes") + [(ALT, 0)] + lit(" no") + [(ALT, 0)] + lit(" maybe so")], [" yes", " maybe so", " no"]),
    # root ::= " " word rest ; rest ::= " " word rest | "." ; word ::= [a-z] wtail ; wtail ::= [a-z] wtail | (empty)
    "words": ([[(CHAR, 32), (REF, 2), (REF, 1)],
               [(CHAR, 32), (REF, 2), (REF, 1), (ALT, 0), (CHAR, ord("."))],
               [(CHAR, ord("a")), (RNG, ord("z")), (REF, 3)],
               [(CHAR, ord("a")), (RNG, ord("z")), (REF, 3), (ALT, 0)]], [" ask not what your country can do.", " hello world."]),
    # root ::= item item* "!" ; item ::= [^0-9,.!]   (negated class with alternatives), then unicode literals
    "negated": ([[(REF, 1), (REF, 2)],
                 [(NOT, ord("0")), (RNG, ord("9")), (CALT, ord(",")), (CALT, ord(".")), (CALT, ord("!"))],
                 [(REF, 1), (REF, 2), (ALT, 0), (CHAR, ord("!"))]], [" naïve café 東京!", " what a day!"]),
    # root ::= " 東京" | " café" | " 東洋"  (multi-byte code points: tokens may end inside a UTF-8 sequence)
    "unicode": ([lit(" 東京") + [(ALT, 0)] + lit(" café") + [(ALT, 0)] + lit(" 東洋")], [" 東京", " café", " 東洋"]),
}


@pytest.mark.parametrize("stub", ["for-tests-ggml-tiny.en.bin", "for-tests-ggml-tiny.bin"])
@pytest.mark.parametrize("gname", sorted(GRAMMARS))
def test_grammar_filter_matches_reference(lib, ref, stub, gname):
    if not hasattr(ref, "wref_process_logits_grammar"):
        pytest.skip("oracle/_ref predates wref_process_logits_grammar (rebuild with make -C oracle)")
    L = bind_whisper_api(lib); R = bind_whisper_api(ref)
    path = data_file(stub).encode()
    cp = R.whisper_context_default_params(); cp.use_gpu = False
    rctx = R.whisper_init_from_file_with_params(path, cp)
    assert rctx
    R.wref_ctx_state.restype = vp; R.wref_ctx_state.argtypes = [vp]
    sig = [C.POINTER(FullParams), C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.c_float, C.POINTER(C.c_int), C.c_int, vp, vp, vp, vp,
           C.POINTER(TokenData), C.POINTER(C.c_int)]
    R.wref_process_logits_grammar.argtypes = [vp, vp] + sig
    L.wb200_dbg_process_logits_grammar.argtypes = [C.c_char_p] + sig
    R.whisper_tokenize.argtypes = [vp, C.c_char_p, vp, C.c_int]
    n_vocab = R.whisper_n_vocab(rctx)
    rules, texts = GRAMMARS[gname]
    ptrs, keep = build(rules)
    rng = np.random.default_rng(len(gname))
    n_rejected_seen = 0
    for text in texts:
        buf = (C.c_int * 128)()
        nt = R.whisper_tokenize(rctx, text.encode("utf-8"), buf, 128)
        assert nt > 0
        toks = list(buf[:nt])
        for n_acc in range(nt + 1):                         # the grammar state after every prefix of the tokenised text
            fp = R.whisper_full_default_params(0)
            fp.grammar_rules = C.cast(ptrs, vp); fp.n_grammar_rules = len(rules); fp.i_start_rule = 0
            fp.grammar_penalty = 100.0 if n_acc % 2 == 0 else 7.5
            logits = (rng.standard_normal(n_vocab) * 2.0).astype(np.float32)
            logits[:50256] += 3.0                           # keep the text tokens ahead of the timestamp mass: the grammar branch runs
            hist = (C.c_int * max(1, n_acc))(*toks[:n_acc])
            acc = (C.c_int * max(1, n_acc))(*toks[:n_acc])
            res = []
            for which in (0, 1):
                lo = np.empty(n_vocab, np.float32); lp = np.empty(n_vocab, np.float32); pr = np.empty(n_vocab, np.float32)
                td = TokenData(); ns = C.c_int(-1)
                args = (C.byref(fp), hist, n_acc, 0, 0, C.c_float(0.0), acc, n_acc, logits.ctypes.data_as(vp), lo.ctypes.data_as(vp),
                        lp.ctypes.data_as(vp), pr.ctypes.data_as(vp), C.byref(td), C.byref(ns))
                rc = L.wb200_dbg_process_logits_grammar(path, *args) if which == 0 else R.wref_process_logits_grammar(rctx, R.wref_ctx_state(rctx), *args)
                assert rc == 0
                res.append((lo, lp, pr, td.id, td.p, ns.value))
            a, b = res
            assert a[5] == b[5], (text, n_acc, a[5], b[5])                      # live parses
            assert np.array_equal(a[0], b[0]), (text, n_acc)                    # penalised ids and amounts
            assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
            assert a[3] == b[3] and a[4] == b[4]
            n_rejected_seen += int((np.isfinite(b[0]) & (b[0] < logits - 1.0)).sum())
    assert n_rejected_seen > 0                                                  # the grammar did bite
    R.whisper_free(rctx)
