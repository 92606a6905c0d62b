"""GPU: whisper_full with token_timestamps + max_len through the C ABI.  The algorithm is pinned bit for bit on CPU by
tests/test_token_timestamps_cpu.py; here the INTEGRATION is checked: the segments a real run produced (token ids, tid / pt / ptsum from the
on-device sampler, segment times, the clip's signal energy, the t_beg / t_last / tid_last state carried from segment to segment) are
replayed through the reference's whisper_exp_compute_token_level_timestamps and must give the same t0 / t1 / vlen for every token.
(No absolute range is asserted: with random weights all timestamp probabilities can underflow to 0, tid stays 0 and the reference
itself then yields segment times of seek - 2*token_beg.)"""
import ctypes as C
import os
import numpy as np
import pytest

from wbtest import DATA_DIR, data_file, read_wav_f32, Q5_0, TokenData
from e2e_util import Side, synth
from test_full_scripted_cpu import Script

pytestmark = pytest.mark.gpu
vp = C.c_void_p


@pytest.mark.parametrize("scripted", [False, True])
def test_token_timestamps_and_max_len(lib, ref, tmp_path, scripted):
    """scripted = False: 2-layer model (the reference's distil rule forces no_timestamps), tokens picked by the on-device sampler;
    scripted = True: 3-text-layer model with the transcript scripted through logits_filter_callback (timestamps, several segments, host sampler)"""
    path = str(tmp_path / "m.bin")
    cfg = (51864, 1500, 384, 6, 1, 448, 384, 6, 3, 80) if scripted else "test-2l.en"
    synth.write_model(path, cfg, Q5_0, seed=11, vocab_from=data_file("for-tests-ggml-tiny.en.bin"))
    pcm = read_wav_f32(os.path.join(DATA_DIR, "jfk.wav"))
    A = Side(lib, path, False)
    try:
        L = A.L
        L.whisper_full_get_token_data.restype = TokenData
        L.whisper_full_get_token_data.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.whisper_full_get_segment_text.restype = C.c_char_p
        eot = L.whisper_token_eot(A.ctx)

        keep = []

        def run(max_len):
            fp = L.whisper_full_default_params(0)
            fp.print_progress = False; fp.temperature_inc = 0.0; fp.greedy.best_of = 1
            fp.token_timestamps = True; fp.max_len = max_len; fp.split_on_word = False
            if scripted:
                script = Script(L, A.ctx, 31, "peaked", use_segments=False); keep.append(script)    # history-only script: the wrapped run must see the same logits
                fp.logits_filter_callback = C.cast(script.cb, vp); fp.no_speech_thold = 2.0
            assert L.whisper_full(A.ctx, fp, pcm.ctypes.data_as(C.c_void_p), len(pcm)) == 0, L.wb200_last_error()
            segs = []
            for i in range(L.whisper_full_n_segments(A.ctx)):
                toks = [L.whisper_full_get_token_data(A.ctx, i, j) for j in range(L.whisper_full_n_tokens(A.ctx, i))]
                segs.append((L.whisper_full_get_segment_t0(A.ctx, i), L.whisper_full_get_segment_t1(A.ctx, i),
                             L.whisper_full_get_segment_text(A.ctx, i).decode("utf-8", "replace"), [(t.id, t.t0, t.t1, t.vlen, t.tid, t.pt, t.ptsum) for t in toks]))
            return segs

        plain = run(0)
        assert len(plain) >= 1 and sum(len(s[3]) for s in plain) > 0
        if scripted:
            assert len(plain) >= 3 and sum(len(s[3]) for s in plain) > 30
        # replay through the reference
        B = Side(ref, path, True)
        try:
            R = B.L
            SIG = [vp, vp, vp, vp, C.c_int, C.c_int64, C.c_int64, vp, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int]
            R.wref_token_timestamps.argtypes = [vp, vp] + SIG
            R.wref_signal_energy.argtypes = [vp, C.c_int, C.c_int, vp]
            energy = np.empty_like(pcm)
            assert R.wref_signal_energy(pcm.ctypes.data, len(pcm), 32, energy.ctypes.data) == 0
            carry = np.zeros(3, np.int64)
            fpd = L.whisper_full_default_params(0)
            for s0, s1, text, toks in plain:
                n = len(toks)
                ids = np.array([t[0] for t in toks], np.int32); tids = np.array([t[4] for t in toks], np.int32)
                pt = np.array([t[5] for t in toks], np.float32); ptsum = np.array([t[6] for t in toks], np.float32)
                tok = np.full((n, 2), -7, np.int64); vlen = np.zeros(n, np.float32); pieces = np.full((8, 3), -7, np.int64)
                k = R.wref_token_timestamps(B.ctx, B.state, ids.ctypes.data, tids.ctypes.data, pt.ctypes.data, ptsum.ctypes.data, n, s0, s1,
                                            energy.ctypes.data, len(energy), C.c_float(fpd.thold_pt), C.c_float(fpd.thold_ptsum), 0, 0,
                                            carry.ctypes.data, tok.ctypes.data, vlen.ctypes.data, pieces.ctypes.data, 8)
                assert k == 1
                assert [t[1] for t in toks] == tok[:, 0].tolist() and [t[2] for t in toks] == tok[:, 1].tolist(), (s0, s1, toks[:4], tok[:4])
                assert np.array_equal(np.array([t[3] for t in toks], np.float32), vlen)
        finally:
            B.free()
        wrapped = run(24)
        assert len(wrapped) >= len(plain)
        if any(len(text) > 60 and sum(1 for t in toks if t[0] < eot) >= 6 for _, _, text, toks in plain):
            assert len(wrapped) > len(plain)                     # long segments were cut
        assert [t[0] for s in wrapped for t in s[3]] == [t[0] for s in plain for t in s[3]]   # wrapping keeps the token sequence
    finally:
        A.free()
