"""Diagnostic (not a pytest): run the same calls on libwhisper_b200 (GPU) and the reference (CPU) and print how far
apart every stage is.  Usage: python tests/e2e_report.py [config] [wtype ...]"""
import os
import sys
import tempfile
import time
import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ["WB200_DEBUG_TAPS"] = "1"
from wbtest import load_lib, load_ref, DATA_DIR, data_file, read_wav_f32, F16, Q4_0, Q5_0, Q8_0, Q4_K, Q5_K, ref_quantize
from e2e_util import Side, synth, taps, rel_err, rms_err

NAMES = {F16: "f16", Q4_0: "q4_0", Q5_0: "q5_0", Q8_0: "q8_0", Q4_K: "q4_k", Q5_K: "q5_k"}


def main():
    cfg = sys.argv[1] if len(sys.argv) > 1 else "test-2l.en"
    wtypes = [int(a) for a in sys.argv[2:]] or [F16, Q5_0]
    lib, ref = load_lib(), load_ref()
    lib.whisper_log_set(None, None) if False else None
    stub = data_file("for-tests-ggml-tiny.en.bin" if cfg.endswith(".en") else "for-tests-ggml-tiny.bin")
    pcm = read_wav_f32(os.path.join(DATA_DIR, "jfk.wav"))
    tmp = tempfile.mkdtemp()
    for wt in wtypes:
        path = os.path.join(tmp, f"{cfg}-{NAMES[wt]}.bin")
        quantizer = (lambda t, w: ref_quantize(ref, t, w)) if wt in (Q4_K, Q5_K) else None
        synth.write_model(path, cfg, wt, seed=7, vocab_from=stub, quantizer=quantizer)
        print(f"=== {cfg} {NAMES[wt]}  ({os.path.getsize(path) / 1e6:.1f} MB)", flush=True)
        A = Side(lib, path, False); B = Side(ref, path, True)
        A.pcm_to_mel(pcm); B.pcm_to_mel(pcm)
        t0 = time.time(); A.encode(0); ta = time.time() - t0
        t0 = time.time(); B.encode(0); tb = time.time() - t0
        ta_, tb_ = taps(A), taps(B)
        print(f"encode wall: b200 {ta * 1e3:.1f} ms  ref {tb * 1e3:.1f} ms")
        for k in ("mel", "conv", "enc", "kc", "kv"):
            print(f"  {k:5s} max-rel {rel_err(ta_[k], tb_[k]):.3e}  rms-rel {rms_err(ta_[k], tb_[k]):.3e}  shape {ta_[k].shape}")
        print("  pad rows zero:", float(np.abs(ta_['kc'][:, 1500:]).max()), float(np.abs(tb_['kc'][:, 1500:]).max()))
        sot = A.L.whisper_token_sot(A.ctx)
        toks = [sot]
        n_past = 0
        agree = 0
        for step in range(12):
            la = A.decode(toks[-1:] if step else toks, n_past); lb = B.decode(toks[-1:] if step else toks, n_past)
            n_past += 1 if step else len(toks)
            ia, ib = int(la.argmax()), int(lb.argmax())
            srt = np.sort(lb)[::-1]
            print(f"  step {step:2d} logits max-rel {rel_err(la, lb):.3e} rms-rel {rms_err(la, lb):.3e} std {lb.std():.3f} argmax {ia} vs {ib} margin/std {(srt[0] - srt[1]) / lb.std():.3f}")
            agree += ia == ib
            toks.append(ib)
        print(f"  teacher-forced argmax agreement {agree}/12")
        for kw in (dict(temperature_inc=0.0), dict(temperature_inc=0.0, no_timestamps=True)):
            t0 = time.time(); ra, sa = A.full(pcm, **kw); ta = time.time() - t0
            t0 = time.time(); rb, sb = B.full(pcm, **kw); tb = time.time() - t0
            fa = [t for s in sa for t in s[2]]; fb = [t for s in sb for t in s[2]]
            common = 0
            for x, y in zip(fa, fb):
                if x != y: break
                common += 1
            print(f"  full {kw}: rc {ra}/{rb} segs {len(sa)}/{len(sb)} tokens {len(fa)}/{len(fb)} common-prefix {common}  wall b200 {ta:.2f}s ref {tb:.2f}s")
            print("     b200:", [(s[0], s[1], len(s[2])) for s in sa][:6])
            print("     ref :", [(s[0], s[1], len(s[2])) for s in sb][:6])
        A.free(); B.free()


if __name__ == "__main__":
    main()
