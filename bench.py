#!/usr/bin/env python
"""bench.py -- xRT (audio seconds / wall seconds) + encode ms of the Whisper hot path on B200.

Workload (BASELINE.json configs[3]): large-v3 Q5_0, synthetic weights (no checkpoints offline), a batch of 64 independent
30 s chunks per GPU, greedy decode (best_of=1, no temperature fallback), text tokens only (see full_params).  A "step" is one pass over the
rank's 64 chunks (all 64 sequences advance in lock-step: one batched encoder pass, one decode launch per token step).  Multi-GPU = independent chunks per rank, no collective on the data path
(weak scaling); torch.distributed is used only for the barrier and the max-over-ranks time.

  value  : xRT with the PCM already resident in HBM before the timed region (device pointers through the library's queue driver
           wb200_full_batch_ex, which runs whisper_full_with_state on pool states -- an input mode whisper.h itself does not have)
  e2e    : xRT through whisper.h ONLY, host PCM in, segments out: ONE call of whisper_full_parallel(ctx, params, pcm, n, 64) on the
           concatenation of the rank's 64 chunks (src/whisper.cpp:7813-7941 semantics: 64 states, one slice each).  H2D of the samples
           and D2H of the sampled tokens happen inside the timed region.  `e2e_threads` is the other reference-legal form: 64 caller
           threads x whisper_full_with_state on 64 states of the context (include/whisper.h:45-46).
  roofline / cpu_baseline : see DESIGN.md section 6

`--impl reference` times the reference's own CPU implementation (oracle/_ref, unmodified whisper.cpp) on a bounded
sample of the same workload (1 chunk per step) with all host threads.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from __graft_entry__ import load_pkg  # noqa: E402

CHUNKS_PER_GPU = 64
CHUNK_SECONDS = 30.0
MODEL_CFG = "large-v3"
WORKLOAD = "large-v3 Q5_0 (synthetic weights), %d x 30 s chunks per GPU, greedy best_of=1, no fallback, no_timestamps (224 tokens per chunk)" % CHUNKS_PER_GPU


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            j = json.load(f)
        return float(j.get("hbm_gbs", 6650.0)), float(j.get("bf16_tflops_sustained", 1400.0)), "measured"
    return 6650.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for i, n in enumerate(names):
                if len(r) > 4 + i and r[4 + i].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


_LOG_CB = C.CFUNCTYPE(None, C.c_int, C.c_char_p, C.c_void_p)
_quiet = _LOG_CB(lambda level, text, ud: None)


def silence(lib):
    """route the library's INFO chatter away from stdout/stderr (whisper_log_set, whisper.h:763)"""
    if os.environ.get("WB200_VERBOSE"):
        return
    lib.whisper_log_set.argtypes = [_LOG_CB, C.c_void_p]
    lib.whisper_log_set(_quiet, None)


def make_inputs(rank, n_chunks, seconds=CHUNK_SECONDS):
    """the chunks of one rank: independent work per GPU, seeded by rank (no data is exchanged between ranks)"""
    synth = load_pkg().synth
    return [synth.synth_audio(seed=1000 * rank + i, seconds=seconds) for i in range(n_chunks)]


def max_over_ranks(dt, world, device="cuda"):
    """the job is as slow as its slowest rank"""
    if world <= 1:
        return dt
    import torch
    import torch.distributed as dist
    t = torch.tensor([dt], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def ensure_model(path, wtype_name="q5_0"):
    synth = load_pkg().synth
    if not os.path.exists(path):
        tmp = path + ".tmp.%d" % os.getpid()
        synth.write_model(tmp, MODEL_CFG, synth.Q5_0, seed=0, fast_pool=True)
        os.replace(tmp, path)
    return path


def full_params(L, n_threads):
    p = L.whisper_full_default_params(0)
    p.print_progress = False
    p.greedy.best_of = 1
    p.temperature_inc = 0.0
    # Random weights never learn the timestamp grammar: with timestamps on, `seek` advances by whatever pair of timestamp tokens
    # happens to win, so some chunks crawl through 10+ windows while others finish in one (measured: 166 windows for 64 chunks,
    # 2677 decode steps of which most serve 1-3 straggler sequences).  Text-only decoding makes every chunk do the same, maximal
    # work: 1 window, n_text_ctx/2 = 224 tokens (2-3x the token rate of real speech), identical for the reference arm.
    p.no_timestamps = True
    p.n_threads = n_threads
    return p


def count_tokens(L, state):
    n = 0
    for i in range(L.whisper_full_n_segments_from_state(state)):
        n += L.whisper_full_n_tokens_from_state(state, i)
    return n


def collect_outputs(L, states):
    """what a caller of the timed path receives for each chunk: its tokens with their probabilities and the segment times, as arrays
    padded to the longest chunk (n_tokens / n_segments hold the true lengths)"""
    L.whisper_full_get_token_data_from_state.restype = load_pkg().TokenData
    L.whisper_full_get_token_data_from_state.argtypes = [C.c_void_p, C.c_int, C.c_int]
    toks, segs = [], []
    for st in states:
        n_seg = L.whisper_full_n_segments_from_state(st)
        segs.append([(L.whisper_full_get_segment_t0_from_state(st, s), L.whisper_full_get_segment_t1_from_state(st, s)) for s in range(n_seg)])
        toks.append([L.whisper_full_get_token_data_from_state(st, s, j) for s in range(n_seg) for j in range(L.whisper_full_n_tokens_from_state(st, s))])
    n_tok = max(1, max(len(t) for t in toks)); n_seg = max(1, max(len(s) for s in segs))
    arrays = {"token_ids": np.full((len(toks), n_tok), -1.0), "token_p": np.zeros((len(toks), n_tok), np.float32),
              "token_plog": np.zeros((len(toks), n_tok), np.float32), "n_tokens": np.array([len(t) for t in toks], np.float64),
              "segment_t0": np.full((len(segs), n_seg), -1.0), "segment_t1": np.full((len(segs), n_seg), -1.0),
              "n_segments": np.array([len(s) for s in segs], np.float64)}
    for i, t in enumerate(toks):
        arrays["token_ids"][i, :len(t)] = [d.id for d in t]
        arrays["token_p"][i, :len(t)] = [d.p for d in t]
        arrays["token_plog"][i, :len(t)] = [d.plog for d in t]
    for i, s in enumerate(segs):
        arrays["segment_t0"][i, :len(s)] = [a for a, _ in s]
        arrays["segment_t1"][i, :len(s)] = [b for _, b in s]
    return arrays


def dump_outputs(arrays, out_dir, rank):
    """<out_dir>/<name>.npy for each array of collect_outputs"""
    os.makedirs(out_dir, exist_ok=True)
    suffix = "_rank%d" % rank if rank else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def ref_threads():
    """thread budget of the reference CPU arm: all logical CPUs (WB200_REF_THREADS overrides)"""
    if os.environ.get("WB200_REF_THREADS"):
        return int(os.environ["WB200_REF_THREADS"])
    return os.cpu_count() or 1


def run_reference(args, rank, world):
    """reference arm: the unmodified whisper.cpp CPU path (oracle/_ref) with ALL host threads it can use.  A step is a bounded sample of
    the workload: P chunks through ONE whisper_full_parallel call (P states x cores/P ggml threads each).  (P, threads) is chosen by a
    sweep before the timed steps: a single stream stops scaling around 16-32 threads (per-node barriers of the 1-token graphs), several
    streams side by side use the rest of the cores -- the best of the sweep is what is timed and reported."""
    if rank != 0:
        return
    pkg = load_pkg()
    ref_path = os.path.join(ROOT, "oracle", "_ref", "libwhisper_ref.so")
    R = pkg.bind_whisper_api(C.CDLL(ref_path))
    silence(R)
    R.whisper_print_system_info.restype = C.c_char_p
    model = ensure_model(os.path.join(tempfile.gettempdir(), "wb200-%s-q5_0.bin" % MODEL_CFG))
    cp = R.whisper_context_default_params(); cp.use_gpu = False
    ctx = R.whisper_init_from_file_with_params(model.encode(), cp)
    assert ctx
    cores = ref_threads()
    pcms = make_inputs(0, 8)

    def one(P, nt, max_tokens=0):
        buf = np.ascontiguousarray(np.concatenate(pcms[:P]))
        p = full_params(R, nt)
        if max_tokens:
            p.max_tokens = max_tokens
        R.whisper_reset_timings(ctx)
        t0 = time.perf_counter()
        rc = R.whisper_full_parallel(ctx, p, buf.ctypes.data_as(C.c_void_p), len(buf), P) if P > 1 else R.whisper_full(ctx, p, buf.ctypes.data_as(C.c_void_p), len(buf))
        dt = time.perf_counter() - t0
        assert rc == 0
        return dt, float(R.whisper_get_timings(ctx).contents[1])

    cands = [(1, min(cores, 32))]
    if cores > 32: cands.append((1, cores))
    for P in (2, 4, 8):
        if cores // P >= 4: cands.append((P, cores // P))
    if os.environ.get("WB200_REF_NO_SWEEP"):
        cands = cands[:1]
    # the sweep runs a SHORT version of a step (whole encoder, 32 decoded tokens per chunk) and is bounded in time: on a 128-thread host
    # the full-length sweep alone took more than 7 minutes
    sweep = []
    t_sweep = time.perf_counter()
    for P, nt in cands:
        dt, _ = one(P, nt, max_tokens=32)
        sweep.append({"streams": P, "threads_per_stream": nt, "s_per_chunk_32_tokens": dt / P})
        if time.perf_counter() - t_sweep > 150.0:
            break
    best = min(sweep, key=lambda r: r["s_per_chunk_32_tokens"])
    P, nt = best["streams"], best["threads_per_stream"]
    times = []; enc_ms = []
    for it in range(args.warmup + args.steps):
        dt, enc = one(P, nt)
        if it >= args.warmup:
            times.append(dt); enc_ms.append(enc)
    total = sum(times)
    xrt = CHUNK_SECONDS * P * len(times) / total
    sample = "%d x 30 s chunk(s) per step, whisper_full%s greedy, %d stream(s) x %d threads (best of a sweep over %d settings)" % (P, "_parallel" if P > 1 else "", P, nt, len(sweep))
    out = {"impl": "reference", "metric": "xRT (audio-s/wall-s)", "value": xrt, "unit": "x real time", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "int8xint8->i32 block dot (Q5_0 x Q8_0), f32 accumulate", "data": "synthetic",
           "config": {"workload": WORKLOAD, "sample": sample},
           "encode_ms": float(np.mean(enc_ms)), "system_info": R.whisper_print_system_info().decode(), "host_logical_cpus": os.cpu_count(), "thread_sweep": sweep,
           "cpu_baseline": {"value": xrt, "unit": "x real time", "cores": P * nt, "kind": "reference", "sample": sample},
           "e2e": {"value": xrt, "unit": "x real time", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def _open_engine(pkg, model, local):
    silence(pkg.bind_whisper_api(C.CDLL(pkg.LIB_PATH)))
    eng = pkg.WhisperB200(model, gpu_device=local)
    L = eng.L
    vp = C.c_void_p
    L.whisper_full_with_state.argtypes = [vp, vp, pkg.FullParams, vp, C.c_int]
    L.wb200_counters.argtypes = [C.POINTER(C.c_double), C.c_int]
    return eng, L


def _timings(L, ctx):
    t = L.whisper_get_timings(ctx).contents
    return {"sample_ms": float(t[0]), "encode_ms": float(t[1]), "decode_ms": float(t[2]), "batchd_ms": float(t[3]), "prompt_ms": float(t[4])}


def run_config2(args, local):
    """BASELINE configs[1]: base.en Q5_0, single B200, ONE 30 s chunk, encoder + greedy decode with timestamps, through whisper_full"""
    import torch
    pkg = load_pkg(); synth = pkg.synth
    model = synth.cached_model("base.en", synth.Q5_0, seed=4, tag="s4")
    eng, L = _open_engine(pkg, model, local)
    pcm = torch.from_numpy(synth.synth_audio(seed=1234, seconds=30.0)).pin_memory()
    p = L.whisper_full_default_params(0); p.print_progress = False; p.greedy.best_of = 1; p.temperature_inc = 0.0; p.n_threads = 4
    times = []; tm = None; toks = 0
    for it in range(args.warmup + args.steps):
        L.whisper_reset_timings(eng.ctx)
        torch.cuda.synchronize(); t0 = time.perf_counter()
        assert L.whisper_full(eng.ctx, p, C.c_void_p(pcm.data_ptr()), pcm.numel()) == 0
        torch.cuda.synchronize(); dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt); tm = _timings(L, eng.ctx)
            toks = sum(L.whisper_full_n_tokens(eng.ctx, i) for i in range(L.whisper_full_n_segments(eng.ctx)))
    dt = float(np.mean(times))
    out = {"metric": "xRT (audio-s/wall-s)", "value": CHUNK_SECONDS / dt, "unit": "x real time", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 tcgen05 (encode) / int8 mma block dot (decode), f32 accumulate", "data": "synthetic",
           "config": {"workload": "BASELINE configs[1]: base.en Q5_0 (synthetic weights), one 30 s chunk, greedy best_of=1, timestamps on, whisper_full with host PCM"},
           "encode_ms": tm["encode_ms"], "decode_ms_per_token": tm["decode_ms"], "prompt_ms_per_token": tm["prompt_ms"], "decoded_tokens": toks,
           "e2e": {"value": CHUNK_SECONDS / dt, "unit": "x real time", "h2d_bytes_per_step": pcm.numel() * 4, "d2h_bytes_per_step": None}}
    print(json.dumps(out), flush=True)
    eng.close()


def run_config3(args, local):
    """BASELINE configs[2]: large-v3 Q4_K, single B200, beam_size 5, ONE 30-minute synthetic clip (60 x the 30 s generator, seeds 1234+i), whisper_full;
    a step is one whisper_full call on the whole clip"""
    import torch
    pkg = load_pkg(); synth = pkg.synth
    model = synth.cached_model("large-v3", synth.Q4_K, seed=0, fast_pool=True)
    eng, L = _open_engine(pkg, model, local)
    minutes = float(os.environ.get("WB200_CFG3_MINUTES", "30"))
    n_tiles = max(1, int(round(minutes * 2)))
    pcm = torch.from_numpy(np.concatenate([synth.synth_audio(seed=1234 + i, seconds=30.0) for i in range(n_tiles)])).pin_memory()
    p = L.whisper_full_default_params(1); p.print_progress = False; p.beam_search.beam_size = 5; p.temperature_inc = 0.0; p.n_threads = 4
    times = []
    for it in range(args.warmup + args.steps):
        if it == args.warmup:
            c0 = (C.c_double * 8)(); L.wb200_counters(c0, 8)
        L.whisper_reset_timings(eng.ctx)
        torch.cuda.synchronize(); t0 = time.perf_counter()
        assert L.whisper_full(eng.ctx, p, C.c_void_p(pcm.data_ptr()), pcm.numel()) == 0
        torch.cuda.synchronize(); times.append(time.perf_counter() - t0)
    c1 = (C.c_double * 8)(); L.wb200_counters(c1, 8)
    cd = [(c1[i] - c0[i]) / args.steps for i in range(8)]          # per timed step
    dt = float(np.mean(times[args.warmup:]))
    tm = _timings(L, eng.ctx)
    audio = pcm.numel() / 16000.0
    out = {"metric": "xRT (audio-s/wall-s)", "value": audio / dt, "unit": "x real time", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 tcgen05 (encode) / int8 block dot (decode), f32 accumulate", "data": "synthetic",
           "config": {"workload": "BASELINE configs[2]: large-v3 Q4_K (synthetic weights), beam_size 5, one %.0f-minute clip, whisper_full with host PCM (sequential windows: one stream)" % (audio / 60)},
           "encode_ms": tm["encode_ms"], "batchd_ms_per_token": tm["batchd_ms"], "sample_ms": tm["sample_ms"], "windows": cd[5], "decode_passes": cd[0], "rows_per_pass": cd[1] / max(1.0, cd[0]),
           "decoded_tokens": sum(L.whisper_full_n_tokens(eng.ctx, i) for i in range(L.whisper_full_n_segments(eng.ctx))),
           "e2e": {"value": audio / dt, "unit": "x real time", "h2d_bytes_per_step": pcm.numel() * 4, "d2h_bytes_per_step": None}}
    print(json.dumps(out), flush=True)
    eng.close()


def run_config5(args, rank, local, world):
    """BASELINE configs[4]: large-v3-turbo Q8_0, throughput sweep over the number of concurrent 30 s chunks (1 .. 64 per GPU = 1 .. 512 on 8 GPUs):
    c caller threads x whisper_full_with_state on c states of one context (whisper.h only); aggregate xRT and p50 / p99 chunk latency"""
    import torch
    import torch.distributed as dist
    pkg = load_pkg(); synth = pkg.synth
    if local == 0:
        synth.cached_model("large-v3-turbo", synth.Q8_0, seed=0, fast_pool=True)
    if world > 1:
        torch.cuda.set_device(local); dist.init_process_group("nccl", device_id=torch.device("cuda", local)); dist.barrier()
    model = synth.cached_model("large-v3-turbo", synth.Q8_0, seed=0, fast_pool=True)
    eng, L = _open_engine(pkg, model, local)
    vp = C.c_void_p
    pcms = [torch.from_numpy(x).pin_memory() for x in make_inputs(rank, 64)]
    p = full_params(L, 4)
    states = [L.whisper_init_state(eng.ctx) for _ in range(64)]
    assert all(states), L.wb200_last_error()
    rows = []
    for c in (1, 2, 4, 8, 16, 32, 64):
        lat = []
        def work(i, out):
            t0 = time.perf_counter()
            rc = L.whisper_full_with_state(eng.ctx, states[i], p, vp(pcms[i].data_ptr()), pcms[i].numel())
            out[i] = (rc, time.perf_counter() - t0)
        reps = 1 + args.steps
        wall = 0.0
        for rep in range(reps):
            res = [None] * c
            th = [threading.Thread(target=work, args=(i, res)) for i in range(c)]
            if world > 1: dist.barrier()
            torch.cuda.synchronize(); t0 = time.perf_counter()
            for t in th: t.start()
            for t in th: t.join()
            torch.cuda.synchronize(); dt = time.perf_counter() - t0
            assert all(r[0] == 0 for r in res)
            if rep > 0:
                wall += max_over_ranks(dt, world); lat += [r[1] for r in res]
        rows.append({"concurrent_chunks": c * world, "xrt": CHUNK_SECONDS * c * world * (reps - 1) / wall, "chunk_latency_ms_p50": 1e3 * float(np.percentile(lat, 50)),
                     "chunk_latency_ms_p99": 1e3 * float(np.percentile(lat, 99)), "ms_per_wave": 1e3 * wall / (reps - 1)})
    if rank == 0:
        best = max(rows, key=lambda r: r["xrt"])
        out = {"metric": "xRT (audio-s/wall-s)", "value": best["xrt"], "unit": "x real time", "n_gpus": world, "steps": args.steps, "warmup": 1, "ms_per_step": best["ms_per_wave"],
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 tcgen05 (encode) / int8 mma block dot (decode), f32 accumulate", "data": "synthetic",
               "config": {"workload": "BASELINE configs[4]: large-v3-turbo Q8_0 (synthetic weights), sweep of concurrent 30 s chunks (threads x whisper_full_with_state, whisper.h only), greedy, no_timestamps"},
               "sweep": rows, "latency_note": "chunk latency of rank 0's chunks (submit -> transcript), rank-local clocks",
               "e2e": {"value": best["xrt"], "unit": "x real time", "h2d_bytes_per_step": None, "d2h_bytes_per_step": None}}
        print(json.dumps(out), flush=True)
    for st in states: L.whisper_free_state(st)
    eng.close()
    if world > 1: dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chunks", type=int, default=CHUNKS_PER_GPU, help="chunks per GPU (weak scaling)")
    ap.add_argument("--chunks-total", type=int, default=0, help="strong scaling: this many chunks in total, split over the ranks")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ragged", action="store_true", help="skip the timestamps-on extra step")
    ap.add_argument("--config", type=int, default=4, choices=[2, 3, 4, 5], help="BASELINE.json configs[i-1]: 4 = the default line; 2, 3, 5 print their own JSON line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the tokens and segments of the last timed step as DIR/<name>.npy (default workload only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config != 4):
        ap.error("--dump-outputs applies to the default workload (--impl b200 --config 4)")

    rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.config == 2:
        return run_config2(args, local) if rank == 0 else None
    if args.config == 3:
        return run_config3(args, local) if rank == 0 else None
    if args.config == 5:
        return run_config5(args, rank, local, world)

    import torch
    import torch.distributed as dist
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pkg = load_pkg()
    model = os.path.join(tempfile.gettempdir(), "wb200-%s-q5_0.bin" % MODEL_CFG)
    if local == 0:
        ensure_model(model)
    if world > 1:
        dist.barrier()

    silence(pkg.bind_whisper_api(C.CDLL(pkg.LIB_PATH)))
    eng = pkg.WhisperB200(model, gpu_device=local)
    L = eng.L
    vp = C.c_void_p
    L.whisper_full_with_state.argtypes = [vp, vp, pkg.FullParams, vp, C.c_int]
    L.wb200_pcm_upload.argtypes = [vp, vp, C.c_int]
    L.wb200_traffic.argtypes = [C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.wb200_profile_collect.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.wb200_last_encode_ms.argtypes = [vp, C.POINTER(C.c_float)]
    n_chunks = args.chunks
    scaling = "weak"
    if args.chunks_total > 0:
        assert args.chunks_total % world == 0, "--chunks-total must be a multiple of the number of ranks"
        n_chunks = args.chunks_total // world; scaling = "strong"
    pcms = make_inputs(rank, n_chunks)
    pinned = [torch.from_numpy(p).pin_memory() for p in pcms]          # e2e copies start from pinned host memory
    resident = [t.cuda(local, non_blocking=False) for t in pinned]     # `value`: PCM already in HBM
    L.wb200_full_batch_ex.argtypes = [vp, pkg.FullParams, C.POINTER(vp), C.POINTER(C.c_int), C.c_int, C.POINTER(vp), C.c_int]
    p = full_params(L, 4)
    n_arr = (C.c_int * n_chunks)(*[len(x) for x in pcms])
    host_ptrs = (vp * n_chunks)(*[t.data_ptr() for t in pinned])
    dev_ptrs = (vp * n_chunks)(*[t.data_ptr() for t in resident])
    last = {"tokens": 0, "enc": None}

    concat = torch.from_numpy(np.concatenate(pcms)).pin_memory()       # whisper_full_parallel input: one host buffer, sliced by the library
    states = []

    def run_pass(mode, keep=False):
        """one step = all chunks of this rank.  mode "device": PCM resident in HBM (library queue driver); "parallel": one
        whisper_full_parallel call on host PCM; "threads": one caller thread per chunk, whisper_full_with_state on its own state.
        keep (device mode): copy the results into last["outputs"] before the states are freed, and the host time that takes into
        last["keep_s"]"""
        if mode == "parallel":
            rc = L.whisper_full_parallel(eng.ctx, p, vp(concat.data_ptr()), concat.numel(), n_chunks)
            assert rc == 0, (rc, L.wb200_last_error())
            last["tokens"] = sum(L.whisper_full_n_tokens(eng.ctx, i) for i in range(L.whisper_full_n_segments(eng.ctx)))
            return
        if mode == "threads":
            while len(states) < n_chunks:
                st = L.whisper_init_state(eng.ctx); assert st, L.wb200_last_error()
                states.append(st)
            rcs = [None] * n_chunks

            def work(i):
                rcs[i] = L.whisper_full_with_state(eng.ctx, states[i], p, host_ptrs[i], n_arr[i])
            th = [threading.Thread(target=work, args=(i,)) for i in range(n_chunks)]
            for t in th: t.start()
            for t in th: t.join()
            assert rcs == [0] * n_chunks, (rcs, L.wb200_last_error())
            last["tokens"] = sum(count_tokens(L, st) for st in states)
            return
        outs = (vp * n_chunks)()
        rc = L.wb200_full_batch_ex(eng.ctx, p, dev_ptrs, n_arr, n_chunks, outs, 1)
        assert rc == 0, (rc, L.wb200_last_error())
        last["tokens"] = sum(count_tokens(L, outs[i]) for i in range(n_chunks))
        if keep:
            t0 = time.perf_counter()
            last["outputs"] = collect_outputs(L, [outs[i] for i in range(n_chunks)])
            last["keep_s"] = time.perf_counter() - t0
        for i in range(n_chunks):
            L.whisper_free_state(outs[i])

    def timed(mode, steps, warmup, keep_last=False):
        for _ in range(warmup):
            run_pass(mode)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        h0, d0 = C.c_uint64(), C.c_uint64(); L.wb200_traffic(C.byref(h0), C.byref(d0))
        n0 = eng.launch_count()
        t0 = time.perf_counter()
        for i in range(steps):
            run_pass(mode, keep=keep_last and i == steps - 1)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0 - last.pop("keep_s", 0.0)      # the copy for --dump-outputs is host work outside the step
        h1, d1 = C.c_uint64(), C.c_uint64(); L.wb200_traffic(C.byref(h1), C.byref(d1))
        launches = eng.launch_count() - n0
        dt = max_over_ranks(dt, world)
        return dt, launches, (h1.value - h0.value) / steps, (d1.value - d0.value) / steps

    def counters():
        a = (C.c_double * 8)(); L.wb200_counters(a, 8); return [a[i] for i in range(8)]
    L.wb200_counters.argtypes = [C.POINTER(C.c_double), C.c_int]

    # ---- device-resident inputs ("value")
    sampler = ClockSampler(local); sampler.start()
    for _ in range(args.warmup):
        run_pass("device")
    c0 = counters()
    dt_res, launches, _, _ = timed("device", args.steps, 0, keep_last=bool(args.dump_outputs))
    c1 = counters()
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(last.pop("outputs"), args.dump_outputs, rank)
    cd = [b - a for a, b in zip(c0, c1)]
    engine_stats = {"decode_passes_per_step": cd[0] / args.steps, "decode_rows_per_pass": cd[1] / max(cd[0], 1), "decode_gpu_ms_per_pass": cd[2] / max(cd[0], 1),
                    "decode_host_ms_per_pass": cd[3] / max(cd[0], 1), "encode_calls_per_step": cd[4] / args.steps, "encode_windows_per_step": cd[5] / args.steps,
                    "encode_gpu_ms_per_window": cd[6] / max(cd[5], 1), "graph_replays_per_step": cd[7] / args.steps}
    audio_s = CHUNK_SECONDS * n_chunks * args.steps * world
    value = audio_s / dt_res
    tokens = last["tokens"]

    # ---- host buffers through the C ABI ("e2e")
    dt_e2e, _, h2d, d2h = timed("parallel", args.steps, max(1, args.warmup))
    e2e = audio_s / dt_e2e
    tokens_e2e = last["tokens"]
    dt_thr, _, h2d_t, d2h_t = timed("threads", args.steps, max(1, args.warmup))
    e2e_threads = audio_s / dt_thr

    # ---- encode ms of ONE 30 s window (whisper-bench "Enc." semantics: conv + encoder + cross, bench.cpp:63-150) on the default state
    st0 = L.wb200_ctx_state(eng.ctx)
    L.whisper_pcm_to_mel.argtypes = [vp, vp, C.c_int, C.c_int]
    assert L.whisper_pcm_to_mel(eng.ctx, vp(pinned[0].data_ptr()), len(pcms[0]), 1) == 0
    enc = (C.c_float * 4)()
    enc_runs = []
    for _ in range(5):
        assert L.whisper_encode(eng.ctx, 0, 1) == 0
        L.wb200_last_encode_ms(st0, enc)
        enc_runs.append([float(enc[i]) for i in range(4)])
    enc = enc_runs[-1]

    # ---- encoder against the tensor roofline: algorithmic FLOPs of one window (SURVEY.md 8d: conv + encoder with the 1536 padded keys + cross K/V)
    hp = {k: getattr(L, "whisper_model_" + k)(eng.ctx) for k in ("n_audio_state", "n_audio_layer", "n_text_layer", "n_mels", "n_audio_ctx")}
    d_, La_, Lt_, M_, T_ = hp["n_audio_state"], hp["n_audio_layer"], hp["n_text_layer"], hp["n_mels"], hp["n_audio_ctx"]
    Tp_ = (T_ + 255) // 256 * 256
    enc_flops = 2 * 2 * T_ * 3 * M_ * d_ + 2 * T_ * 3 * d_ * d_ + La_ * (24 * T_ * d_ * d_ + 4 * T_ * Tp_ * d_) + Lt_ * 4 * T_ * d_ * d_
    _, tf_sus, how = measured_peaks()
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            tf_burst = float(json.load(f).get("bf16_tflops", tf_sus))
    except Exception:  # noqa: BLE001
        tf_burst = tf_sus
    enc_b_ms = engine_stats["encode_gpu_ms_per_window"]; enc_1_ms = float(enc[1] + enc[2] + enc[3])
    encode_roofline = {"bound": "tensor", "flops_per_window": enc_flops, "unit": "TFLOP/s", "peak_source": how,
                       "batched": {"ms_per_window": enc_b_ms, "achieved": enc_flops / enc_b_ms / 1e9, "peak": tf_sus, "frac": enc_flops / enc_b_ms / 1e9 / tf_sus, "peak_kind": "sustained bf16 (timed inside a long step)"},
                       "single_window": {"ms": enc_1_ms, "achieved": enc_flops / enc_1_ms / 1e9, "peak": tf_burst, "frac": enc_flops / enc_1_ms / 1e9 / tf_burst, "peak_kind": "burst bf16 (timed alone)"}}

    # ---- the same 64 chunks with TIMESTAMPS ON (one untimed-by-the-driver extra step): windows end where the sampled timestamps say, so the
    # sequences are ragged, rows drop out of the passes at different times and some chunks need several windows (random weights never learn
    # the timestamp grammar: this is a worst case for lock-step batching, reported beside the text-only workload, never as `value`)
    ragged = None
    if not args.no_ragged:
        p_ts = full_params(L, 4); p_ts.no_timestamps = False
        c0 = counters(); torch.cuda.synchronize(); t0 = time.perf_counter()
        rc = L.whisper_full_parallel(eng.ctx, p_ts, vp(concat.data_ptr()), concat.numel(), n_chunks)
        torch.cuda.synchronize(); dt_r = time.perf_counter() - t0; c1 = counters()
        assert rc == 0, (rc, L.wb200_last_error())
        cr = [b - a for a, b in zip(c0, c1)]
        ragged = {"value": CHUNK_SECONDS * n_chunks / dt_r, "unit": "x real time", "ms": 1e3 * dt_r, "decode_passes": cr[0], "rows_per_pass": cr[1] / max(cr[0], 1),
                  "encode_windows": cr[5], "tokens": sum(L.whisper_full_n_tokens(eng.ctx, i) for i in range(L.whisper_full_n_segments(eng.ctx))),
                  "what": "same chunks, timestamps on, one whisper_full_parallel call (rank 0's share)"}

    out = {"metric": "xRT (audio-s/wall-s)", "value": value, "unit": "x real time", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": 1e3 * dt_res / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
           "dtype": "f16 tcgen05 (encode) / int8 mma block dot (decode), f32 accumulate", "data": "synthetic",
           "config": {"workload": WORKLOAD, "chunks_per_gpu": n_chunks, "decode": "lock-step batch of up to 64 sequences per GPU, one persistent cooperative kernel per token step", "l2": "weights (1.08 GB) + KV (0.3 GB/sequence) streamed every step exceed the 126 MB L2",
                      "timing": "host wall clock between device synchronisations around whole steps (a step contains host control flow), max over ranks; per-kernel numbers from CUDA events on the launching stream"},
           "encode_ms": float(enc[1] + enc[2] + enc[3]), "encode_ms_parts": {"mel": float(enc[0]), "conv": float(enc[1]), "encoder": float(enc[2]), "cross": float(enc[3])},
           "decoded_tokens_per_step": tokens, "engine": engine_stats, "clocks": clocks, "gpu_launches": int(launches),
           "encode_roofline": encode_roofline, "ragged": ragged,
           "e2e": {"value": e2e, "unit": "x real time", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * dt_e2e / args.steps,
                   "api": "whisper_full_parallel(ctx, params, host_pcm, n_samples, n_processors=%d) -- whisper.h only" % n_chunks, "decoded_tokens_per_step": tokens_e2e},
           "e2e_threads": {"value": e2e_threads, "unit": "x real time", "h2d_bytes_per_step": int(h2d_t), "d2h_bytes_per_step": int(d2h_t),
                           "api": "%d threads x whisper_full_with_state(ctx, state_i, params, host_pcm_i, n) -- whisper.h only" % n_chunks}}

    if rank == 0:
        # ---- roofline of the dominant kernel class: separate pass of ONE chunk with per-launch CUDA events (library side,
        # on the launching stream); not inside the timed region so the event overhead does not perturb `value`
        L.wb200_profile_enable(1)
        run_pass("device")
        ms = (C.c_double * 4)(); ln = (C.c_uint64 * 4)(); by = (C.c_double * 4)(); fl = (C.c_double * 4)()
        L.wb200_profile_collect(ms, ln, by, fl)
        L.wb200_profile_enable(0)
        hbm, tf, how = measured_peaks()
        names = ["tcgen05_gemm", "decode_pass_persistent", "decode_attention", "other"]
        classes = {names[i]: {"ms": ms[i], "launches": int(ln[i]), "GBps": (by[i] / 1e9) / (ms[i] / 1e3) if ms[i] > 0 else 0.0,
                              "TFLOPs": (fl[i] / 1e12) / (ms[i] / 1e3) if ms[i] > 0 else 0.0} for i in range(4)}
        dom = max(range(3), key=lambda i: ms[i])
        if dom == 0:
            roof = {"kernel": names[0], "bound": "tensor", "achieved": classes[names[0]]["TFLOPs"], "peak": tf, "unit": "TFLOP/s", "frac": classes[names[0]]["TFLOPs"] / tf, "traffic": None, "peak_source": how + " (sustained bf16)"}
        else:
            roof = {"kernel": names[dom], "bound": "hbm", "achieved": classes[names[dom]]["GBps"], "peak": hbm, "unit": "GB/s", "frac": classes[names[dom]]["GBps"] / hbm, "traffic": None, "peak_source": how}
        # DRAM traffic of one launch of the dominant kernel from the committed `ncu --set full` capture (profiles/), if it is the same kernel
        try:
            with open(os.path.join(ROOT, "profiles", "r02_ncu_decode_pass.json")) as f:
                cap = json.load(f)
            if dom == 1 and cap.get("rows") == min(n_chunks, 64):
                roof["traffic"] = cap["dram_bytes_read"] + cap["dram_bytes_write"]
                roof["traffic_source"] = "profiles/r02_ncu_decode_pass.json (one launch, %d rows)" % cap["rows"]
                roof["algorithmic_bytes_per_launch"] = (by[dom] / ln[dom]) if ln[dom] else None
        except Exception:  # noqa: BLE001
            pass
        out["roofline"] = roof
        out["kernel_classes"] = classes
        if not args.no_cpu_baseline:
            # the unmodified reference on ONE chunk of the same workload, in a child process so that it can be bounded in time
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                                   capture_output=True, text=True, timeout=420)
                j = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
                out["cpu_baseline"] = dict(j["cpu_baseline"], encode_ms=j.get("encode_ms"))
            except Exception as e:  # noqa: BLE001
                out["cpu_baseline"] = {"value": None, "unit": "x real time", "cores": ref_threads(), "kind": "reference",
                                       "sample": "1 x 30 s chunk (did not finish: %s)" % type(e).__name__}
        if os.environ.get("WB200_BENCH_REF_TOOL", "1") == "1" and world == 1:
            # the reference's OWN benchmark program, unmodified, linked against this library
            # (oracle/_ref/whisper-bench-b200 = examples/bench/bench.cpp): encode / decode / batched / prompt ms per run as whisper_print_timings reports
            try:
                import re
                exe = os.path.join(ROOT, "oracle", "_ref", "whisper-bench-b200")
                r = subprocess.run([exe, "-m", model, "-t", "4"], capture_output=True, text=True, timeout=300)
                out["whisper_bench_tool"] = {name: {"ms_per_run": float(per), "runs": int(runs)} for name, total, runs, per in
                                             re.findall(r"(\w+) time =\s*([\d.]+) ms /\s*(\d+) runs \(\s*([\d.]+) ms per run\)", r.stderr + r.stdout)}
            except Exception as e:  # noqa: BLE001
                out["whisper_bench_tool"] = {"error": type(e).__name__}
        print(json.dumps(out), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
