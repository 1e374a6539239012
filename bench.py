#!/usr/bin/env python
"""bench.py -- the BASELINE.json metric: clips/sec for 10 s @ 44.1 kHz stereo clips through
LUFS-normalise (-24) + log-mel (n_fft 2048, hop 512, 128 mels)  [BASELINE.json configs[1]].

  python bench.py [--gpus N --steps K --warmup W] [--dump-outputs DIR] our arm (CUDA, one rank per GPU)
  python bench.py --impl reference [--gpus N --steps K --warmup W]    the reference's CPU path (oracle port)

--dump-outputs DIR writes what the last timed step returned on rank 0 (see dump_sample) as DIR/<name>.npy, float32:
the inputs are seeded, so two builds run with the same arguments can be compared output for output.

One "step" = one pass of the hot path over one batch of 64 clips per GPU (weak scaling): the
loudness kernels, then the fused gain + STFT + mel + log kernel.  Outputs per step: normalised
waveform [B,2,441000], log-mel [B,2,128,862], LUFS [B].

  value     whole-job clips/s with inputs resident in HBM (device-timed, max over ranks)
  e2e       the same metric through the public AudioSignal API with HOST (pinned) buffers on both sides: the H2D
            copy of every step's batch and the D2H copy of ALL its results (normalised waveform, log-mel, LUFS)
            are inside the timed region (copies double-buffered on their own streams)
  roofline  the dominant kernel (fused spectral) vs the measured HBM copy bandwidth
  cpu_baseline  the oracle (CPU port of the reference path) on this box's host cores, bounded sample
Timing hygiene: >= 3 warm-ups plus a >= 1 s identical pre-roll, barrier, one untimed post-barrier step, then
EXACTLY K steps between CUDA events on the launching stream (max over ranks); inputs rotate over 3 distinct
226 MB batches (each > the 126 MB L2); nvidia-smi clocks are sampled from before the pre-roll to the end of a
>= 2 s sustained loop of the same step (reported next to the K-step figure).  At N > 1 the per-item LUFS
exchange (csrc/peer.cu) runs on its own stream, never waits for another rank inside a step, and is validated
once, untimed, against an NCCL all_gather of the same vector.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

SR, T, C = 44100, 441000, 2
N_FFT, HOP, N_MELS, TARGET_DB = 2048, 512, 128, -24.0
N_FRAMES = 1 + T // HOP
BYTES_X = C * T * 4
BYTES_MEL = C * N_MELS * N_FRAMES * 4
WORKLOAD = "batch=64/GPU 2ch 10s@44.1kHz LUFS-normalize(-24)+log-mel(n_fft=2048,hop=512,n_mels=128)"


def make_batch(B, seed, device="cpu"):
    """SURVEY.md §8d synthetic input: 0.1*randn clipped, per-item gain U(0.05, 1)."""
    import torch

    g = torch.Generator().manual_seed(seed)
    x = (0.1 * torch.randn(B, C, T, generator=g)).clamp(-1, 1)
    x = x * (0.05 + 0.95 * torch.rand(B, 1, 1, generator=g))
    return x.float().to(device)


DUMP_MAX_ELEMS = 1 << 22  # 16 MiB of float32 per array: a step's two large outputs and three [B] vectors stay < 64 MB


def dump_sample(arrays):
    """Host float32 copies of the device tensors ``arrays``.  One with more than DUMP_MAX_ELEMS elements is replaced by
    DUMP_MAX_ELEMS of its flattened elements, one drawn from each of that many equal strides by a generator seeded
    with 0: the same shape always gives the same positions."""
    import numpy as np
    import torch

    out = {}
    for name, t in arrays.items():
        n = t.numel()
        if n > DUMP_MAX_ELEMS:
            stride = n // DUMP_MAX_ELEMS
            idx = np.arange(DUMP_MAX_ELEMS) * stride + np.random.default_rng(0).integers(0, stride, DUMP_MAX_ELEMS)
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        out[name] = t.float().cpu().numpy()
    return out


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path
# ----------------------------------------------------------------------------------------------
def cpu_pipeline(x):
    from oracle import signal_path as sp

    y, lufs = sp.normalize(x, SR, TARGET_DB)
    mel = sp.mel_spectrogram(y, SR, N_MELS, window_length=N_FFT, hop_length=HOP, window_type="hann")
    return y, sp.log_mel(mel), lufs


def time_cpu(n_clips, reps, warmup):
    """Time the CPU port on ``n_clips`` clips.  torch's default (one thread per core) oversubscribes torch.stft /
    lfilter on a many-core host, so the thread count is calibrated first on a 4-clip sample and the fastest setting
    is used: the reference arm gets its best configuration, not an accidental slow one."""
    import torch

    cores = os.cpu_count() or 1
    x = make_batch(n_clips, 1234)
    cand = sorted({c for c in (cores, 64, 32, 16, 8) if 1 <= c <= cores}, reverse=True)
    best, best_t = cores, float("inf")
    if len(cand) > 1:
        xs = x[: min(4, n_clips)]
        torch.set_num_threads(cand[0])
        cpu_pipeline(xs)  # page in, build windows / filterbanks
        for c in cand:
            torch.set_num_threads(c)
            t0 = time.perf_counter()
            cpu_pipeline(xs)
            dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = c, dt
    torch.set_num_threads(best)
    for _ in range(warmup):
        cpu_pipeline(x)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        cpu_pipeline(x)
        ts.append(time.perf_counter() - t0)
    return ts, best


def make_config(world, B, exchange_kind=None):
    """The `config` object of the JSON line: identical for both arms at the same N (the driver compares them)."""
    return {"workload": WORKLOAD, "global_batch": world * B, "per_gpu_batch": B,
            "parallelism": f"batch-sharded x{world}, no data-path collective"
                           + (" (+ per-item LUFS exchange on a side stream)" if world > 1 else ""),
            "l2": f"inputs rotate over 3 distinct {B * BYTES_X / 1e6:.0f} MB batches (> 126 MB L2)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    n_clips = args.batch  # one step = the full per-GPU batch of the workload, on this box's host cores
    ts, cores = time_cpu(n_clips, reps=max(1, args.steps), warmup=max(1, args.warmup))
    total = sum(ts)
    value = n_clips * len(ts) / total
    line = {
        "impl": "reference", "metric": "clips/sec (10s@44.1kHz) log-mel+LUFS pipeline", "value": value,
        "unit": "clips/s", "n_gpus": args.gpus, "steps": len(ts), "warmup": max(1, args.warmup),
        "ms_per_step": 1e3 * total / len(ts), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": make_config(max(world, args.gpus), args.batch),
        "cpu_baseline": {"value": value, "unit": "clips/s", "cores": cores, "kind": "port",
                         "sample": f"the full {n_clips}-clip batch per step, {len(ts)} steps after {max(1, args.warmup)} "
                                   f"warm-ups; torch threads calibrated over {{all cores, 64, 32, 16, 8}} on 4 clips, "
                                   f"fastest used; one host (rank 0) whatever N"},
        "e2e": {"value": value, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference CPU path = the in-repo oracle port (torch.stft + torchaudio.lfilter + restated "
                "pyloudnorm/librosa); the reference package itself cannot be installed here (see DESIGN.md)",
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi polled every 100 ms for one GPU, each row stamped with the host clock so that windows (pre-roll,
    timed region, sustained loop) can be cut out afterwards."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass

    def summary(self, t_lo=None, t_hi=None):
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in self.rows:
            if (t_lo is not None and ts < t_lo) or (t_hi is not None and ts > t_hi):
                continue
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                pw.append(float(r[2]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    import __graft_entry__ as graft

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a B200: there is no CPU fallback. Use --impl reference "
                         "for the CPU path.")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        graft.build()
    if world > 1:
        dist.barrier()
    from audiotools_b200 import AudioSignal, _lib
    from audiotools_b200.engine import get_engine

    eng = get_engine()
    if args.tc:  # A/B switch: the tensor-core spectral kernel (csrc/spectral_tc.cu) instead of the default FP32 kernel
        eng.lib.b2a_spectral_tc_enable(1)
    B = args.batch
    NBUF = 3
    xs = [make_batch(B, 100 + 7 * rank + i, dev) for i in range(NBUF)]
    db = torch.tensor([TARGET_DB], device=dev)
    win = AudioSignal.get_window("hann", N_FFT, dev)
    fb, lo, hi = AudioSignal._mel_tables(SR, N_FFT, N_MELS, 0.0, None, dev)

    # Whole-batch loudness statistics (the path's only exchange: 256 B per rank and step), logging data.  One-sided
    # stores into every peer's buffer over NVLink (csrc/peer.cu) on the exchange's OWN stream: a put and a
    # non-blocking read of the newest statistics per step; no rank ever waits for another inside a step.  Fallback if
    # the peer mapping cannot be set up: NCCL all-gather on a side stream, consumed one step late.
    exchange, gather, exchange_kind = None, None, "none"
    if world > 1 and not os.environ.get("B2A_BENCH_NO_GATHER"):
        try:
            if os.environ.get("B2A_BENCH_NCCL_GATHER"):
                raise RuntimeError("NCCL all-gather requested")
            from audiotools_b200.parallel import PeerLoudnessExchange

            exchange = PeerLoudnessExchange(n_max=B)
            exchange_kind = "peer-store (cudaIpc + NVLink P2P stores, csrc/peer.cu), side stream, non-blocking"
        except Exception as e:  # noqa: BLE001
            from audiotools_b200.parallel import LoudnessGather

            gather = LoudnessGather(side_stream=torch.cuda.Stream(device=dev))
            exchange_kind = f"nccl all_gather on a side stream ({type(e).__name__}: {e})"
    spec_events = []
    stats = {}  # newest whole-batch statistics seen (values, per-rank sequence numbers): logging data

    def step(i, timed=False):
        x = xs[i % NBUF]
        lu = eng.lufs(x, SR, target_db=db)
        if exchange is not None:
            stats["seq"] = exchange.put(lu["loud"])
            stats["latest"] = exchange.latest()
        elif gather is not None:
            gather.wait()  # the previous step's gather (long complete)
            stats["all"] = gather(lu["loud"])
        if timed:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        out = eng.spectral(x, N_FFT, HOP, win, gain=lu["gain"], want_scaled=True, mel_fb=fb, mel_lo=lo, mel_hi=hi,
                           post=_lib.POST_LOG10, post_eps=1e-5, post_power=2.0, want_stft=False)
        if timed:
            e1.record()
            spec_events.append((e0, e1))
        return out, lu

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-resident timing.  The clock sampler starts BEFORE everything (its fork is expensive and differs
    #      per rank: it must never sit between the barrier and t0).
    with ClockSampler(local) as clocks:
        for i in range(args.warmup):
            step(i)
        torch.cuda.synchronize()
        # every rank must run the SAME number of steps (the exchange's sequence numbers advance per put): rank 0 sizes
        # the pre-roll and the sustained loop from its own step time and broadcasts the counts
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for i in range(10):
            step(i)
        c1.record()
        torch.cuda.synchronize()
        est_ms = max(c0.elapsed_time(c1) / 10.0, 1e-3)
        counts = torch.tensor([max(20, int(args.preroll * 1e3 / est_ms)) if args.preroll > 0 else 0,
                               max(args.steps, int(args.sustain * 1e3 / est_ms)) if args.sustain > 0 else 0],
                              device=dev, dtype=torch.int64)
        if world > 1:
            dist.broadcast(counts, src=0)
        n_pre, n_sus = int(counts[0].item()), int(counts[1].item())
        w_pre0 = time.perf_counter()
        for i in range(n_pre):  # identical steps: clocks / power settle under the real load
            step(i)
        torch.cuda.synchronize()
        barrier()
        step(0)  # one untimed post-barrier step: absorbs the rank skew of leaving the barrier
        torch.cuda.synchronize()
        launches0 = eng.launches
        xl0 = exchange.launches if exchange is not None else 0
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(args.steps):
            last = step(args.warmup + i, timed=True)
            if i + 1 < args.steps:
                last = None  # freed before the next step, whose outputs then reuse the memory
        t1.record()
        torch.cuda.synchronize()
        dumped = None
        if args.dump_outputs and rank == 0:  # the last timed step's results: dict(lufs, loud, gain, mel, scaled)
            dumped = dump_sample({k: v for d in (last[1], last[0]) for k, v in d.items() if v is not None})
        last = None
        w_timed1 = time.perf_counter()
        ms_rank = t0.elapsed_time(t1)
        launches = eng.launches - launches0 + (exchange.launches - xl0 if exchange is not None else 0)
        # sustained figure: the same step for >= args.sustain seconds (SM clocks settle under the power cap)
        sus = None
        if n_sus > 0:
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for i in range(n_sus):
                step(i)
            s1.record()
            torch.cuda.synchronize()
            sus = (n_sus, s0.elapsed_time(s1))
        w_end = time.perf_counter()
        barrier()
    spec_ms = sum(a.elapsed_time(b) for a, b in spec_events) / max(1, len(spec_events))
    per_rank = [ms_rank]
    if world > 1:
        tms = torch.tensor([ms_rank], device=dev, dtype=torch.float64)
        allms = [torch.zeros_like(tms) for _ in range(world)]
        dist.all_gather(allms, tms)
        per_rank = [float(t.item()) for t in allms]
    ms = max(per_rank)
    value = world * B * args.steps / (ms * 1e-3)
    sus_line = None
    if sus is not None:
        tsu = torch.tensor([sus[1] / sus[0]], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tsu, op=dist.ReduceOp.MAX)
        sus_line = {"ms_per_step": float(tsu.item()), "steps": sus[0], "value": world * B / (float(tsu.item()) * 1e-3),
                    "unit": "clips/s", "clocks": clocks.summary(w_timed1, w_end)}

    # ---- untimed validation of the exchange: the gathered vector of one step equals NCCL's all_gather of it
    exchange_line = None
    if world > 1:
        exchange_line = {"kind": exchange_kind}
        out, lu = step(1)
        torch.cuda.synchronize()
        ref = torch.empty(world * B, device=dev)
        dist.all_gather_into_tensor(ref, lu["loud"].contiguous())
        if exchange is not None:
            vals, seqs = stats["latest"]
            exchange.wait()
            torch.cuda.synchronize()
            lag = int(stats["seq"]) - int(seqs.min().item())  # how stale the non-blocking read of the last step was
            got, cseqs = exchange.collect(stats["seq"], return_seqs=True)
            exchange.wait()
            torch.cuda.synchronize()
            ok = bool(torch.equal(got, ref)) and cseqs.tolist() == [stats["seq"]] * world and exchange.status() == 0
            exchange_line.update({"validated_vs_nccl_all_gather": ok, "last_read_lag_steps": lag,
                                  "waits_inside_step": 0})
        else:
            gather.wait()
            torch.cuda.synchronize()
            ok = bool(torch.equal(stats["all"], ref))
            exchange_line.update({"validated_vs_nccl_all_gather": ok})
        flag = torch.tensor([1.0 if ok else 0.0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        assert flag.item() == 1.0, "per-item LUFS exchange disagrees with NCCL all_gather"

    # ---- end to end through the public API: HOST (pinned) inputs and HOST (pinned) results, copies double-buffered
    hx = [make_batch(B, 500 + i).pin_memory() for i in range(2)]
    copy_in, copy_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    dbuf = [torch.empty(B, C, T, device=dev) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]
    h_y = [torch.empty(B, C, T, pin_memory=True) for _ in range(2)]
    h_mel = [torch.empty(B, C, N_MELS, N_FRAMES, pin_memory=True) for _ in range(2)]
    h_lufs = [torch.empty(B, pin_memory=True) for _ in range(2)]
    full_d2h = not args.e2e_features_only

    def e2e_run(n):
        cur = torch.cuda.current_stream()
        for e in freed:
            e.record(cur)
        with torch.cuda.stream(copy_in):
            copy_in.wait_event(freed[0])
            dbuf[0].copy_(hx[0], non_blocking=True)
            ready[0].record(copy_in)
        for i in range(n):
            b = i % 2
            if i + 1 < n:  # prefetch the next batch while this one computes
                with torch.cuda.stream(copy_in):
                    copy_in.wait_event(freed[1 - b])
                    dbuf[1 - b].copy_(hx[(i + 1) % 2], non_blocking=True)
                    ready[1 - b].record(copy_in)
            cur.wait_event(ready[b])
            sig = AudioSignal(dbuf[b], SR)
            sig.normalize(TARGET_DB)
            logmel = sig.mel_spectrogram(n_mels=N_MELS, window_length=N_FFT, hop_length=HOP, window_type="hann",
                                         log=True)
            y = sig.audio_data  # normalised waveform (came out of the same pass)
            lufs = sig._measured_loudness
            assert y.data_ptr() != dbuf[b].data_ptr()
            freed[b].record(cur)
            done[b].record(cur)
            with torch.cuda.stream(copy_out):  # the step's results back to the host (pinned), off the compute stream
                copy_out.wait_event(done[b])
                h_mel[b].copy_(logmel, non_blocking=True)
                h_lufs[b].copy_(lufs, non_blocking=True)
                if full_d2h:
                    h_y[b].copy_(y, non_blocking=True)
                for t_ in (logmel, lufs, y):
                    t_.record_stream(copy_out)
        cur.wait_stream(copy_out)
        return logmel

    e2e_steps = max(3, min(args.steps, 20))
    e2e_run(3)
    barrier()
    w0 = time.perf_counter()
    e2e_run(e2e_steps)
    barrier()
    e2e_s = time.perf_counter() - w0
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * B * e2e_steps / float(te.item())
    if exchange is not None:
        exchange.close()  # collective (barrier inside): all ranks, before the non-zero ranks leave

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel
    peaks_path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    alg_bytes = B * (2 * BYTES_X + BYTES_MEL)  # read x + write y + write log-mel, each once
    achieved = alg_bytes / (spec_ms * 1e-3) / 1e9
    lufs_ms = ms / args.steps - spec_ms
    kernel_name = eng.spectral_kernel_name(N_FFT, HOP) if hasattr(eng, "spectral_kernel_name") else \
        "spectral_warp_kernel<10,0>"
    # DRAM traffic of one launch: from the committed `ncu --set full` capture of THIS kernel at B = 64 (bench.py cannot
    # run under ncu); null when no capture of the kernel in use has been committed
    traffic, traffic_src = None, None
    tpath = os.path.join(REPO, "profiles", "spectral_traffic.json")
    if os.path.exists(tpath):
        rec = json.load(open(tpath)).get(kernel_name.split("<")[0])
        if rec:
            traffic = (rec["dram_bytes_read"] + rec["dram_bytes_write"]) * B / rec["batch"]
            traffic_src = rec["source"]
    roof = {"kernel": kernel_name + " (gain + STFT + |.| + mel + log10, fused)", "bound": "hbm",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": spec_ms,
            "rest_of_step_ms": lufs_ms,
            "rest_of_step": "lufs kernels (read x once: %.0f GB/s algorithmic)" % (B * BYTES_X / max(lufs_ms, 1e-9) / 1e6),
            "whole_step_frac": alg_bytes / (ms / args.steps * 1e-3) / 1e9 / peak}

    # ---- CPU baseline: the oracle port on this box's host cores, rank 0 at N = 1 only, a bounded sample of the same
    #      workload (the full 64-clip batch, 3 reps after a warm-up: ~10-15 s of CPU work)
    cpu = None
    if not args.no_cpu and world == 1:
        n_clips = B
        ts, cores = time_cpu(n_clips, reps=3, warmup=1)
        cpu = {"value": n_clips * len(ts) / sum(ts), "unit": "clips/s", "cores": cores, "kind": "port",
               "sample": f"the full {n_clips}-clip batch per rep, {len(ts)} reps after 1 warm-up; torch threads calibrated "
                         f"over {{all cores, 64, 32, 16, 8}} on 4 clips, fastest used"}

    clk = clocks.summary(w_pre0, w_end)
    clk["window"] = (f"pre-roll {args.preroll:g} s + the {args.steps} timed steps + sustained loop {args.sustain:g} s: one "
                     f"continuous run of the identical step (the timed region alone is {ms:.1f} ms)")
    sorted_ms = sorted(per_rank)
    d2h = B * 4 + B * BYTES_MEL + (B * BYTES_X if full_d2h else 0)
    line = {
        "metric": "clips/sec (10s@44.1kHz) log-mel+LUFS pipeline", "value": value, "unit": "clips/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(world, B),
        "per_rank_ms_per_step": {"min": sorted_ms[0] / args.steps, "median": sorted_ms[len(sorted_ms) // 2] / args.steps,
                                 "max": sorted_ms[-1] / args.steps},
        "roofline": roof, "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": "clips/s", "h2d_bytes_per_step": B * BYTES_X,
                "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                "result_d2h": "log-mel + LUFS" + (" + normalised waveform" if full_d2h else ""),
                "api": "AudioSignal(x).normalize(-24).mel_spectrogram(..., log=True)"},
        "sustained": sus_line, "exchange": exchange_line,
        "gpu_launches": launches, "clocks": clk,
    }
    if dumped is not None:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=64, help="clips per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--preroll", type=float, default=1.0, help="seconds of identical untimed steps before the barrier")
    ap.add_argument("--sustain", type=float, default=2.0, help="seconds of the sustained loop after the timed steps")
    ap.add_argument("--tc", action="store_true", help="use the opt-in tensor-core spectral kernel (A/B measurements)")
    ap.add_argument("--e2e-features-only", action="store_true",
                    help="e2e leg copies back log-mel + LUFS only (not the normalised waveform)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs (rank 0) to DIR/<name>.npy: lufs, loud, gain [B], "
                         "mel (log-mel) and scaled (normalised waveform); an array of more than 2**22 elements as a "
                         "fixed, seeded sample of that many")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps our arm's outputs (--impl ours)")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
