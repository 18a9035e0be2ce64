#!/usr/bin/env python
"""bench.py — spectra/s of the fused window+R2C-FFT+mag+EMA+dBFS path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W          # this repo's CUDA engine (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N ...          # the reference's own CPU path (oracle/_ref), all host cores
  python bench.py ... --dump-outputs DIR                  # also save what the last timed step computed (see dump_outputs)

One "step" = one pass of the hot path over one batch of synthetic 48 kHz PCM already resident in HBM:
65 536 mono frames of N=2048 per GPU, laid out as 4096 independent streams x 16 consecutive frames (hop = N)
so that the EMA recurrence state stays on-chip between frames (DESIGN.md §Measurement).  Inputs (512 MiB)
and outputs (256 MiB) are each larger than the 126 MB L2, so every step streams from/to HBM.

Besides the contract's keys the line carries (DESIGN.md §5):
  parity            the measured launch (same engine geometry, fresh state) against the reference's generic CPU path on a
                    sample of streams: SURVEY.md §8(d) "first 256 frames/shard" + streams from the far ends of the grid
  config.extra      the other layouts of the same 65 536-frame batch (65536x1 ... 256x256) with their roofline fractions, the
                    other BASELINE.json configs / kernel families (other_shapes: N=4096, 8192, 800, 1920, c1, c2, c4, c5, fused display outputs),
                    a strong-scaling number (65 536 frames TOTAL over the N GPUs) and BASELINE.json configs[4]
                    (N=16384, 128 streams x 256 ticks per GPU, NCCL MAX all-reduce + normalise pass inside the timed loop)
  cpu_baseline      all-cores AVX2 (the value) plus AVX2 on one core and the generic path on one core
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "spectra/sec fused window+R2C-FFT+mag+smooth N=2048 batch=65536; %HBM roofline"
UNIT = "spectra/s"
SETTINGS = {"fft_size": 2048, "window": "hann", "temporal_smoothing": "exp_moving_avg", "gravity": 0.65,
            "channel_mode": "mono"}
N_FFT = 2048
BINS = N_FFT // 2
BYTES_PER_FRAME = N_FFT * 4 + BINS * 4  # SURVEY.md §8(d): PCM in + bins out
STATE_BYTES_PER_STREAM = 2 * BINS * 4   # EMA state read + written once per stream and launch (reported separately, §8(d))
LAYOUTS = [(65536, 1), (16384, 4), (8192, 8), (4096, 16), (2048, 32), (1024, 64), (512, 128), (256, 256)]
ALL_CPUS = sorted(os.sched_getaffinity(0))  # the CPUs this process may use, before any NUMA binding


def load_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this same command
    (profiles/traffic.json, written by tools/ncu_summary.py --traffic from the raw CSV next to it); None if absent."""
    p = ROOT / "profiles" / "traffic.json"
    try:
        d = json.loads(p.read_text())
        return float(d["dram_bytes_per_launch"]), d.get("source")
    except Exception:
        return None, None


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation (oracle/_ref), or the oracle port if _ref is absent
# ----------------------------------------------------------------------------------------------------
def cpu_reference_throughput(frames_per_thread: int, threads: int, chunk_frames: int = 512, impl: str = "avx2"):
    """Spectra/s of the reference's CPU path on `threads` host threads, N=2048 Hann EMA dBFS.

    Each thread owns one WAVSource (+ its FFTW plan) and walks `frames_per_thread` consecutive frames
    (hop = N) of its own channel through capture_audio()/tick(); the PCM chunk is reused so it stays in cache,
    which is how the plugin sees audio too.  ctypes releases the GIL, so the threads run in parallel.
    impl: "avx2" = WAVSourceAVX2 (what the plugin runs on this class of CPU), "generic" = WAVSourceGeneric (the parity target).
    """
    import numpy as np

    from oracle import refbind

    kind = "reference"
    if refbind.available():
        which = refbind.IMPL_AVX2 if impl == "avx2" else refbind.IMPL_GENERIC
        mk = lambda: refbind.RefSource(dict(SETTINGS), impl=which, channels=1)
        desc = ("oracle/_ref: WAVSourceAVX2::tick_spectrum" if impl == "avx2" else "oracle/_ref: WAVSourceGeneric::tick_spectrum") \
            + " + vendored FFTW 3.3.11 (AVX2 codelets)"
    else:
        from oracle import oraclebind
        kind = "port"
        mk = lambda: oraclebind.OracleSource(dict(SETTINGS), channels=1)
        desc = "oracle/liboracle.so: scalar C restatement of source_generic.cpp"
    rng = np.random.default_rng(0xB200)
    srcs = [mk() for _ in range(threads)]
    pcms = [(0.25 * rng.uniform(-1, 1, (1, (chunk_frames + 1) * N_FFT))).astype(np.float32) for _ in range(threads)]
    reps = max(1, frames_per_thread // chunk_frames)

    def work(i):
        for _ in range(reps):
            srcs[i].run_stft(pcms[i], chunk_frames, N_FFT, want_db=False)

    # warm-up (page in, FFTW plan, caches)
    for i in range(threads):
        srcs[i].run_stft(pcms[i], 8, N_FFT, want_db=False)
    ts = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    t0 = time.perf_counter()
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    dt = time.perf_counter() - t0
    frames = threads * reps * chunk_frames
    return frames / dt, {"kind": kind, "cores": threads, "desc": desc, "frames": frames, "seconds": dt}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = len(ALL_CPUS)
    per_thread = 8192
    vals = []
    for _ in range(args.warmup):
        cpu_reference_throughput(1024, cores)
    info = None
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v, info = cpu_reference_throughput(per_thread, cores)
        vals.append(v)
    dt = time.perf_counter() - t0
    value = statistics.median(vals)
    frames_per_step = info["frames"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(), "fft_size": N_FFT, "frames_per_step": frames_per_step,
                   "note": "CPU arm: bounded sample of the same workload per step, all host threads"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": info["cores"], "kind": info["kind"],
                         "sample": f"{frames_per_step} frames/step ({info['desc']}), hop=N, data cache-resident",
                         "affinity_cpus": cores, "os_cpu_count": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_id: str):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", gpu_id], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def wait_first(self, timeout=3.0):
        t0 = time.perf_counter()
        while self.proc and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def stop(self, t_begin, t_end):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        # nvidia-smi stamps a sample up to one period after the state it shows; take the samples around the timed region
        rows = [r for (t, r) in self.rows if t_begin <= t <= t_end + 0.05] or \
               [r for (t, r) in self.rows if t_begin - 0.1 <= t <= t_end + 0.15] or [r for (_, r) in self.rows]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def workload_name():
    return ("c3: 65536 mono frames/GPU, N=2048 Hann, EMA g=0.65, dBFS; 4096 streams x 16 consecutive frames, hop=N "
            "(BASELINE.json configs[2])")


def make_pcm_on_device(torch, S, T, device, seed):
    """SURVEY.md §8(d) synthetic signal, generated on the device: noise + two sines per stream, 1% all-zero frames."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    ns = T * N_FFT
    n = torch.arange(ns, device=device, dtype=torch.float32)
    c = torch.arange(S, device=device, dtype=torch.float32)
    fc = 110.0 * torch.pow(2.0, torch.remainder(c, 60.0) / 12.0)
    pcm = torch.empty((S, 1, ns), device=device, dtype=torch.float32)
    chunk = max(1, (1 << 24) // ns)
    for s0 in range(0, S, chunk):
        s1 = min(S, s0 + chunk)
        ph = 2.0 * torch.pi * fc[s0:s1, None] * n[None, :] / 48000.0
        x = 0.25 * (2.0 * torch.rand((s1 - s0, ns), device=device, generator=g) - 1.0)
        x += 0.5 * torch.sin(ph) + 0.1 * torch.sin(3.01 * ph)
        pcm[s0:s1, 0] = x
    zero = torch.rand((S, T), device=device, generator=g) < 0.01
    pcm.view(S, T, N_FFT)[zero] = 0.0
    return pcm


def time_steps(torch, stream, step, steps, warmup):
    """CUDA-event time per step (ms) of `step()` launched on `stream`: list of per-step times."""
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    evs[0].record(stream)
    for k in range(steps):
        step()
        evs[k + 1].record(stream)
    torch.cuda.synchronize()
    return [evs[k].elapsed_time(evs[k + 1]) for k in range(steps)]


DUMP_BYTES = 48 << 20  # all ranks together: a dump stays well under 64 MB, so two builds can be compared output for output


def dump_outputs(torch, out_dir, out, rank, world):
    """Save the dB spectra the last timed step wrote ([streams, frames, 1, bins] float32) as db.npy, and the indices of the
    streams saved as db_streams.npy (float64).  Each rank gets DUMP_BYTES / world; when its output is larger, a fixed seeded
    sample of streams is saved, so the same arguments always select the same streams.  Ranks other than 0 add a _rank<r>
    suffix."""
    import numpy as np

    S = out.shape[0]
    n = min(S, max(1, DUMP_BYTES // world // (out[0].numel() * out.element_size())))
    idx = np.arange(S) if n == S else np.sort(np.random.default_rng(0xB200).choice(S, n, replace=False))
    sel = out.index_select(0, torch.as_tensor(idx, device=out.device)).cpu().numpy()
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    sfx = "" if rank == 0 else f"_rank{rank}"
    np.save(d / f"db{sfx}.npy", sel)
    np.save(d / f"db_streams{sfx}.npy", idx.astype(np.float64))


def parity_subset(torch, device, pcm, S, T):
    """SURVEY §8(d): run the MEASURED launch geometry once from a fresh state and compare the first 256 frames of the
    shard plus streams from the far ends of the grid with the reference's generic CPU path (oracle/_ref; the C port if
    the compiled reference is absent).  Criterion = tests/helpers.py::parity_report (DESIGN.md §2)."""
    import numpy as np

    sys.path.insert(0, str(ROOT / "tests"))
    from helpers import parity_report
    from oracle import refbind
    from waveform_b200 import Engine

    eng = Engine(dict(SETTINGS), channels=1, max_streams=S, device=device.index)
    out = eng.process(pcm, T, N_FFT)
    torch.cuda.synchronize()
    kernel = eng.last_kernel_name()
    n_first = max(1, min(S, -(-256 // T)))
    pick = sorted(set(range(n_first)) | {S - 1, S - 2, S // 2, S // 3, 147 % S, 148 % S, (148 * 16) % S, (148 * 16 + 147) % S,
                                         (148 * 27) % S} | set(range(0, S, max(1, S // 40))))
    idx = torch.tensor(pick, device=device)
    got = out["db"][idx].cpu().numpy()
    got_sil = out["silent"][idx].cpu().numpy()
    rows = pcm[idx].cpu().numpy()
    if refbind.available():
        mk = lambda: refbind.RefSource(dict(SETTINGS), impl=refbind.IMPL_GENERIC, channels=1)
        against = "oracle/_ref WAVSourceGeneric::tick_spectrum (the unmodified reference, compiled)"
    else:
        from oracle import oraclebind
        mk = lambda: oraclebind.OracleSource(dict(SETTINGS), channels=1)
        against = "oracle/liboracle.so (C restatement of source_generic.cpp)"
    ref, ref_sil = [], []
    for r in rows:
        o = mk().run_stft(r, T, N_FFT)
        ref.append(o["db"])
        ref_sil.append(o["silent"])
    ref, ref_sil = np.stack(ref), np.stack(ref_sil)
    rep = parity_report(got, ref, db_min=eng.db_min)
    return {"ok": bool(rep["ok"] and rep["normwise"] < 1e-6 and np.array_equal(got_sil, ref_sil)),
            "streams_checked": len(pick), "frames_checked": len(pick) * T, "normwise": rep["normwise"],
            "frac_bins_within_1e-5_rel": rep["frac_rel_1e5"], "max_db_err_strong_bins": rep["max_db_strong"],
            "silent_flags_equal": bool(np.array_equal(got_sil, ref_sil)), "silent_ticks_in_sample": int(ref_sil.sum()),
            "kernel": kernel, "against": against,
            "criterion": "|gpu-ref| <= 1e-5|ref| + 1e-6 frame_peak (linear), normwise < 1e-6, identical DB_MIN pattern and silent flags"}


def run_layouts(torch, device, stream, peak_gbs, steps):
    """The same 65 536-frame batch in every streams x frames factorisation of SURVEY §8(d) C3."""
    from waveform_b200 import Engine

    res = []
    out = torch.empty((65536, 1, BINS), device=device, dtype=torch.float32)
    for (S, T) in LAYOUTS:
        eng = Engine(dict(SETTINGS), channels=1, max_streams=S, device=device.index)
        pcm = make_pcm_on_device(torch, S, T, device, seed=0xB200)
        step = lambda: eng.process_raw(pcm.data_ptr(), S, T, N_FFT, T * N_FFT, T * N_FFT, out_db=out.data_ptr(),
                                       stream=stream.cuda_stream, sync=False)
        ms = statistics.mean(time_steps(torch, stream, step, steps, 3))
        gbs = 65536 * BYTES_PER_FRAME / (ms * 1e-3) / 1e9
        with_state = (65536 * BYTES_PER_FRAME + S * STATE_BYTES_PER_STREAM) / (ms * 1e-3) / 1e9
        res.append({"streams": S, "frames": T, "value": 65536 / (ms * 1e-3), "kernel_ms": ms, "frac": gbs / peak_gbs,
                    "frac_incl_state_bytes": with_state / peak_gbs, "kernel": eng.last_kernel_name()})
        del eng, pcm
    return res


def run_c5(torch, dist, device, world, steps):
    """BASELINE.json configs[4]: N=16384, 128 streams x 256 ticks per GPU (262 144 frames over 8 GPUs), cross-GPU peak
    normalisation: kernel (with the per-tick peak) -> NCCL all_reduce(MAX) of 256 floats -> normalise pass, all inside the
    timed loop and on one stream.  Value = frames of all ranks / max-over-ranks device time."""
    from waveform_b200 import Engine
    from waveform_b200.shard import ShardedEngine

    N, S, T = 16384, 128, 256
    eng = Engine({"fft_size": N, "window": "hann"}, channels=1, max_streams=S, device=device.index)
    sh = ShardedEngine(eng)
    g = torch.Generator(device=device)
    g.manual_seed(0xC5 + int(os.environ.get("RANK", "0")))
    pcm = (torch.rand((S, 1, T * N), device=device, generator=g) - 0.5) * (0.1 + 0.05 * int(os.environ.get("RANK", "0")))
    # correctness of the exchange on the measured shape: all-reduced peak == max of the local peaks, output == local + gain
    plain = eng.process(pcm, T, N, want_peak=True)
    local_peak = plain["peak"].clone()
    local_db = plain["db"].clone()
    del plain
    eng2 = Engine({"fft_size": N, "window": "hann"}, channels=1, max_streams=S, device=device.index)
    out = ShardedEngine(eng2).process_normalized(pcm, T, N, target_db=-3.0, max_gain=30.0)
    if world > 1:
        allp = [torch.empty_like(local_peak) for _ in range(world)]
        dist.all_gather(allp, local_peak)
        want = torch.stack(allp).max(dim=0).values
    else:
        want = local_peak
    gain = torch.clamp(-3.0 - want, max=30.0)
    local_db[..., 1:] += gain[None, :, None, None]
    ok = bool(torch.equal(out["peak"], want) and torch.equal(out["db"], local_db))
    del out, local_db, eng2
    torch.cuda.empty_cache()
    for _ in range(2):
        sh.process_normalized(pcm, T, N)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        sh.process_normalized(pcm, T, N)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / steps], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    frames = S * T * world
    bytes_per_frame = N * 4 + (N // 2) * 4
    return {"workload": f"c5: N=16384 Hann, {S} streams x {T} ticks per GPU ({frames} frames total), per-tick peak -> "
                        f"{'NCCL all_reduce(MAX) of ' + str(T) + ' floats' if world > 1 else 'no exchange (1 GPU)'} -> normalise pass",
            "value": frames / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
            "frac_per_gpu": (S * T * bytes_per_frame / (ms * 1e-3) / 1e9) / load_peaks()[0],
            "exchange_exact": ok, "kernel": eng.last_kernel_name()}


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    from waveform_b200 import Engine
    from waveform_b200.hostbind import bind_to_gpu_node

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    # NUMA: pin this rank to its GPU's node BEFORE any pinned buffer exists (first touch decides where the pages live)
    numa = bind_to_gpu_node(local_rank) if not args.no_numa_bind else {"bound": False, "why": "--no-numa-bind"}
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    S, T = args.streams, args.frames
    frames_per_gpu = S * T
    eng = Engine(dict(SETTINGS), channels=1, max_streams=S, device=local_rank)
    pcm = make_pcm_on_device(torch, S, T, device, seed=0xB200 + rank)
    out = torch.empty((S, T, 1, BINS), device=device, dtype=torch.float32)
    stream = torch.cuda.Stream(device=device)  # a real (non-default) stream: timed events and launches share it
    torch.cuda.synchronize()

    def step():
        eng.process_raw(pcm.data_ptr(), S, T, N_FFT, T * N_FFT, T * N_FFT, out_db=out.data_ptr(),
                        stream=stream.cuda_stream, sync=False)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    props = torch.cuda.get_device_properties(device)
    gpu_id = "GPU-" + str(props.uuid) if hasattr(props, "uuid") else str(local_rank)
    sampler = ClockSampler(gpu_id) if rank == 0 else None
    if sampler:
        sampler.wait_first()
    for _ in range(max(3, args.warmup)):
        step()
    barrier()
    launches0 = eng.launch_count
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    t_begin = time.perf_counter()
    evs[0].record(stream)
    for k in range(args.steps):
        step()
        evs[k + 1].record(stream)
    torch.cuda.synchronize()
    t_end = time.perf_counter()
    launches = eng.launch_count - launches0
    kernel_name = eng.last_kernel_name()
    total_ms = evs[0].elapsed_time(evs[-1])
    per_launch = [evs[k].elapsed_time(evs[k + 1]) for k in range(args.steps)]
    clocks = sampler.stop(t_begin, t_end) if sampler else None
    if args.dump_outputs:
        dump_outputs(torch, args.dump_outputs, out, rank, world)
    ms_per_step = max_over_ranks(total_ms) / args.steps
    value = frames_per_gpu * world / (ms_per_step * 1e-3)

    # ---- strong scaling: the literal "batch = 65536" split over the N GPUs (4096/N streams x 16 frames per GPU) ----
    strong = None
    if world > 1:
        Ss = max(1, S // world)
        steps_s = min(args.steps, 50)
        step_s = lambda: eng.process_raw(pcm.data_ptr(), Ss, T, N_FFT, T * N_FFT, T * N_FFT, out_db=out.data_ptr(),
                                         stream=stream.cuda_stream, sync=False)
        for _ in range(3):
            step_s()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps_s):
            step_s()
        e1.record(stream)
        torch.cuda.synchronize()
        ms_s = max_over_ranks(e0.elapsed_time(e1)) / steps_s
        strong = {"value": Ss * T * world / (ms_s * 1e-3), "unit": UNIT, "frames_total": Ss * T * world,
                  "streams_per_gpu": Ss, "ms_per_step": ms_s, "scaling": "strong",
                  "note": "65 536 frames TOTAL per step; per-GPU launches shrink with N (launch-latency territory at N=8)"}

    # ---- end-to-end: host (pinned) buffers through the C-ABI, H2D + kernel + D2H inside the timed region ----
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    h_pcm = torch.empty((S, 1, T * N_FFT), dtype=torch.float32, pin_memory=True)
    h_pcm.copy_(pcm)
    h_out = torch.empty((S, T, 1, BINS), dtype=torch.float32, pin_memory=True)

    def step_e2e():
        eng.process_raw(h_pcm.data_ptr(), S, T, N_FFT, T * N_FFT, T * N_FFT, out_db=h_out.data_ptr(),
                        stream=stream.cuda_stream, sync=False)

    # the host ceiling of this rank, measured: a bare pinned H2D copy of the same bytes (no kernel, no D2H)
    d_probe = torch.empty_like(pcm)
    with torch.cuda.stream(stream):
        d_probe.copy_(h_pcm, non_blocking=True)
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record(stream)
    with torch.cuda.stream(stream):
        for _ in range(3):
            d_probe.copy_(h_pcm, non_blocking=True)
    c1.record(stream)
    torch.cuda.synchronize()
    h2d_gbs_alone = 3 * h_pcm.numel() * 4 / (c0.elapsed_time(c1) * 1e-3) / 1e9
    del d_probe

    step_e2e()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(e2e_steps):
        step_e2e()
    e1.record(stream)
    torch.cuda.synchronize()
    e2e_rank_ms = e0.elapsed_time(e1) / e2e_steps
    e2e_ms = max_over_ranks(e2e_rank_ms)
    e2e_value = frames_per_gpu * world / (e2e_ms * 1e-3)
    checksum = float(h_out[:: max(1, S // 64)].double().sum())  # host read of the step's result
    h2d_rank = torch.tensor([h_pcm.numel() * 4 / (e2e_rank_ms * 1e-3) / 1e9, h2d_gbs_alone], device=device, dtype=torch.float64)
    if world > 1:
        allr = [torch.empty_like(h2d_rank) for _ in range(world)]
        dist.all_gather(allr, h2d_rank)
        h2d_all = torch.stack(allr).cpu().tolist()
        numa_all = [None] * world
        dist.all_gather_object(numa_all, numa)
    else:
        h2d_all, numa_all = [h2d_rank.cpu().tolist()], [numa]
    del h_pcm, h_out

    # ---- parity of the measured launch geometry (after the timed regions) ----
    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_subset(torch, device, pcm, S, T)

    # ---- config 5 with its collective (every N; N=1 has no exchange) ----
    c5 = None
    if not args.no_c5:
        del out
        torch.cuda.empty_cache()
        c5 = run_c5(torch, dist, device, world, steps=5)
        out = torch.empty((S, T, 1, BINS), device=device, dtype=torch.float32)

    if rank == 0:
        peak_gbs, peak_src = load_peaks()
        traffic, traffic_src = load_traffic() if (S, T) == (4096, 16) else (None, None)
        kernel_ms = statistics.mean(per_launch)
        achieved = frames_per_gpu * BYTES_PER_FRAME / (kernel_ms * 1e-3) / 1e9
        layouts, other = None, None
        if world == 1 and not args.no_layouts:
            layouts = run_layouts(torch, device, stream, peak_gbs, steps=20)
            sys.path.insert(0, str(ROOT / "tools"))
            from bench_shapes import run_shapes
            other = run_shapes(torch, iters=5, peak_gbs=peak_gbs)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, ALL_CPUS)  # the CPU arm uses every core the box grants, not just the GPU's NUMA node
            cores = len(ALL_CPUS)
            v, info = cpu_reference_throughput(args.cpu_frames_per_thread, cores)
            v1, i1 = cpu_reference_throughput(32768, 1)
            vg, ig = cpu_reference_throughput(16384, 1, impl="generic")
            cpu = {"value": v, "unit": UNIT, "cores": info["cores"], "kind": info["kind"],
                   "sample": f"{info['frames']} frames in {info['seconds']:.2f}s wall ({info['desc']}), hop=N, "
                             "same N=2048 Hann EMA dBFS settings, data cache-resident",
                   "affinity_cpus": cores, "os_cpu_count": os.cpu_count(),
                   "avx2_1core": {"value": v1, "unit": UNIT, "cores": 1, "sample": f"{i1['frames']} frames in {i1['seconds']:.2f}s"},
                   "generic_1core": {"value": vg, "unit": UNIT, "cores": 1,
                                     "sample": f"{ig['frames']} frames in {ig['seconds']:.2f}s ({ig['desc']}; the parity target)"}}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(), "fft_size": N_FFT, "streams_per_gpu": S, "frames_per_stream": T,
                       "hop": N_FFT, "frames_per_step_per_gpu": frames_per_gpu,
                       "l2_policy": "inputs 512 MiB + outputs 256 MiB per step exceed the 126 MB L2 (no flush needed)",
                       "parallelism": f"streams sharded over {world} GPU(s), no data-path collective",
                       "extra": {"layouts_same_batch": layouts, "strong_scaling": strong, "c5": c5, "other_shapes": other}},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(S * T * N_FFT * 4),
                    "d2h_bytes_per_step": int(S * T * BINS * 4), "steps": e2e_steps, "checksum": checksum,
                    "per_gpu_h2d_gbs_in_e2e": [round(r[0], 2) for r in h2d_all],
                    "per_gpu_h2d_gbs_copy_alone": [round(r[1], 2) for r in h2d_all],
                    "numa_binding": numa_all},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                         "frac": achieved / peak_gbs, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src, "kernel": kernel_name, "kernel_ms": kernel_ms,
                         "bytes_per_launch": frames_per_gpu * BYTES_PER_FRAME},
            "parity": parity,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=4096, help="independent streams per GPU")
    ap.add_argument("--frames", type=int, default=16, help="consecutive frames per stream")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-frames-per-thread", type=int, default=16384)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-layouts", action="store_true")
    ap.add_argument("--no-c5", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="save the spectra of the last timed step as .npy files in DIR")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs saves the GPU path's spectra; the reference arm only measures throughput")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
