#!/usr/bin/env python
"""bench.py -- headline benchmark: Msamples/s of the Complex<f32> 256-tap FIR on 64 Mi-sample
chunks (BASELINE.json configs[1]) at N GPUs, with the HBM roofline fraction of the dominant
kernel and the reference's CPU path timed beside it; the other BASELINE configs ride along in a
`secondary` array of the same JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the FIR over one 64 Mi-sample chunk per GPU, taken from a device-resident
ring (b2s_ring_*).  Weak scaling: each rank owns the next contiguous chunk of ONE logical stream;
the only exchange is the 255-sample overlap region, which the FIR kernel's TMA loader reads from
the left neighbour's ring over NVLink (CUDA-IPC peer mapping + two device counters per ring;
futuresdr_b200/shard.py) -- `--exchange nccl` times the NCCL all-gather variant instead.
Prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NTAPS = 256
CHUNK = 64 * 1024 * 1024          # samples per GPU per step (BASELINE configs[1])
BYTES_PER_SAMPLE = 16             # 8 B in + 8 B out (BASELINE.md §3; taps/halo amortise to 0)
SEED = 0x5EED
FALLBACK_HBM_GBS = 6650.0         # /opt/skills/guides/B200_PROFILING.md fallback


def _peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        d = json.load(open(p))
        for k in ("hbm_gbs", "hbm_gb_s", "hbm_GBs"):
            if k in d:
                return float(d[k]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _taps(n=NTAPS, seed=7):
    return np.random.default_rng(seed).uniform(-1, 1, n).astype(np.float32)


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (NVML polled every ~2 ms from a
    background thread; falls back to one nvidia-smi query if NVML is unavailable)."""

    def __init__(self, index=0):
        self.index, self.thread, self.stop_flag = index, None, False
        self.sm, self.reasons, self.max_sm = [], set(), None

    def _poll(self):
        import pynvml as nv
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
        }
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = get_reasons(h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None

    def stop(self):
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(1.0)
        if self.sm:
            return {"sm_mhz": statistics.median(self.sm), "sm_max_mhz": self.max_sm,
                    "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}
        try:   # fallback: a single nvidia-smi reading right after the region
            q = "clocks.sm,clocks.max.sm"
            o = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                str(self.index)], capture_output=True, text=True, timeout=10).stdout.split(",")
            return {"sm_mhz": float(o[0]), "sm_max_mhz": float(o[1]), "reasons": [], "samples": 1,
                    "source": "nvidia-smi after region"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}


# ------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path (oracle port of
# crates/futuredsp/src/fir.rs:52-91; the Rust cannot be compiled here), all host threads.
# ------------------------------------------------------------------------------------------
_CPU_THREADS = None


def _cpu_threads():
    """Thread count for the CPU legs: all the host threads this process may use.  OpenMP's default
    can exceed the container's CPU allowance (oversubscription made the 128-thread run 8x slower
    than the 64-thread one), so a few candidates are timed on a small sample and the best is kept."""
    global _CPU_THREADS
    if _CPU_THREADS is not None:
        return _CPU_THREADS
    import oracle as orc
    cand = {orc.max_threads()}
    try:
        cand.add(len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            cand.add(max(1, int(int(q[0]) / int(q[1]))))
    except Exception:
        pass
    m = max(cand)
    cand |= {max(1, m // 2), max(1, m // 4), min(m, 32), min(m, 16)}
    rng = np.random.default_rng(1)
    n = 1 << 22
    x = (rng.standard_normal(n + NTAPS - 1) + 1j * rng.standard_normal(n + NTAPS - 1)).astype(np.complex64)
    out = np.zeros(n, np.complex64)
    taps = _taps()
    best, best_t = None, None
    for th in sorted(cand):
        dt = None
        for _ in range(3):                      # first pass warms the thread pool; keep the best
            t0 = time.perf_counter()
            orc.fir_c32_f32_mt(taps, x, th, fast=True, out=out)
            d1 = time.perf_counter() - t0
            dt = d1 if dt is None else min(dt, d1)
        if best_t is None or dt < best_t:
            best, best_t = th, dt
    _CPU_THREADS = best
    return best


_CPU_NOISE = {}


def _cpu_noise(n):
    """White noise for the CPU legs (generated once per size: 64 Mi complex samples take seconds in numpy)."""
    if n not in _CPU_NOISE:
        rng = np.random.default_rng(SEED)
        x = np.empty(n, np.complex64)
        v = x.view(np.float32)
        blk = 1 << 24
        for i in range(0, v.size, blk):
            v[i:i + blk] = rng.standard_normal(min(blk, v.size - i), dtype=np.float32)
        _CPU_NOISE.clear()
        _CPU_NOISE[n] = x
    return _CPU_NOISE[n]


_CPU_OUT = {}


def _cpu_out(n):
    if n not in _CPU_OUT:
        _CPU_OUT.clear()
        _CPU_OUT[n] = np.zeros(n, np.complex64)
    return _CPU_OUT[n]


def cpu_fir(sample_items: int, reps: int = 1, ntaps: int = NTAPS, variants=(False, True)):
    """The reference's FIR loop (oracle port of fir.rs:52-91) on all host threads over contiguous shards; both the
    stable strict-order loop and the nightly re-associated (-ffast-math) one, the faster is reported."""
    import oracle as orc
    threads = _cpu_threads()
    x = _cpu_noise(sample_items + ntaps - 1)
    taps = _taps(ntaps)
    out = _cpu_out(sample_items)                  # touched once: no page faults inside the timed calls
    best = {}
    for fast in variants:
        orc.fir_c32_f32_mt(taps, x[: 65536 + ntaps - 1], threads, fast=fast)     # warm
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            orc.fir_c32_f32_mt(taps, x, threads, fast=fast, out=out)
            ts.append(time.perf_counter() - t0)
        best["nightly_reassoc" if fast else "stable_strict"] = min(ts)
    variant = min(best, key=best.get)
    return {"seconds": best[variant], "variant": variant, "threads": threads, "all": best,
            "msps": sample_items / best[variant] / 1e6}


def run_reference(args):
    """Reference arm: the SAME workload as our arm (one 64 Mi-sample chunk of the 256-tap c32 FIR per step), computed
    by the reference's CPU loop on every host thread.  The strict-order variant is timed once (it is ~4x slower),
    the faster re-associated one every step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = CHUNK
    strict = cpu_fir(n, reps=1, variants=(False,))
    times, last = [], None
    for i in range(args.warmup + args.steps):
        r = cpu_fir(n, reps=1, variants=(True,))
        last = r
        if i >= args.warmup:
            times.append(r["seconds"])
    sec = statistics.mean(times)
    v = n / sec / 1e6
    line = {
        "impl": "reference", "metric": "Msamples/s", "value": v, "unit": "Msamples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic white noise",
        "config": {"workload": "single-B200 Complex<f32> 256-tap FIR on 64 Mi-sample chunks via device-resident ring (BASELINE configs[1])",
                   "ntaps": NTAPS, "chunk_items": CHUNK,
                   "note": "the reference's CPU loop on the same chunk; host arm, no device, no ring"},
        "cpu_baseline": {"value": v, "unit": "Msamples/s", "cores": last["threads"], "kind": "port",
                         "sample": f"{n} samples/step (the full chunk), oracle port of futuredsp fir.rs:52-91 "
                                   f"(nightly re-associated loop; the stable strict-order loop runs at "
                                   f"{strict['msps']:.1f} Msamples/s), {last['threads']} OpenMP threads over contiguous shards"},
        "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
# helpers for our arm
# ------------------------------------------------------------------------------------------
def _events(torch, n):
    return [torch.cuda.Event(enable_timing=True) for _ in range(n)]


def _time_passes(torch, fn, reps, warm=1):
    """mean seconds of fn() over `reps` passes, CUDA events on the current stream, synchronize both sides"""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e = _events(torch, 2)
    e[0].record()
    for _ in range(reps):
        fn()
    e[1].record()
    torch.cuda.synchronize()
    return e[0].elapsed_time(e[1]) * 1e-3 / reps


DUMP_HEAD = 4096                  # --dump-outputs keeps the first outputs (their window reaches into the history) ...
DUMP_SAMPLES = 1 << 20            # ... and a seeded sample of the rest: 8 MiB of values, 8 MiB of indices


def dump_outputs(path, out, consumed, produced, status):
    """Writes what the last timed step returned to its caller, so that two builds can be compared output for output:
    fir_counts.npy = (consumed, produced, status), fir_out.npy = (re, im) float32 of the outputs at fir_out_index.npy.
    The indices are the same in every run (all 64 Mi outputs would be 512 MiB)."""
    import torch
    os.makedirs(path, exist_ok=True)
    pick = np.random.default_rng(SEED).choice(produced, size=min(produced, DUMP_SAMPLES), replace=False)
    idx = np.union1d(np.arange(min(produced, DUMP_HEAD)), pick)
    vals = torch.view_as_real(out[:produced].index_select(0, torch.from_numpy(idx).to(out.device)))
    np.save(os.path.join(path, "fir_counts.npy"), np.array([consumed, produced, int(status)], np.float64))
    np.save(os.path.join(path, "fir_out_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(path, "fir_out.npy"), vals.cpu().numpy())


def _roofline(alg_bytes, sec, note=None):
    peak, src = _peak_hbm()
    ach = alg_bytes / sec / 1e9
    r = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
         "peak_source": src, "algorithmic_bytes": alg_bytes}
    if note:
        r["note"] = note
    return r


def host_copy_ceiling(torch, dev, h_in, h_out, reps=5):
    """What the host side can deliver: concurrent H2D + D2H of the e2e buffers with plain async copies on two
    streams (no kernel).  The e2e figure cannot exceed min(h2d, d2h) / 8 B per sample."""
    d_a = torch.empty_like(h_in, device=dev)
    d_b = torch.empty_like(h_out, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    torch.cuda.synchronize()
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        with torch.cuda.stream(s1):
            d_a.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_b, non_blocking=True)
        s1.synchronize(); s2.synchronize()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    gbs_in = h_in.numel() * h_in.element_size() / best / 1e9
    gbs_out = h_out.numel() * h_out.element_size() / best / 1e9
    return {"h2d_GBs": gbs_in, "d2h_GBs": gbs_out, "concurrent": True,
            "ceiling_Msamples_s": min(gbs_in, gbs_out) * 1e9 / 8 / 1e6}


class HostPipe:
    """Generic end-to-end leg for the secondary configs: pinned host input -> H2D (side stream) -> device work on the
    current stream -> D2H (side stream) into pinned host output, chunk by chunk over two device slots, so copies of
    chunk k+1 / k-1 overlap the work on chunk k.  `work(d_in, n_in_items, d_out) -> n_out_items` queues the device
    work of one chunk (blocks keep their own state); d_in has `halo` items of the previous chunk in front."""

    def __init__(self, torch, dev, in_dtype, out_dtype, chunk_items, out_cap_items, halo=0):
        self.t, self.dev = torch, dev
        self.chunk, self.halo, self.out_cap = chunk_items, halo, out_cap_items
        self.d_in = [torch.empty(halo + chunk_items, dtype=in_dtype, device=dev) for _ in range(2)]
        self.d_out = [torch.empty(out_cap_items, dtype=out_dtype, device=dev) for _ in range(2)]
        self.s_in, self.s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def run(self, h_in, h_out, work):
        t = self.t
        main = t.cuda.current_stream(self.dev)
        n = h_in.numel()
        nchunks = (n + self.chunk - 1) // self.chunk
        ev_in = [t.cuda.Event() for _ in range(2)]
        ev_k = [t.cuda.Event() for _ in range(2)]
        ev_out = [t.cuda.Event() for _ in range(2)]
        produced = 0
        for c in range(nchunks):
            s = c & 1
            lo, hi = c * self.chunk, min(n, (c + 1) * self.chunk)
            with t.cuda.stream(self.s_in):
                if c >= 2:
                    self.s_in.wait_event(ev_k[s])              # slot's previous chunk has been consumed
                self.d_in[s][self.halo:self.halo + hi - lo].copy_(h_in[lo:hi], non_blocking=True)
                ev_in[s].record(self.s_in)
            main.wait_event(ev_in[s])
            if c >= 2:
                main.wait_event(ev_out[s])                     # slot's previous output has left
            if self.halo and c:
                prev = self.d_in[s ^ 1]
                self.d_in[s][:self.halo].copy_(prev[self.chunk:self.chunk + self.halo])
            first = self.halo if c == 0 else 0                 # the first chunk of a stream has no history
            n_out = work(self.d_in[s][first:self.halo + hi - lo], self.d_out[s])
            ev_k[s].record(main)
            with t.cuda.stream(self.s_out):
                self.s_out.wait_event(ev_k[s])
                h_out[produced:produced + n_out].copy_(self.d_out[s][:n_out], non_blocking=True)
                ev_out[s].record(self.s_out)
            produced += n_out
        self.s_out.synchronize()
        main.synchronize()
        return produced

    def timed(self, h_in, h_out, work, reset, reps=2):
        reset()
        self.run(h_in, h_out, work)                            # warm (also faults the pinned pages in)
        best = None
        for _ in range(reps):
            reset()
            self.t.cuda.synchronize()
            t0 = time.perf_counter()
            p = self.run(h_in, h_out, work)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        return best, p


# ------------------------------------------------------------------------------------------
# secondary configs (BASELINE.json configs[0], [2], [3], [4])
# ------------------------------------------------------------------------------------------
def sec_config1_perf_fir(torch, fb, dev, args):
    """configs[0] `perf/fir` (perf/fir/fir.rs:40-109): `pipes` x `stages` 64-tap f32 FIRs on 1 M samples.  CPU arm =
    the reference's loop (one thread per pipe = the smoln scheduler's best case); GPU = the same pipes x stages chain
    of FirFilter calls on device-resident buffers (launch-bound at this size, which is the point of the config)."""
    import oracle as orc
    from concurrent.futures import ThreadPoolExecutor
    pipes, stages, n, ntaps = 5, 6, 1_000_000, 64
    taps = np.random.default_rng(2).random(ntaps).astype(np.float32)          # rand::random::<f32>() = U[0,1)
    x = np.random.default_rng(1).uniform(-1, 1, n).astype(np.float32)

    def cpu_pipe(_):
        cur = x
        for _s in range(stages):
            _, p, _, cur = orc.fir(taps, cur, cur.size)
        return cur.size
    with ThreadPoolExecutor(pipes) as ex:
        list(ex.map(cpu_pipe, range(pipes)))
        t0 = time.perf_counter()
        outs = list(ex.map(cpu_pipe, range(pipes)))
        cpu_s = time.perf_counter() - t0
    assert all(o == n - stages * (ntaps - 1) for o in outs)                   # fir.rs:94-98
    fir = fb.FirFilter(taps, sample_dtype=np.float32)
    xd = torch.from_numpy(x).to(dev)
    bufs = [torch.empty(n, dtype=torch.float32, device=dev) for _ in range(2)]
    got = []

    def gpu_pass():
        got.clear()
        for _p in range(pipes):
            cur, m = xd, n
            for s in range(stages):
                c, p, st = fir.filter(cur[:m], bufs[s & 1])
                cur, m = bufs[s & 1], p
            got.append(m)
    sec = _time_passes(torch, gpu_pass, reps=10, warm=2)
    assert all(m == n - stages * (ntaps - 1) for m in got)
    # the same 30 launches captured ONCE in a CUDA graph and replayed (launch-bound inner loops belong in graphs):
    # a context on a dedicated stream, the plan created before capture, the pass captured on that stream
    graph_sec = None
    par_sec = None
    try:
        gs = torch.cuda.Stream(dev)
        with torch.cuda.stream(gs):
            gctx = fb.Context(dev.index, stream=gs.cuda_stream)
            gfir = fb.FirFilter(taps, sample_dtype=np.float32, ctx=gctx)

            def graph_body():
                for _p in range(pipes):
                    cur, m = xd, n
                    for s_ in range(stages):
                        c, p, st = gfir.filter(cur[:m], bufs[s_ & 1])
                        cur, m = bufs[s_ & 1], p

            def replay_time(body):
                body()
                gs.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=gs):
                    body()
                for _ in range(3):
                    g.replay()
                gs.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(gs)
                for _ in range(20):
                    g.replay()
                e1.record(gs)
                gs.synchronize()
                return e0.elapsed_time(e1) * 1e-3 / 20
            graph_sec = replay_time(graph_body)
            # the pipes are independent flowgraph branches (perf/fir/fir.rs:60-86 connects `pipes` separate chains): one
            # stream, one context and one pair of buffers per pipe, forked from / joined to the capturing stream, so the
            # graph holds `pipes` parallel chains of `stages` kernels
            pstreams = [torch.cuda.Stream(dev) for _ in range(pipes)]
            pctx = [fb.Context(dev.index, stream=ps.cuda_stream) for ps in pstreams]
            pfir = [fb.FirFilter(taps, sample_dtype=np.float32, ctx=c) for c in pctx]
            pbufs = [[torch.empty(n, dtype=torch.float32, device=dev) for _ in range(2)] for _ in range(pipes)]
            pgot = [0] * pipes

            def parallel_body():
                for i in range(pipes):
                    pstreams[i].wait_stream(gs)
                    cur, m = xd, n
                    for s_ in range(stages):
                        c, p, st = pfir[i].filter(cur[:m], pbufs[i][s_ & 1])
                        cur, m = pbufs[i][s_ & 1], p
                    pgot[i] = m
                for i in range(pipes):
                    gs.wait_stream(pstreams[i])
            par_sec = replay_time(parallel_body)
            assert all(m == n - stages * (ntaps - 1) for m in pgot)
            # the parallel chains computed what the serial chain computes
            graph_body()
            gs.synchronize()
            ref_out = bufs[(stages - 1) & 1][: pgot[0]].clone()
            for i in range(pipes):
                assert torch.equal(pbufs[i][(stages - 1) & 1][: pgot[i]], ref_out), "parallel pipe differs from the serial chain"
    except Exception as e:  # noqa: BLE001
        graph_err = repr(e)[:200]
        print(f"[bench] perf/fir graph section: {graph_err}", file=sys.stderr)
    # end to end: host vector in, host vector out per pipe (VectorSource / VectorSink roles)
    h_in = torch.from_numpy(x).pin_memory()
    h_out = torch.empty(n, dtype=torch.float32).pin_memory()

    def e2e_pass():
        for _p in range(pipes):
            d = bufs[1]
            d.copy_(h_in, non_blocking=True)
            cur, m = d, n
            for s in range(stages):
                c, p, st = fir.filter(cur[:m], bufs[s & 1])
                cur, m = bufs[s & 1], p
            h_out[:m].copy_(cur[:m], non_blocking=True)
        torch.cuda.synchronize()
    e2e_pass()
    t0 = time.perf_counter()
    for _ in range(5):
        e2e_pass()
    e2e_s = (time.perf_counter() - t0) / 5
    val = pipes * n / sec / 1e6
    return {
        "config": {"workload": "perf/fir: pipes x stages of 64-tap f32 FirFilter on 1 M samples (BASELINE configs[0])",
                   "pipes": pipes, "stages": stages, "samples": n, "ntaps": ntaps, "algo": {1: "direct", 2: "tensor", 3: "fft"}.get(fir.algo)},
        "metric": "Msamples/s", "value": val, "unit": "Msamples/s (pipes x samples / elapsed, as perf/fir prints elapsed)",
        "ms_per_pass": sec * 1e3, "gpu_launches_per_pass": pipes * stages,
        "cuda_graph": ({"value": pipes * n / graph_sec / 1e6, "unit": "Msamples/s", "ms_per_pass": graph_sec * 1e3,
                        "note": "the same pipes x stages launches captured once in a CUDA graph and replayed"}
                       if graph_sec else {"error": locals().get("graph_err")}),
        "cuda_graph_parallel_pipes": ({"value": pipes * n / par_sec / 1e6, "unit": "Msamples/s", "ms_per_pass": par_sec * 1e3,
                                       "note": "one stream / context / buffer pair per pipe, forked and joined inside one CUDA graph: "
                                               "the pipes are independent branches of the flowgraph; outputs equal the serial chain's bit for bit"}
                                      if par_sec else {"error": locals().get("graph_err")}),
        "roofline": _roofline(8.0 * n * stages * pipes, min(sec, graph_sec or sec, par_sec or sec), "8 B/sample/stage; 30 launches of ~4 MB each: launch-latency bound (best of eager / graph replay); at this slice size AUTO runs the CUDA-core kernel (the tensor kernel's fixed cost is ~12 us per launch)"),
        "cpu_baseline": {"value": pipes * n / cpu_s / 1e6, "unit": "Msamples/s", "cores": pipes, "kind": "port",
                         "sample": "the whole config: 5 pipes x 6 stages x 1 M samples, oracle port of fir.rs:52-91 (strict order), one thread per pipe"},
        "e2e": {"value": pipes * n / e2e_s / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": 4 * n * pipes,
                "d2h_bytes_per_step": 4 * (n - stages * (ntaps - 1)) * pipes},
    }


def sec_ring_vulkan(torch, fb, dev, args):
    """The reference's accelerator-buffer benchmark (perf/vulkan/vulkan.rs:48-78, tests/vulkan.rs:56-76): 100 M random
    f32 from a host vector through H2D buffers -> compute kernel (x * 12) -> D2H buffers into a host vector, equality
    with orig * 12 and length preserved.  Here: VectorSource role -> b2s_ring_* (pinned staging per slot, async H2D,
    slot events) -> b2s_apply (in place in the slot) -> async D2H -> VectorSink role."""
    import ctypes as C
    from futuresdr_b200._lib import lib, check, EAGAIN
    from futuresdr_b200 import blocks as B
    n, chunk, n_slots = 100_000_000, 8 * 1024 * 1024, 4
    x = np.random.default_rng(3).random(n, dtype=np.float32)
    y = np.empty(n, np.float32)
    ctx = fb.default_context(dev.index)
    ring = C.c_void_p()
    check(lib.b2s_ring_create(ctx.handle, 4, chunk, 0, n_slots, 1, C.byref(ring)), ctx.handle)
    sc = B.Apply(B.ApplyOp.ScaleF32, 12.0)

    def host_view(slot, items):
        return np.frombuffer((C.c_char * (items * 4)).from_address(lib.b2s_slot_host_ptr(slot)), dtype=np.float32, count=items)

    def one_pass():
        pos, done, inflight = 0, 0, []
        while done < n:
            # source edge: fill every free slot
            while pos < n:
                slot = C.c_void_p()
                rc = lib.b2s_ring_acquire_empty(ring, C.byref(slot))
                if rc == EAGAIN:
                    break
                check(rc, ctx.handle)
                m = min(chunk, n - pos)
                host_view(slot, m)[:] = x[pos:pos + m]
                check(lib.b2s_ring_submit_full(ring, slot, m, 1), ctx.handle)
                # the GPU block: take the full slot, run the kernel in place, start the D2H
                full, valid = C.c_void_p(), C.c_size_t(0)
                check(lib.b2s_ring_acquire_full(ring, C.byref(full), C.byref(valid)), ctx.handle)
                dptr = lib.b2s_slot_device_ptr(full)
                cc, pp = C.c_size_t(0), C.c_size_t(0)
                check(lib.b2s_apply_exec(sc._h, C.c_void_p(dptr), valid.value, C.c_void_p(dptr), valid.value,
                                         C.byref(cc), C.byref(pp)), ctx.handle)
                check(lib.b2s_slot_fetch_to_host(full, valid.value), ctx.handle)
                inflight.append((full, pos, m))
                pos += m
            # sink edge: drain the oldest slot
            full, p0, m = inflight.pop(0)
            check(lib.b2s_slot_wait(full), ctx.handle)
            y[p0:p0 + m] = host_view(full, m)
            check(lib.b2s_ring_release(ring, full), ctx.handle)
            done += m
    one_pass()
    t0 = time.perf_counter()
    one_pass()
    sec = time.perf_counter() - t0
    ok = bool(np.all(np.abs(y - x * np.float32(12.0)) <= np.finfo(np.float32).eps * 12))   # tests/vulkan.rs:73-75
    lib.b2s_ring_destroy(ring)
    # device-resident figure for the same kernel (what the ring feeds)
    xd = torch.from_numpy(x[:64 * 1024 * 1024]).to(dev)
    dsec = _time_passes(torch, lambda: sc.apply(xd, xd), reps=10, warm=2)
    return {
        "config": {"workload": "accelerator-buffer ring: 100 M f32 host vector -> H2D ring -> x*12 kernel -> D2H -> host vector (perf/vulkan/vulkan.rs:48-78)",
                   "items": n, "slot_items": chunk, "n_slots": n_slots, "length_preserved_and_equal": ok},
        "metric": "Msamples/s", "value": xd.numel() / dsec / 1e6, "unit": "Msamples/s (f32 items, kernel on device-resident slots)",
        "roofline": _roofline(8.0 * xd.numel(), dsec, "4 B in + 4 B out per item"),
        "cpu_baseline": None,
        "e2e": {"value": n / sec / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": 4 * n, "d2h_bytes_per_step": 4 * n,
                "note": "includes the VectorSource / VectorSink memcpy into and out of the pinned slot staging, one host thread"},
    }


def _fm_chain(torch, fb, dev):
    from futuresdr_b200 import blocks as B
    dec = B.FirBuilder.decimating(4)
    dem = B.Apply(B.ApplyOp.QuadDemodC32)
    # prototype low-pass of the resampler from the product's own tap design (b2s_firdes_*; bit-identical to the
    # reference's firdes::kaiser::lowpass, tests/test_abi_symbols.py)
    ptaps = (fb.firdes.kaiser.lowpass(0.4 / 32, 0.1 / 32, 1e-3) * 32).astype(np.float32)[: 32 * 16]
    pfb = B.PfbArbResampler(0.768, ptaps, 32)
    return dec, dem, pfb, ptaps


def sec_config3_fm_chain(torch, fb, dev, args, h_in, h_out):
    """configs[2]: FirBuilder::decimating(4) (52-tap kaiser) -> Apply(quadrature demod, packed as Complex{phi, 0}) ->
    PfbArbResampler(0.768, 32 arms x 16 taps) on 256 Mi samples, 64 Mi-sample chunks, device-resident between blocks
    (examples/fm-receiver/src/main.rs:99-104, src/blocks/pfb/arb_resampler.rs:193-231)."""
    from futuresdr_b200 import blocks as B
    import oracle as orc
    total, S = 256 * 1024 * 1024, CHUNK
    nchunks = total // S
    H = 52                                                    # ceil(51 / 4) * 4: history keeping the decimator phase
    # synthetic input (SURVEY 8d): an FM signal (sinusoidal message, closed-form phase evaluated in f64) + white noise at
    # -26 dB.  Pure noise would make the parity spot check meaningless: arg() jumps by 2*pi wherever a decimator output
    # differs in the last bit near the negative real axis.
    x = torch.empty(total, dtype=torch.complex64, device=dev)
    g = torch.Generator(device=dev).manual_seed(SEED + 3)
    seg = 16 * 1024 * 1024
    for c0 in range(0, total, seg):
        tt = torch.arange(c0, c0 + seg, dtype=torch.float64, device=dev)
        ph = (-(0.05 / 0.0007)) * torch.cos(2 * np.pi * 0.0007 * tt)
        xs = torch.view_as_real(x[c0:c0 + seg])
        xs.normal_(generator=g)
        xs.mul_(0.05)
        xs[:, 0] += torch.cos(ph).float()
        xs[:, 1] += torch.sin(ph).float()
        del tt, ph
    d1 = torch.empty(S // 4 + 16, dtype=torch.complex64, device=dev)
    d2 = torch.empty(S // 4 + 16, dtype=torch.complex64, device=dev)
    d3 = torch.empty(int(S // 4 * 0.768) + 4096, dtype=torch.complex64, device=dev)
    dec, dem, pfb, ptaps = _fm_chain(torch, fb, dev)
    counts = {}

    def chunk_work(src, out3):
        c, p, st = dec.filter.filter(src, d1)
        q = dem.apply(d1[:p], d2)
        off, outn = 0, 0
        while off < q:                                        # window fill sets call_again on the very first call
            pfb.input.set(d2[off:q])
            pfb.output.data, pfb.output.len = out3[outn:], 0
            io = B.WorkIo()
            pfb.work(io)
            off += pfb.input.pos
            outn += pfb.output.len
            if pfb.input.pos == 0 and not io.call_again:
                break
        return p, outn

    def one_pass():
        pfb.reset(); dem.reset()
        tot_p = tot_o = 0
        for c in range(nchunks):
            src = x[:S] if c == 0 else x[c * S - H:(c + 1) * S]
            p, o = chunk_work(src, d3)
            tot_p += p; tot_o += o
        counts["decim"], counts["out"] = tot_p, tot_o
    sec = _time_passes(torch, one_pass, reps=3, warm=1)
    # exact output counts against the reference's arithmetic: decimator (decimating_fir.rs:70-78), resampler = oracle run
    assert counts["decim"] == (total - 51) // 4, counts
    # algorithmic bytes per INPUT sample, fused ideal (SURVEY 8d): 8 in + 8 * 0.768 / 4 out
    alg = total * (8 + 8 * 0.768 / 4)
    # cpu_baseline leg: the same chain with the oracle functions on a bounded sample -- the first 4 Mi samples of THIS
    # run's input, one thread (PfbArb is a sequential state machine).  Its output doubles as the checker of the device
    # chain on the same samples (counts exact, values compared).
    n_cpu = 4 * 1024 * 1024
    xs = x[:n_cpu].cpu().numpy()
    dtaps = orc.kaiser_lowpass(0.25, 0.1, 1e-4)
    t0 = time.perf_counter()
    _, _, _, dref = orc.decim_fir(dtaps, 4, xs, n_cpu)
    ph, _ = orc.quad_demod(dref)
    yref = orc.PfbArb(0.768, ptaps, 32).run(ph.astype(np.complex64), out_cap_per_call=1 << 22)
    cpu_s = time.perf_counter() - t0
    pfb.reset(); dem.reset()
    p, o = chunk_work(x[:n_cpu], d3)
    torch.cuda.synchronize()
    ydev = d3[:o].cpu().numpy()
    parity = {"n_in": n_cpu, "count_match": bool(o == yref.size), "n_out": int(o),
              "max_abs_err": float(np.max(np.abs(ydev - yref[:o]))) if o else None,
              "note": "device chain on the first 4 Mi samples of this run's input against the cpu_baseline run on the same samples; phases are O(pi)"}
    # end to end through host buffers: 64 Mi samples in 4 chunks of 16 Mi
    n_e = h_in.numel() - (h_in.numel() % 4)
    ce = 16 * 1024 * 1024
    pipe = HostPipe(torch, dev, torch.complex64, torch.complex64, ce, int(ce // 4 * 0.768) + 4096, halo=H)

    def reset():
        pfb.reset(); dem.reset()

    def work(src, dout):
        p, o = chunk_work(src, dout)
        return o
    e2e_s, prod = pipe.timed(h_in[:n_e], h_out, work, reset)
    return {
        "config": {"workload": "FM-receiver chain: FirBuilder decimator x4 -> Apply(demod) -> PfbArbResampler, 1 GPU, 256 Mi samples (BASELINE configs[2])",
                   "chunk_items": S, "decim_taps": 52, "decim_algo": {1: "direct", 2: "tensor", 3: "fft"}.get(dec.filter.algo),
                   "resampler": "rate 0.768, 32 arms x 16 taps", "demod": "quadrature, packed Complex{phi,0} (the chain does not type-check in the reference as written, SURVEY 7)"},
        "metric": "Msamples/s", "value": total / sec / 1e6, "unit": "Msamples/s (input samples)", "ms_per_pass": sec * 1e3,
        "outputs": counts, "parity_spot_check": parity,
        "roofline": _roofline(alg, sec, "fused-ideal bytes 8 + 8*0.768/4 per input sample; three kernels with HBM hand-offs in between"),
        "cpu_baseline": {"value": n_cpu / cpu_s / 1e6, "unit": "Msamples/s", "cores": 1, "kind": "port",
                         "sample": f"{n_cpu} input samples, oracle chain (decimating_fir.rs, fm-receiver demod closure, arb_resampler.rs), 1 thread"},
        "e2e": {"value": n_e / e2e_s / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": 8 * n_e, "d2h_bytes_per_step": 8 * prod,
                "note": "pinned host in -> H2D -> chain -> D2H -> pinned host out, 16 Mi-sample chunks, copies overlapped"},
    }


def sec_config4_fft(torch, fb, dev, args, h_in, h_out):
    """configs[3]: Fft block 4096-pt Complex<f32> over 1 Gi samples in 64 Mi-sample chunks (src/blocks/fft.rs:160-221);
    the fused spectrum pipe (FFT + |x|^2 + MovingAvg) is reported next to it."""
    from futuresdr_b200 import blocks as B
    total, S, N = 1024 * 1024 * 1024, CHUNK, 4096
    nchunks = total // S
    x = torch.empty(total, dtype=torch.complex64, device=dev)
    g = torch.Generator(device=dev).manual_seed(SEED + 4)
    for c in range(nchunks):                                   # chunked: normal_ on 2 Gi floats at once overflows int32 paths
        torch.view_as_real(x[c * S:(c + 1) * S]).normal_(generator=g)
    y = torch.empty(total, dtype=torch.complex64, device=dev)
    fft = B.Fft(N)

    def one_pass():
        for c in range(nchunks):
            fft.transform(x[c * S:(c + 1) * S], y[c * S:(c + 1) * S])
    sec = _time_passes(torch, one_pass, reps=2, warm=1)
    # parity spot check: 64 frames against numpy's pocketfft in double precision
    xs = x[:64 * N].cpu().numpy().astype(np.complex128).reshape(64, N)
    ref = np.fft.fft(xs, axis=1)
    got = y[:64 * N].cpu().numpy().reshape(64, N)
    err = float(np.max(np.abs(got - ref)) / np.max(np.abs(ref)))
    del y
    # fused spectrum pipe on the same stream: 8 B/sample in, N floats per 3 frames out
    sp = B.SpectrumPipe(N, 0.1, 3)
    po = torch.empty(S // 3 + 2 * N, dtype=torch.float32, device=dev)

    def spec_pass():
        for c in range(nchunks):
            sp.process(x[c * S:(c + 1) * S], po)
    ssec = _time_passes(torch, spec_pass, reps=2, warm=1)
    # CPU twin: pocketfft (scipy, all cores) -- NOT rustfft, which is not available here
    n_cpu = 16 * 1024 * 1024
    xc = _cpu_noise(n_cpu).reshape(-1, N)
    try:
        import scipy.fft as sfft
        workers = _cpu_threads()
        sfft.fft(xc[:64], axis=1, workers=workers)
        t0 = time.perf_counter()
        sfft.fft(xc, axis=1, workers=workers)
        cpu_s = time.perf_counter() - t0
        lib = f"scipy.fft (pocketfft, c64, {workers} workers)"
    except Exception:
        workers = 1
        t0 = time.perf_counter()
        np.fft.fft(xc, axis=1)
        cpu_s = time.perf_counter() - t0
        lib = "numpy.fft (pocketfft, 1 thread)"
    # end to end: 64 Mi samples through host buffers, 16 Mi-sample chunks
    n_e = (h_in.numel() // N) * N
    ce = 16 * 1024 * 1024
    pipe = HostPipe(torch, dev, torch.complex64, torch.complex64, ce, ce)

    def work(src, dout):
        return fft.transform(src, dout)
    e2e_s, prod = pipe.timed(h_in[:n_e], h_out, work, lambda: None)
    return {
        "config": {"workload": "Fft block 4096-pt Complex<f32> spectrum pipe, 1 Gi samples, 1 GPU (BASELINE configs[3])",
                   "fft_size": N, "chunk_items": S, "transforms": total // N},
        "metric": "Msamples/s", "value": total / sec / 1e6, "unit": "Msamples/s", "ms_per_pass": sec * 1e3,
        "parity_spot_check": {"frames": 64, "max_err_rel_to_max": err, "against": "numpy.fft in f64"},
        "roofline": _roofline(16.0 * total, sec, "16 B/sample: one pass through shared memory"),
        "fused_spectrum_pipe": {"workload": "Fft(4096, shift) -> |x|^2 -> MovingAvg<4096>(0.1, 3) in one pass (b2s_spectrum_*)",
                                "value": total / ssec / 1e6, "unit": "Msamples/s", "ms_per_pass": ssec * 1e3,
                                "roofline": _roofline((8.0 + 4.0 / 3.0) * total, ssec, "8 B/sample in + 4/3 B/sample out")},
        "cpu_baseline": {"value": n_cpu / cpu_s / 1e6, "unit": "Msamples/s", "cores": workers, "kind": "port",
                         "sample": f"{n_cpu} samples = {n_cpu // N} transforms, {lib}; NOT rustfft (un-vendored crate, no Rust toolchain)"},
        "e2e": {"value": n_e / e2e_s / 1e6, "unit": "Msamples/s", "h2d_bytes_per_step": 8 * n_e, "d2h_bytes_per_step": 8 * prod},
    }


def sec_config5_sharded_1024(torch, fb, dist, dev, args, world, rank):
    """configs[4]: sharded 1024-tap FIR, 1 Gi samples per rank in 64 Mi-sample chunks (8 Gi at 8 GPUs), the overlap
    region fetched from the left neighbour's ring; scaling = weak."""
    from futuresdr_b200.shard import ShardedFir
    ntaps, steps = 1024, 16
    taps = _taps(ntaps, seed=11)
    sh = ShardedFir(taps, CHUNK, np.complex64, device=dev, exchange=args.exchange)
    g = torch.Generator(device=dev).manual_seed(SEED + 50 + rank)
    if sh.exchange == "peer":
        for tns in sh.slot_tensors():
            torch.view_as_real(tns).normal_(generator=g)
    else:
        torch.view_as_real(sh.chunk).normal_(generator=g)
    out = torch.empty(CHUNK, dtype=torch.complex64, device=dev)
    for _ in range(3):
        sh.step(out)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e = _events(torch, 2)
    e[0].record()
    for _ in range(steps):
        sh.step(out)
    e[1].record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e[0].elapsed_time(e[1])
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec = float(t.item()) * 1e-3
    algo = sh._filter.algo
    if hasattr(sh, "close"):
        sh.close()
    res = None
    if rank == 0:
        cpu = cpu_fir(2 * 1024 * 1024, reps=1, ntaps=ntaps)
        res = {
            "config": {"workload": "sharded 1024-tap FIR with overlap-region exchange, 1 Gi samples per GPU, scaling at 1/2/4/8 (BASELINE configs[4]: 8 Gi at 8 GPUs)",
                       "ntaps": ntaps, "chunk_items": CHUNK, "steps": steps, "n_gpus": world, "total_samples": CHUNK * steps * world,
                       "algo": {1: "direct", 2: "tensor", 3: "fft (overlap-save)"}.get(algo), "exchange": sh.exchange},
            "metric": "Msamples/s", "value": CHUNK * steps * world / sec / 1e6, "unit": "Msamples/s", "ms_per_step": sec * 1e3 / steps,
            "scaling": "weak",
            "roofline": _roofline(16.0 * CHUNK * steps, sec, "16 B/sample per GPU; step time incl. exchange"),
            "cpu_baseline": {"value": cpu["msps"], "unit": "Msamples/s", "cores": cpu["threads"], "kind": "port",
                             "sample": f"2 Mi samples, oracle port of fir.rs:52-91 ({cpu['variant']}), {cpu['threads']} threads"},
            "e2e": None,
        }
    return res


# ------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    import futuresdr_b200 as fb
    from futuresdr_b200.numa import local_to_gpu
    from futuresdr_b200.shard import ShardedFir

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert args.gpus == world, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    taps = _taps()
    algo = {"auto": fb.ALGO_AUTO, "direct": fb.ALGO_DIRECT, "tensor": fb.ALGO_TENSOR}[args.algo]
    sh = ShardedFir(taps, CHUNK, np.complex64, device=dev, algo=algo, exchange=args.exchange)
    ctx = sh._filter.ctx
    # synthetic white noise generated on the device (Philox), per-rank subsequence; every ring slot is filled
    # before the timed region (inputs resident in HBM when it starts)
    g = torch.Generator(device=dev).manual_seed(SEED + rank)
    if sh.exchange == "peer":
        for tns in sh.slot_tensors():
            torch.view_as_real(tns).normal_(generator=g)
    else:
        torch.view_as_real(sh.chunk).normal_(generator=g)
    out = torch.empty(CHUNK, dtype=torch.complex64, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput (`value`): inputs already in HBM
    for _ in range(args.warmup):
        sh.step(out)
    # Nothing rank-specific may sit between the barrier and the timed loop: a 20-step region is ~5 ms, and the few
    # milliseconds NVML takes to start on rank 0 alone used to be charged to every other rank as a wait for rank 0's
    # first chunk (round 1's "0.155 ms per step of exchange" was exactly that).
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    l0 = ctx.launch_count
    ev = _events(torch, args.steps + 1)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    ev[0].record()
    produced = 0
    host_t0 = time.perf_counter()
    for i in range(args.steps):
        # the FIR kernel alone (for the roofline): events on the launching stream around the launch
        if sh.exchange == "peer":
            sh.on_kernel = lambda tag, _i=i: kev[_i][0 if tag == "begin" else 1].record()
            c, p, st = sh.step(out)
            sh.on_kernel = None
        else:
            orig = sh.compute

            def timed(src, o, _i=i, _f=orig):
                kev[_i][0].record()
                r = _f(src, o)
                kev[_i][1].record()
                return r
            sh.compute = timed
            c, p, st = sh.step(out)
            sh.compute = orig
        produced += p
        ev[i + 1].record()
    host_step_us = (time.perf_counter() - host_t0) / args.steps * 1e6      # host enqueue time per step
    if os.environ.get("B2S_HOST_TIMING"):
        print(f"host_step rank {rank}: {host_step_us:.1f} us to enqueue one step", file=sys.stderr, flush=True)
    barrier()
    launches = ctx.launch_count - l0
    if args.dump_outputs and rank == 0:          # before the sustained run below overwrites `out`
        dump_outputs(args.dump_outputs, out, c, p, st)
    clocks = sampler.stop() if rank == 0 else None
    total_ms = ev[0].elapsed_time(ev[-1])
    kern_ms = [a.elapsed_time(b) for a, b in kev]
    t = torch.tensor([total_ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    my_total_ms = total_ms
    total_ms = float(t.item())
    value = (CHUNK * world * args.steps) / (total_ms * 1e-3) / 1e6
    ctx.sync()                                   # reports a cross-GPU flag time-out, if any
    per_rank = None
    if world > 1:                                # who is the slow one, and is it the kernel or the gaps between kernels
        mine = torch.tensor([my_total_ms / args.steps, statistics.mean(kern_ms), max(kern_ms)], device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = [{"rank": i, "ms_per_step": float(v[0]), "kernel_ms_mean": float(v[1]), "kernel_ms_max": float(v[2])}
                    for i, v in enumerate(allr)]

    # ---- sustained regime: the same step back to back for >= 1 s (the board settles at its power-capped clock)
    sustained = None
    if not args.no_sustained:
        n_s = max(args.steps, int(1.0 / max(total_ms / args.steps * 1e-3, 1e-6)) + 1)
        s_sampler = ClockSampler(local)
        if rank == 0:
            s_sampler.start()
        barrier()
        se = _events(torch, 2)
        se[0].record()
        for _ in range(n_s):
            sh.step(out)
        se[1].record()
        barrier()
        s_clk = s_sampler.stop() if rank == 0 else None
        ts = torch.tensor([se[0].elapsed_time(se[1])], device=dev)
        if world > 1:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        s_ms = float(ts.item())
        peak, _ = _peak_hbm()
        sustained = {"steps": n_s, "seconds": s_ms * 1e-3, "ms_per_step": s_ms / n_s,
                     "value": CHUNK * world * n_s / (s_ms * 1e-3) / 1e6, "unit": "Msamples/s",
                     "roofline_frac_step": BYTES_PER_SAMPLE * CHUNK / (s_ms / n_s * 1e-3) / 1e9 / peak,
                     "clocks": s_clk}
        ctx.sync()

    # ---- end to end through the C-ABI host-slice call (`e2e`): pinned host in/out, H2D + D2H timed
    fir = sh._filter
    n_e2e = CHUNK
    with local_to_gpu(local) as numa:            # pinned pages on the GPU's NUMA node
        h_in = torch.empty(n_e2e + NTAPS - 1, dtype=torch.complex64).pin_memory()
        torch.view_as_real(h_in).normal_(generator=torch.Generator().manual_seed(SEED + 100 + rank))
        h_out = torch.empty(n_e2e, dtype=torch.complex64).pin_memory()
        h_out.zero_()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        fir.filter(h_in, h_out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        c, p, st = fir.filter(h_in, h_out)          # returns when h_out is filled
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = (n_e2e * world * e2e_steps) / float(te.item()) / 1e6
    assert p == n_e2e
    barrier()
    ceiling = host_copy_ceiling(torch, dev, h_in, h_out)          # all ranks copy at once, like the e2e leg
    if world > 1:
        tc = torch.tensor([ceiling["ceiling_Msamples_s"]], device=dev)
        dist.all_reduce(tc, op=dist.ReduceOp.SUM)
        ceiling["ceiling_Msamples_s_all_ranks"] = float(tc.item())
    ceiling["numa"] = numa

    # ---- secondary configs
    secondary = []
    if not args.no_secondary:
        def guarded(name, fn):
            try:
                r = fn()
                if r is not None:
                    secondary.append(r)
            except Exception as e:  # noqa: BLE001
                if rank == 0:
                    secondary.append({"config": {"workload": name}, "error": repr(e)[:300]})
        del sh, out
        torch.cuda.empty_cache()
        if world == 1:
            guarded("perf/fir (configs[0])", lambda: sec_config1_perf_fir(torch, fb, dev, args))
            guarded("perf/vulkan ring", lambda: sec_ring_vulkan(torch, fb, dev, args))
            guarded("FM chain (configs[2])", lambda: sec_config3_fm_chain(torch, fb, dev, args, h_in[:CHUNK], h_out))
            torch.cuda.empty_cache()
            guarded("Fft 4096 (configs[3])", lambda: sec_config4_fft(torch, fb, dev, args, h_in[:CHUNK], h_out))
            torch.cuda.empty_cache()
        guarded("sharded 1024-tap (configs[4])", lambda: sec_config5_sharded_1024(torch, fb, dist, dev, args, world, rank))

    if rank == 0:
        peak, peak_src = _peak_hbm()
        k_ms = statistics.mean(kern_ms)
        achieved = BYTES_PER_SAMPLE * CHUNK / (k_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "traffic_fir.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get({1: "direct", 2: "tensor"}.get(fir.algo, ""), None)
                traffic_src = "constant from profiles/traffic_fir.json (ncu --set full capture of this kernel, dram__bytes_read+write per launch); not re-measured in this run"
            except Exception:
                traffic = None
        cpu = None
        if world == 1 and not args.no_cpu:
            r = cpu_fir(4 * 1024 * 1024, reps=3)
            cpu = {"value": r["msps"], "unit": "Msamples/s", "cores": r["threads"], "kind": "port",
                   "sample": f"4 Mi samples x3 (best), same taps/noise family; oracle port of futuredsp "
                             f"fir.rs:52-91, variant {r['variant']} (strict {4*1024*1024/r['all']['stable_strict']/1e6:.1f} / "
                             f"reassoc {4*1024*1024/r['all']['nightly_reassoc']/1e6:.1f} Msamples/s)"}
        exch = {"peer": "left neighbour's 255-sample tail read by the FIR kernel's TMA loader over NVLink (CUDA-IPC peer mapping, device flags); one launch per step",
                "nccl": "NCCL all-gather of the 255-sample overlap + head launch",
                "none": "NO exchange: independent replicas (diagnostic)"}[args.exchange]
        line = {
            "metric": "Msamples/s", "value": value, "unit": "Msamples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic white noise (device Philox, per-rank subsequence)",
            "config": {"workload": "single-B200 Complex<f32> 256-tap FIR on 64 Mi-sample chunks via device-resident ring (BASELINE configs[1])",
                       "ntaps": NTAPS, "chunk_items": CHUNK, "algo": {1: "direct", 2: "tensor"}.get(fir.algo),
                       "ring": "b2s_ring_* slots [halo | chunk], 2 slots; chunk t's history = the tail of the previous slot (b2s_fir_exec_hist)" if args.exchange != "nccl" else "torch buffer [halo | chunk]",
                       "l2": "inputs larger than L2 (512 MiB in + 512 MiB out per step)",
                       "sharding": ("contiguous time ranges; " + exch) if world > 1 else "none"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel_ms": k_ms, "algorithmic_bytes_per_launch": BYTES_PER_SAMPLE * CHUNK},
            "sustained": sustained,
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_val, "unit": "Msamples/s", "h2d_bytes_per_step": (n_e2e + NTAPS - 1) * 8,
                    "d2h_bytes_per_step": n_e2e * 8, "steps": e2e_steps,
                    "api": "FirFilter.filter(host_in, host_out) -> b2s_fir_filter_host (pinned host, chunked H2D/kernel/D2H pipeline)",
                    "host_copy_ceiling": ceiling},
            "gpu_launches": int(launches),
            "parity": {"headline": "pinned: FirFilter is checked against the reference's known-answer vectors (fir.rs:283-365) through the oracle and the C ABI; tolerance 1e-5 * ||taps||_1 * max|x|",
                       "secondary": "configs[0], [4]: pinned (FIR).  MovingAvg: pinned (tests/moving_avg.rs).  configs[2] (PfbArbResampler, demod closure), configs[3] (Fft = rustfft, un-vendored), the FFT part of the spectrum pipe: parity UNPINNED -- the reference holds no value test; the oracle is a restatement of the cited lines.  Ring x12: the reference's own check (tests/vulkan.rs:73-75) is applied in the run"},
            "clocks": clocks,
            "per_rank": per_rank, "host_enqueue_us_per_step": host_step_us,
            "secondary": secondary,
        }
        try:
            # explanatory only: the FLOPs the tensor kernel EXECUTES (3 split-bf16 products over the block-Toeplitz
            # operand, K = ntaps + 127 rounded up to 16) against the dense bf16 tensor peak -- at 256 taps this, not
            # HBM, is what the kernel runs into (DESIGN.md 4.2).  The judged roofline above stays the HBM one
            # SURVEY.md 8(d) states for this metric.
            if fir.algo == 2:
                ksteps = -(-(NTAPS + 127) // 16)
                tiles = -(-CHUNK // 8192)
                mma_flops = float(tiles) * 3 * ksteps * 2 * 128 * 128 * 16
                tpeak, tsrc = 1590.0, "fallback (B200_PROFILING.md 1.59 PFLOP/s burst)"
                try:
                    mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
                    if "bf16_tflops" in mp:
                        tpeak, tsrc = float(mp["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops)"
                except Exception:
                    pass
                tach = mma_flops / (k_ms * 1e-3) / 1e12
                line["roofline"]["tensor_executed"] = {"achieved": tach, "peak": tpeak, "unit": "TFLOP/s",
                                                       "frac": tach / tpeak, "flops_per_launch": mma_flops,
                                                       "peak_source": tsrc}
        except Exception:
            pass
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--algo", default="auto", choices=["auto", "direct", "tensor"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary BASELINE configs")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 1 s sustained run")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl", "none"],
                    help="halo exchange of the sharded stream: in-kernel peer fetch over NVLink (default) or NCCL all-gather")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's results (rank 0) to DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the device path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
