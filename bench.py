#!/usr/bin/env python3
"""
bench.py -- Mpixels/s of the rational-Bloom insert+query hot path on 4K YUV444 inter-frames.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path (K1 threshold+count -> exact (k,l,T) -> K2 insert -> K3 query
-> K3b witness [-> NCCL all-gather of the bit arrays when N > 1]) over one synthetic stream of
`--frames` 4K YUV444 frames (BASELINE.json configs[2]: 300 frames, p = 0.05, threshold 3.0), i.e.
frames-1 inter-frame pairs.  `value` is measured with the stream resident in HBM; `e2e` repeats it
through the host-buffer API call with the H2D / D2H copies inside the timed region.

--dump-outputs DIR writes what the last timed step computed (rank 0's pairs) as DIR/<name>.npy, float32 / float64, under
DUMP_BUDGET bytes; the inputs are seeded, so two builds run with the same arguments can be compared array for array.

N > 1 is launched by torchrun (one process per GPU); every rank encodes its own stream (weak
scaling), time = max over ranks of the CUDA-event time, value = all ranks' pixels / that time.

--impl reference times the reference's CPU implementation (oracle/ref_port.py: the loop-for-loop
Python port with python-xxhash; the reference itself is Python source that does not travel) on the
box's host cores, on a bounded sample of the same workload.
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

METRIC = "Mpixels/s bloom insert+query, 4K YUV444 inter-frame"
BYTES_PER_PIXEL = 6            # SURVEY.md 8(d): both frames of the pair read once, 2 * 3 * sizeof(uint8)
DUMP_BUDGET = 48 << 20         # bytes of arrays --dump-outputs writes at most


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------ synthetic stream (SURVEY.md 8d, config 3)
def first_frame(h, w, seed, dtype):
    rng = np.random.default_rng(seed)
    if np.dtype(dtype) == np.uint16:                 # BASELINE configs[4]: 16-bit samples over the whole range (int16 wrap in the diff)
        return rng.integers(0, 65536, (h, w, 3), dtype=np.uint16)
    yy, xx = np.mgrid[0:h, 0:w]
    base = ((yy * 3 + xx * 2) % 240).astype(np.uint8)
    f0 = np.empty((h, w, 3), dtype=np.uint8)
    f0[:, :, 0] = base
    f0[:, :, 1] = base // 2 + 7
    f0[:, :, 2] = base // 3 + 90
    f0 += rng.integers(0, 8, (h, w, 3), dtype=np.uint8)
    return f0


def fill_stream(frames: np.ndarray, seed: int, one_in: int = 20) -> None:
    """frames[t] = frames[t-1] with Bernoulli(1/one_in) pixels having Y,U,V += 64 (mod 256)  [16-bit: += 16384 (mod 65536)]."""
    nfr, h, w, _ = frames.shape
    dt = frames.dtype
    step = dt.type(64 if dt == np.uint8 else 16384)
    frames[0] = first_frame(h, w, seed, dt)
    from concurrent.futures import ThreadPoolExecutor

    def delta(t):                                    # independent of the other frames: generated in parallel
        r = np.random.default_rng(seed + t)
        return (r.integers(0, one_in, (h, w), dtype=np.uint8) == 0).astype(dt) * step

    workers = max(1, min(16, (os.cpu_count() or 2) // max(1, int(os.environ.get("WORLD_SIZE", "1")))))
    with ThreadPoolExecutor(workers) as ex:
        for t0 in range(1, nfr, 32):
            ts = list(range(t0, min(nfr, t0 + 32)))
            for t, d in zip(ts, ex.map(delta, ts)):
                np.add(frames[t - 1], d[:, :, None], out=frames[t])      # uint8 arithmetic wraps


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.tmp.flush()
        self.tmp.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.tmp.read().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.tmp.name)
        except OSError:
            pass
        if sm:
            hot = sorted(sm)[len(sm) // 2:]             # samples under load: upper half
            out.update(sm_mhz=float(np.median(hot)), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------ CPU baseline (reference port on host cores)
def _cpu_worker(args):
    seed, rows, width = args
    from oracle import ref_port
    rng = np.random.default_rng(seed)
    prev = rng.integers(0, 256, (rows, width, 3), dtype=np.uint8)
    curr = prev.copy()
    ch = rng.integers(0, 20, (rows, width), dtype=np.uint8) == 0
    curr[ch] += 64
    t0 = time.perf_counter()
    px = ref_port.encode_pair(prev, curr, 3.0) if rows else 0
    return os.getpid(), px, time.perf_counter() - t0


def host_cores() -> int:
    """CPUs this process may really use: min(affinity mask, cpuset.cpus.effective, ceil(cpu.max quota / period)).
    A container lease often shows all of the box's CPUs in the affinity mask while its CFS quota is far smaller; a pool
    sized from the mask then thrashes (VERDICT r01: 5.8 vs 34 Mpx/s for the same port on "128 cores")."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    def _read(*paths):
        for q in paths:
            try:
                with open(q) as f:
                    return f.read().strip()
            except OSError:
                continue
        return None
    eff = _read("/sys/fs/cgroup/cpuset.cpus.effective", "/sys/fs/cgroup/cpuset/cpuset.effective_cpus")
    if eff:
        cnt = 0
        for part in eff.split(","):
            if "-" in part:
                a, b = part.split("-")
                cnt += int(b) - int(a) + 1
            elif part:
                cnt += 1
        if cnt:
            n = min(n, cnt)
    mx = _read("/sys/fs/cgroup/cpu.max")
    if mx:
        f = mx.split()
        if len(f) == 2 and f[0] != "max":
            n = min(n, max(1, -(-int(f[0]) // int(f[1]))))
    else:
        q, per = _read("/sys/fs/cgroup/cpu/cpu.cfs_quota_us"), _read("/sys/fs/cgroup/cpu/cpu.cfs_period_us")
        if q and per and int(q) > 0:
            n = min(n, max(1, -(-int(q) // int(per))))
    return max(1, n)


def _spin(n):
    t0 = time.perf_counter()
    x = 0
    for i in range(n):
        x += i * i
    return time.perf_counter() - t0


def effective_cores(limit: int) -> float:
    """Measured parallelism: a fixed pure-Python spin on 1 process vs on `limit` processes at once.  Catches CPU quotas the
    cgroup files do not show (effective = limit * t_single / t_parallel)."""
    import multiprocessing as mp
    if limit <= 1:
        return 1.0
    n = 6000000                                                            # ~0.25 s of CPython per task
    with mp.get_context("fork").Pool(limit) as pool:
        pool.map(_spin, [1000] * limit, chunksize=1)                      # start-up
        t1 = min(pool.map(_spin, [n], chunksize=1)[0] for _ in range(2))
        t0 = time.perf_counter()
        pool.map(_spin, [n] * limit, chunksize=1)
        tp = time.perf_counter() - t0
    return max(1.0, min(float(limit), limit * t1 / tp))


def reference_pool_size():
    """-> (workers, note).  One worker per usable core: cgroup/affinity limit, cut down to the measured parallelism."""
    lim = host_cores()
    eff = effective_cores(lim)
    use = max(1, min(lim, int(round(eff))))
    return use, "affinity/cgroup limit %d, measured parallelism %.1f" % (lim, eff)


class CpuReferencePool:
    """One worker process per host core running oracle/ref_port.py (the reference's loops).  The pool is forked and warmed
    (imports done) before anything is timed, so process start-up is not charged to the reference; a sample's time is the
    wall clock of the parallel map (synthetic band generation, ~3 % of a task, included)."""

    def __init__(self, cores: int):
        import multiprocessing as mp
        self.cores = cores
        self.pool = mp.get_context("fork").Pool(cores)
        self.pool.map(_cpu_worker, [(1, 0, 8)] * cores, chunksize=1)

    def sample(self, bands_per_core: int, rows: int, width: int, seed: int = 1000):
        """Each task = one `rows` x `width` band of a 4K YUV444 frame pair (p = 0.05) through the reference port."""
        tasks = [(seed + i, rows, width) for i in range(self.cores * bands_per_core)]
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker, tasks, chunksize=1)
        wall = time.perf_counter() - t0
        px = sum(r[1] for r in res)
        return px / wall / 1e6, px, wall

    def full_frame_check(self, height: int, width: int, tasks: int, seed: int = 777):
        """Calibration of the band sample: `tasks` FULL frames (n = height*width, 7-digit indices like the GPU workload)
        through the same port, one per worker -> Mpx/s per core at full-frame n."""
        tasks = max(1, min(tasks, self.cores))
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker, [(seed + i, height, width) for i in range(tasks)], chunksize=1)
        wall = time.perf_counter() - t0
        per_core = float(np.mean([r[1] / r[2] / 1e6 for r in res]))
        return {"n": height * width, "tasks": tasks, "wall_s": wall, "mpx_per_core": per_core}

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_c_oracle_sample(cores: int, frames: np.ndarray):
    """Extra, stronger CPU number: the C oracle (oracle/rbf_oracle.c), one frame pair per thread."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import c_oracle as co

    def one(t):
        m, _ = co.frame_diff_mask(frames[t], frames[t + 1], 3.0)
        co.compress(m.reshape(-1))
        return m.size
    n = min(cores, frames.shape[0] - 1)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(n) as ex:
        px = sum(ex.map(one, range(n)))
    return px / (time.perf_counter() - t0) / 1e6, n


def run_reference(args):
    """`--impl reference`: the reference's own CPU path (ported loop for loop) on all usable host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    use, note = reference_pool_size()
    rows = 68                                   # 68 x 3840 = 261 120 px per task: ~0.4 s of reference Python
    pool = CpuReferencePool(use)
    vals = []
    for i in range(args.warmup + args.steps):
        mps, px, wall = pool.sample(1, rows, args.width, seed=5000 + 100 * i)
        if i >= args.warmup:
            vals.append((mps, px, wall))
    ffc = pool.full_frame_check(args.height, args.width, 2) if args.full_frame_check else None
    pool.close()
    value = float(np.mean([v[0] for v in vals]))
    ms = float(np.mean([v[2] for v in vals]) * 1e3)
    from oracle import ref_port
    sample = "%d bands of %dx%d px (one per core, p=0.05, threshold 3.0) per step" % (use, rows, args.width)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "Mpixels/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": "4K (3840x2160) YUV444 inter-frame stream, p=0.05, threshold=3.0; bounded sample: " + sample},
            "cpu_baseline": {"value": value, "unit": "Mpixels/s", "cores": use, "mpx_per_core": value / use, "kind": "port",
                             "cores_note": note, "full_frame_check": ffc,
                             "sample": sample + "; " + ref_port.HASH_IMPL},
            "e2e": {"value": value, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------ ours
def pinned_array(cabi, shape, dtype=np.uint8):
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = C.c_void_p()
    cabi.check(cabi.lib().rbf_malloc_host(cabi.ctx(), nbytes, C.byref(p)), cabi.ctx())
    buf = (C.c_uint8 * nbytes).from_address(p.value)
    return np.frombuffer(buf, dtype=dtype).reshape(shape), p


def bind_near_gpu(gpu_index: int) -> bool:
    """N > 1: keep this rank (and the pinned frames it first-touches) on the CPUs NVML reports as local to its GPU, so
    eight ranks streaming 55 GB/s each over PCIe do not all pull from one socket's memory.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if len(cpus) < 4:
            return False
        os.sched_setaffinity(0, cpus)
        return True
    except Exception:
        return False


def stream_frames(F, H, W, seed, lo, hi, out):
    """Frames [lo, hi] of fill_stream(F-frame stream, seed) written to out[0 .. hi-lo] without building the whole stream:
    frame t = frame 0 + sum of the deltas 1..t (unsigned arithmetic wraps, so the sum may be taken in any order)."""
    from concurrent.futures import ThreadPoolExecutor
    dt = out.dtype
    step = dt.type(64 if dt == np.uint8 else 16384)
    f0 = first_frame(H, W, seed, dt)

    def delta(t):
        r = np.random.default_rng(seed + t)
        return (r.integers(0, 20, (H, W), dtype=np.uint8) == 0).astype(dt) * step

    workers = max(1, min(16, (os.cpu_count() or 2) // max(1, int(os.environ.get("WORLD_SIZE", "1")))))
    acc = np.zeros((H, W), dtype=dt)
    with ThreadPoolExecutor(workers) as ex:
        for t0 in range(1, lo + 1, 32):                    # fold the deltas before the shard into one offset
            for d in ex.map(delta, range(t0, min(lo + 1, t0 + 32))):
                acc += d
        np.add(f0, acc[:, :, None], out=out[0])
        for t0 in range(lo + 1, hi + 1, 32):
            ts = list(range(t0, min(hi + 1, t0 + 32)))
            for t, d in zip(ts, ex.map(delta, ts)):
                np.add(out[t - lo - 1], d[:, :, None], out=out[t - lo])


def kernel_counters(qkernel: str):
    """Per-pair ncu counters of the query kernel (profiles/r02_<kernel>_counters.json, written by scripts/ncu_summary.py
    from an `ncu --set full` capture of THIS round), valid only while the kernel sources still hash to what was profiled."""
    import hashlib
    try:
        with open(os.path.join(ROOT, "profiles", "r02_%s_counters.json" % qkernel)) as f:
            c = json.load(f)
        h = hashlib.sha256()
        for name in c.get("sources", []):
            with open(os.path.join(ROOT, name), "rb") as f:
                h.update(f.read())
        c["stale"] = h.hexdigest()[:16] != c.get("sources_sha16")
        return c
    except Exception:
        return None


def dump_outputs(out_dir, res, packed, seed=2024):
    """What one encode hands its caller, as .npy files: every pair's PairResult fields and the popcounts of its packed bitmap
    and witness, plus the packed bytes themselves (one float32 per byte, zero-padded to the longest) for a fixed, seeded sample
    of pairs -- all of them when they fit in DUMP_BUDGET.  `packed[t]` is st.fetch(t)'s (bitmap, witness, ...)."""
    os.makedirs(out_dir, exist_ok=True)
    out = {"pair_" + f: np.array([getattr(r, f) for r in res], dtype=np.float64)
           for f in ("n", "ones", "resid", "l", "wlen", "p", "k", "raw")}
    out["pair_bitmap_popcount"] = np.array([np.bitwise_count(b).sum() for b, *_ in packed], dtype=np.float64)
    out["pair_witness_popcount"] = np.array([np.bitwise_count(w).sum() for _, w, *_ in packed], dtype=np.float64)
    row_bytes = 4 * (max(b.size for b, *_ in packed) + max(w.size for _, w, *_ in packed))
    count = min(len(packed), max(1, DUMP_BUDGET // max(1, row_bytes)))
    pick = np.sort(np.random.default_rng(seed).choice(len(packed), count, replace=False))

    def padded(rows):
        a = np.zeros((len(rows), max(1, max(r.size for r in rows))), dtype=np.float32)
        for i, r in enumerate(rows):
            a[i, :r.size] = r
        return a
    out["sample_pairs"] = pick.astype(np.float64)
    out["sample_bitmap_bytes"] = padded([packed[t][0] for t in pick])
    out["sample_witness_bytes"] = padded([packed[t][1] for t in pick])
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    numa_bound = False
    if world > 1:
        import torch.distributed as dist                 # rendezvous / barriers only; the data path is the library's NCCL
        dist.init_process_group(backend="gloo")
        numa_bound = bind_near_gpu(local)
    import hashlib
    import new_bloom_filter_repo_b200 as pkg
    from new_bloom_filter_repo_b200 import _cabi as cabi, distributed as rdist
    L, ctx = cabi.lib(), cabi.ctx()
    info = cabi.device_info()
    H, W, F = args.height, args.width, args.frames
    n = H * W
    DT = np.uint16 if args.dtype == "u16" else np.uint8
    bpp = 2 * 3 * np.dtype(DT).itemsize                   # SURVEY 8(d): both frames of the pair, 6 B (8-bit) / 12 B (16-bit) per pixel
    strong = args.scaling == "strong" and world > 1
    cabi.check(L.rbf_set_option(ctx, b"k1_variant", args.k1_variant), ctx)
    cabi.check(L.rbf_set_option(ctx, b"query_variant", args.query_variant), ctx)
    if args.ranges is not None:
        cabi.check(L.rbf_set_option(ctx, b"encode_ranges", args.ranges), ctx)

    if strong:                                            # ONE stream of F frames, contiguous blocks of pairs per rank + halo frame
        lo, hi = rdist.shard_pairs(F - 1, rank, world)
        pairs = hi - lo
        slots_per_rank = -(-(F - 1) // world)             # every rank contributes the same number of slots
        nfr = pairs + 1
        frames, pin = pinned_array(cabi, (nfr, H, W, 3), DT)
        stream_frames(F, H, W, 3, lo, hi, frames)
    else:                                                 # weak: one F-frame stream per rank
        lo, pairs, slots_per_rank, nfr = 0, F - 1, F - 1, F
        frames, pin = pinned_array(cabi, (F, H, W, 3), DT)
        fill_stream(frames, seed=3 + 1000 * rank)
    enc = None
    if strong:                                            # the product entry point for a sharded stream
        enc = rdist.ShardedStreamEncoder(dist, H, W, 3, DT, F, gather=args.gather)
        assert (enc.layout["lo"], enc.layout["pairs"], enc.layout["slots"]) == (lo, pairs, slots_per_rank)
        st = enc.stream
        enc.upload(frames)
    else:
        st = pkg.FrameStream(H, W, 3, DT, max_frames=nfr, max_pairs=max(pairs, slots_per_rank))
        st.upload(frames)

    def barrier():
        if dist is not None:
            dist.barrier()
        cabi.check(L.rbf_sync(ctx), ctx)

    # multi-GPU: one all-gather of the packed bit arrays per step
    send = recv = peer = None
    slot = 0
    kw = {}
    res = enc.encode(3.0) if enc is not None else st.encode_consecutive(nfr, 3.0)
    if args.k_star:                                       # BASELINE configs[4]: explicit k*, l = int(p*n*k*/ln2) (SURVEY 8d)
        import math
        kw = {"k_override": [float(args.k_star)] * pairs,
              "l_override": [int((np.uint64(r.ones) / n) * n * args.k_star / math.log(2)) for r in res[:pairs]]}
        res = enc.encode(3.0, **kw) if enc is not None else st.encode_consecutive(nfr, 3.0, **kw)
    gather_used = args.gather if world > 1 else None
    if enc is not None:
        slot = enc.slot
        gather_used = enc.gather
    elif world > 1:
        slot = rdist.agree_slot_bytes(dist, max(r.l for r in res))
        gather_used = args.gather
        if args.gather == "p2p":                      # slots stored straight into every rank's buffer over NVLink peer memory
            peer = rdist.PeerGather.try_create(dist, slots_per_rank, slot)
            if peer is None:
                gather_used = "nccl (p2p unavailable: CUDA IPC failed on some rank)"
        if peer is None:
            rdist.init_nccl_from_torch(dist)
            send = rdist.DeviceBuffer(slot * slots_per_rank)
            recv = rdist.DeviceBuffer(slot * slots_per_rank * world)

    def step():
        if enc is not None:
            return enc.encode(3.0, **kw)
        r = st.encode_consecutive(nfr, 3.0, **kw)
        if peer is not None:
            peer.exchange(st)
        elif world > 1:
            cabi.check(L.rbf_stream_allgather_bitmaps(st._h, slots_per_rank, slot, send.ptr, recv.ptr), ctx)
        return r

    sampler = ClockSampler(local)
    for _ in range(args.warmup):
        step()
    barrier()
    cabi.check(L.rbf_reset_counters(ctx), ctx)
    stage_acc = {}
    cabi.check(L.rbf_timer_start(ctx), ctx)
    for _ in range(args.steps):
        res = step()
        for k_, v in st.stage_ms().items():
            stage_acc[k_] = stage_acc.get(k_, 0.0) + v
    ms = C.c_double()
    cabi.check(L.rbf_timer_stop_ms(ctx, C.byref(ms)), ctx)
    launches = int(L.rbf_get_counter(ctx, b"kernel_launches"))
    barrier()

    # ---- outside the timed region: what was timed is checked
    # (1) every pair decodes back to its mask on the GPU (ivc:268-307 round trip)
    mism = st.decode_verify()
    roundtrip_ok = not bool(mism.any())
    own_bm = [st.fetch(t, want_mask=False) for t in range(pairs)]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, own_bm)
    # (2) N > 1: every received slot equals the owner's bit array
    gather_check = strong_check = None
    if world > 1 and args.verify_gather:
        if enc is not None:
            got = enc._peer.result() if enc._peer is not None else enc._recv.to_host().reshape(world, slots_per_rank, slot)
        else:
            got = peer.result() if peer is not None else recv.to_host().reshape(world, slots_per_rank, slot)
        own = [hashlib.sha256(np.pad(own_bm[t][0], (0, slot))[:slot].tobytes()).hexdigest() for t in range(pairs)]
        table = [None] * world
        dist.all_gather_object(table, own)
        gather_check = all(hashlib.sha256(got[r, t].tobytes()).hexdigest() == table[r][t]
                           for r in range(world) for t in range(len(table[r])))
        gather_check = bool(gather_check and [hashlib.sha256(got[rank, t].tobytes()).hexdigest() for t in range(pairs)] == own)
        flags = [None] * world
        dist.all_gather_object(flags, gather_check)
        gather_check = all(flags)
        hdrs = enc.headers() if enc is not None else None     # collective: every rank calls it
        if strong and rank == 0:                      # (3) the gathered set == a single-GPU encode of the same F-frame stream
            full = np.empty((F, H, W, 3), dtype=DT)
            fill_stream(full, seed=3)
            st1 = pkg.FrameStream(H, W, 3, DT, max_frames=F)
            st1.upload(full)
            r1 = st1.encode_consecutive(F, 3.0)
            if args.k_star:
                import math
                r1 = st1.encode_consecutive(F, 3.0, k_override=[float(args.k_star)] * (F - 1),
                                            l_override=[int((np.uint64(r.ones) / n) * n * args.k_star / math.log(2)) for r in r1])
            flat = enc.gathered()                           # stream order, through the product's own accessor
            strong_check = len(flat) == F - 1 and [h[0] for h in hdrs] == [r.l for r in r1]
            for t in range(F - 1):
                bm1 = st1.fetch(t, want_mask=False)[0]
                strong_check = strong_check and bool(np.array_equal(np.pad(bm1, (0, slot))[:slot], flat[t]))
            st1.close()
            del full
    ms_local = ms.value
    if dist is not None:
        import torch
        t = torch.tensor([ms_local], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    else:
        ms_total = ms_local
    ms_per_step = ms_total / args.steps
    total_px = (F - 1) * n if strong else pairs * n * world
    value = total_px / (ms_per_step * 1e-3) / 1e6
    stage = {k_: v / args.steps for k_, v in stage_acc.items()}

    # ---- end to end: host frames -> C-ABI call -> packed outputs on the host, copies inside the timed region
    bm_slot = n // 8 if args.k_star else (max((r.l + 7) // 8 for r in res) + 15) // 16 * 16
    wt_slot = n // 8 if args.k_star else (max((r.wlen + 7) // 8 for r in res) + 15) // 16 * 16
    out_bm, pin_bm = pinned_array(cabi, (pairs, bm_slot))
    out_wt, pin_wt = pinned_array(cabi, (pairs, wt_slot))
    e2e_steps = max(1, args.e2e_steps)
    st.encode_host(frames, 3.0, bitmap_slot=bm_slot, witness_slot=wt_slot, out_bitmaps=out_bm, out_witness=out_wt)
    r_e2e = st.encode_host(frames, 3.0, bitmap_slot=bm_slot, witness_slot=wt_slot, out_bitmaps=out_bm, out_witness=out_wt)
    if args.k_star:                                       # the host-buffer call derives (k, l) itself: checked by its own round trip
        e2e_ok = not bool(st.decode_verify().any())
    else:
        e2e_ok = all(np.array_equal(out_bm[t, :own_bm[t][0].size], own_bm[t][0]) and
                     np.array_equal(out_wt[t, :own_bm[t][1].size], own_bm[t][1]) for t in range(pairs))
    barrier()
    cabi.check(L.rbf_reset_counters(ctx), ctx)
    cabi.check(L.rbf_timer_start(ctx), ctx)
    for _ in range(e2e_steps):
        st.encode_host(frames, 3.0, bitmap_slot=bm_slot, witness_slot=wt_slot, out_bitmaps=out_bm, out_witness=out_wt)
    ms2 = C.c_double()
    cabi.check(L.rbf_timer_stop_ms(ctx, C.byref(ms2)), ctx)
    h2d = int(L.rbf_get_counter(ctx, b"h2d_bytes")) // e2e_steps
    d2h = int(L.rbf_get_counter(ctx, b"d2h_bytes")) // e2e_steps
    e2e_ms = ms2.value / e2e_steps
    if dist is not None:
        import torch
        t = torch.tensor([e2e_ms], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = total_px / (e2e_ms * 1e-3) / 1e6
    clocks = sampler.stop()            # sampled from the first warm-up step to the end of the e2e region

    # ---- the same call for a caller that holds the planar Y (the reference's yuv_info['y_plane'], fvc:289-300): the mask only
    # needs Y, so a 1-channel stream moves a third of the bytes and produces the same bitmaps / witnesses
    ey = None
    if not args.k_star and not args.no_y_plane:
        yframes, pin_y = pinned_array(cabi, (nfr, H, W), DT)
        np.copyto(yframes, frames[:, :, :, 0])
        sty = pkg.FrameStream(H, W, 1, DT, max_frames=nfr, max_pairs=pairs)
        sty.encode_host(yframes, 3.0, bitmap_slot=bm_slot, witness_slot=wt_slot, out_bitmaps=out_bm, out_witness=out_wt)
        y_ok = all(np.array_equal(out_bm[t, :own_bm[t][0].size], own_bm[t][0]) and
                   np.array_equal(out_wt[t, :own_bm[t][1].size], own_bm[t][1]) for t in range(pairs))
        barrier()
        cabi.check(L.rbf_reset_counters(ctx), ctx)
        cabi.check(L.rbf_timer_start(ctx), ctx)
        ysteps = max(1, e2e_steps // 2)
        for _ in range(ysteps):
            sty.encode_host(yframes, 3.0, bitmap_slot=bm_slot, witness_slot=wt_slot, out_bitmaps=out_bm, out_witness=out_wt)
        ms3 = C.c_double()
        cabi.check(L.rbf_timer_stop_ms(ctx, C.byref(ms3)), ctx)
        y_ms = ms3.value / ysteps
        if dist is not None:
            import torch
            t = torch.tensor([y_ms], dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            y_ms = float(t.item())
        ey = {"value": total_px / (y_ms * 1e-3) / 1e6, "unit": "Mpixels/s", "ms_per_step": y_ms, "steps": ysteps,
              "h2d_bytes_per_step": int(L.rbf_get_counter(ctx, b"h2d_bytes")) // ysteps, "outputs_equal_yuv444_path": bool(y_ok),
              "api": "rbf_stream_encode_host on a 1-channel stream (planar Y in, same packed outputs)"}
        sty.close()

    # a plain pinned H2D copy of the same frames: what the link itself gives this rank (the e2e ceiling)
    cabi.check(L.rbf_sync(ctx), ctx)
    t0 = time.perf_counter()
    st.upload(frames)
    pcie_peak = frames.nbytes / (time.perf_counter() - t0) / 1e9

    if rank == 0:
        peak, peak_src = measured_peaks()
        q_ms = stage["k3_query"]
        coded_px = sum(r.n for r in res if not r.raw)
        qkernel = {5: "k_query4", 6: "k_query4", 0: "k_query"}.get(args.query_variant, "k_query2")
        kc = kernel_counters(qkernel)
        traffic = issue_frac = inst_px = None
        if kc is not None and not kc["stale"]:
            ncoded = sum(1 for r in res if not r.raw)
            traffic = kc["dram_bytes_per_pair"] * ncoded
            issue_frac, inst_px = kc.get("issue_active_frac"), kc.get("thread_inst_per_px")
        achieved = coded_px * bpp / (q_ms * 1e-3) / 1e9
        # (4) bitmap + witness of three pairs against the C oracle on the same frames
        oracle_ok = None
        if not args.no_cpu:
            from concurrent.futures import ThreadPoolExecutor
            from oracle import c_oracle as co

            def against_oracle(t):
                m, ones = co.frame_diff_mask(frames[t], frames[t + 1], 3.0)
                ob, ow, *_rest = co.compress(m.reshape(-1), k_l_override=((kw["k_override"][t], kw["l_override"][t]) if kw else None))
                return (ones == res[t].ones and np.array_equal(own_bm[t][0], np.packbits(ob)) and
                        np.array_equal(own_bm[t][1], np.packbits(ow)))
            picks = sorted({0, pairs // 2, pairs - 1})
            with ThreadPoolExecutor(len(picks)) as ex:
                oracle_ok = all(ex.map(against_oracle, picks))
        parity = bool(roundtrip_ok and e2e_ok and (oracle_ok is not False) and (gather_check is not False) and
                      (strong_check is not False))
        line = {
            "metric": METRIC if (H, W, args.dtype) == (2160, 3840, "u8") else "Mpixels/s bloom insert+query, %dx%d YUV444 %s inter-frame" % (W, H, args.dtype),
            "value": value, "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": ("4K (3840x2160)" if (H, W) == (2160, 3840) else "%dx%d" % (W, H)) + (" 16-bit" if DT == np.uint16 else "") +
                                   (" k*=%g" % args.k_star if args.k_star else "") + " YUV444 %d-frame synthetic stream -> %s, p=0.05, "
                                   "threshold=3.0, seeds 0x12345678/0x87654321/999 (BASELINE configs[%s]%s)" %
                                   (F, ("%d inter-frame pairs block-partitioned over %d GPUs (%d on rank 0)" % (F - 1, world, pairs)) if strong
                                    else "%d inter-frame pairs per GPU" % pairs, "3" if strong else "2",
                                    "; frames sharded per rank + one all-gather of the bit arrays" if world > 1 else ""),
                       "height": H, "width": W, "frames": F, "pairs_per_gpu": pairs, "parallelism": "frame-sharded x%d" % world,
                       "gather": gather_used, "gather_verified": gather_check,
                       "strong_matches_single_gpu": strong_check,
                       "parity_checked": parity,
                       "parity": {"decode_roundtrip_all_pairs": roundtrip_ok, "e2e_outputs_equal_resident": bool(e2e_ok),
                                  "c_oracle_pairs_0_mid_last": oracle_ok},
                       "l2_policy": "inputs larger than L2: %.2f GB of frames per step, no flush needed" % (nfr * n * 3 / 1e9),
                       "k1_variant": "tma-bulk-ring" if args.k1_variant == 1 else "ldg256", "rank_bound_to_gpu_numa_node": numa_bound,
                       "query_variant": {0: "per-lane", 1: "staged-rings", 5: "decade-tiles-carry", 6: "half-decade-tiles-carry"}.get(args.query_variant),
                       "mean_l_bits": float(np.mean([r.l for r in res])), "mean_witness_bits": float(np.mean([r.wlen for r in res]))},
            "roofline": {"bound": "hbm", "kernel": qkernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": coded_px * bpp, "algorithmic_bytes_per_px": bpp, "launch_ms": q_ms,
                         "pipeline_frac": value * 1e6 * bpp / 1e9 / world / peak,
                         "issue_frac": issue_frac, "thread_inst_per_px": inst_px,
                         "counters_source": (None if kc is None else ("profiles/r02_%s_counters.json%s" % (qkernel, " (STALE: kernel sources changed)" if kc["stale"] else ""))),
                         "note": "6 B/px (12 at 16 bit) counts both frames of a pair; consecutive pairs share a frame through L2, DRAM traffic of K1 is ~3.2 B/px",
                         "stage_ms": stage},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "Mpixels/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms, "steps": e2e_steps, "pcie_gbs": (h2d + d2h) / (e2e_ms * 1e-3) / 1e9,
                    "pcie_h2d_copy_gbs": pcie_peak, "pcie_frac_of_plain_copy": h2d / (e2e_ms * 1e-3) / 1e9 / pcie_peak,
                    "api": "rbf_stream_encode_host (pinned host frames in, packed bitmaps + witnesses out)",
                    "y_plane_only": ey},
            "gpu_launches": launches,
            "device": info["name"],
        }
        if world == 1 and not args.no_cpu:
            use, note = reference_pool_size()
            pool = CpuReferencePool(use)
            mps, px, wall = pool.sample(8, 68, W)
            ffc = pool.full_frame_check(H, W, 2) if args.full_frame_check else None
            pool.close()
            line["cpu_baseline"] = {"value": mps, "unit": "Mpixels/s", "cores": use, "mpx_per_core": mps / use, "kind": "port",
                                    "cores_note": note, "full_frame_check": ffc,
                                    "sample": "%d bands of 68x%d px (8 per core, p=0.05) through oracle/ref_port.py in %.1f s"
                                              % (8 * use, W, wall)}
            try:
                cm, cn = cpu_c_oracle_sample(use, frames[: min(nfr, use + 1)])
                line["cpu_baseline_c_oracle"] = {"value": cm, "unit": "Mpixels/s", "cores": cn, "kind": "port",
                                                 "sample": "%d full 4K pairs, one per thread, oracle/rbf_oracle.c" % cn}
            except Exception as e:       # pragma: no cover
                line["cpu_baseline_c_oracle"] = {"error": str(e)}
        print(json.dumps(line))
    st.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True     # the tree may be read-only: the project modules imported below leave no __pycache__ in it
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=300)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--k1-variant", type=int, default=0)
    ap.add_argument("--query-variant", type=int, default=5)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-y-plane", action="store_true", help="skip the planar-Y end-to-end measurement")
    ap.add_argument("--gather", default="p2p", choices=["nccl", "p2p"],
                    help="N > 1: the library's peer-memory push kernel over NVLink (default; validated at 2 and 8 GPUs, 17 %% / 79 %% faster "
                         "than NCCL in the weak / strong 8-GPU runs of profiles/r02_n8_*.json), or ncclAllGather; p2p falls back to nccl "
                         "when CUDA IPC is not available")
    ap.add_argument("--no-verify-gather", dest="verify_gather", action="store_false",
                    help="N > 1: skip the post-run comparison of every received slot with its owner's bit array")
    ap.add_argument("--verify-gather", dest="verify_gather", action="store_true", help="(default) kept for compatibility")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = one --frames stream per rank; strong = ONE --frames stream block-partitioned over the ranks "
                         "(BASELINE configs[3]), every rank ends up with all bit arrays, rank 0 re-encodes the stream alone and compares")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--dtype", default="u8", choices=["u8", "u16"], help="sample type of the synthetic YUV444 stream (u16: BASELINE configs[4])")
    ap.add_argument("--k-star", type=float, default=None, help="explicit k* with l = int(p*n*k*/ln2) instead of _calculate_optimal_params")
    ap.add_argument("--ranges", type=int, default=None, help="split each encode into this many pipelined ranges (library default if unset)")
    ap.add_argument("--no-full-frame-check", dest="full_frame_check", action="store_false",
                    help="CPU baseline: skip the full-frame (n = H*W) calibration sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0's pairs; see dump_outputs)")
    ap.set_defaults(verify_gather=True, full_frame_check=True)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
