#!/usr/bin/env python
"""bench.py -- headline benchmark of the rawspeed_b200 hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference]

Metric (BASELINE.json): MPixels/s decoded (bit-exact); achieved HBM GB/s vs roofline.

Headline workload at every N: BASELINE configs[4] -- a 256-frame batch of configs[2] frames
(DNG lossless-JPEG predictor 1, 14-bit 8256x5504 = 45 MP, 726 tiles of 256x256 each; 256
DISTINCT synthetic frames, seeds 12345+i), sharded 256/N frames per GPU: strong scaling, the
configuration north_star's target is quoted on ("45 MP 14-bit LJPEG decode ... with >= 6x
scaling at 8 GPUs on a 256-frame batch").  `value` = device-timed decode with inputs resident
in HBM (CUDA events, W warm-up + K timed steps, max over ranks); `roofline` for the decode
kernel in SURVEY 8(d)'s in+out bytes (and the read-only variant); `e2e` = the same batch through
the host-buffer C-ABI call (H2D + decode + D2H inside the timed region); `cpu_baseline` = the
reference's AbstractDngDecompressor::decompress() on the box's host cores (bounded sample);
`gather` (N > 1) = decode + NVLink output gather through the C ABI, both to every rank and to
the consumer GPU.  `single_frame` carries configs[2] proper (ONE frame per launch: decode,
roofline, pinned / pageable host runs, the host mirror's drop-in call), `others` configs[0],
[1] and [3] (and, with --all-legs, every secondary kernel).

One JSON line on stdout (rank 0).  A "step" = one pass of the hot path over the batch.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W, H, BPS = 8256, 5504, 14
PIX = W * H


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
        except Exception:
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def ncu_traffic(kernel):
    """DRAM bytes per frame of `kernel` from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(p)).get(kernel)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, idle = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                clk, cmax, util = float(f[0]), float(f[1]), float(f[7])
            except ValueError:
                continue
            mx.append(cmax)
            if util < 50.0:  # not under load: sampler started before the warm-up
                idle.append(clk)
                continue
            sm.append(clk)
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            sm = idle
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)),
                "samples_under_load": len(sm), "samples": len(sm) + len(idle),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------
def unpack_jobs(rs, frames, in_frame_bytes, out_frame_bytes, pitch, out_pitch, order):
    jobs = []
    for f in range(frames):
        j = rs.UnpackJob()
        j.in_offset = f * in_frame_bytes
        j.in_size = pitch * H
        j.out_offset = f * out_frame_bytes
        j.out_pitch = out_pitch
        j.row0, j.rows, j.samples, j.out_col0 = 0, H, W, 0
        j.in_pitch, j.bps, j.order = pitch, BPS, order
        jobs.append(j)
    return jobs


def align(x, a=256):
    return (x + a - 1) // a * a


def time_steps(torch, fn, steps, warmup, dist=None):
    """W untimed + K timed steps, CUDA events on the launching (current) stream,
    barrier + synchronize on both sides, max over ranks.  Returns total ms."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        ms = float(t.item())
    torch.cuda.synchronize()
    return ms


def wall_steps(torch, fn, steps, warmup, dist=None):
    """Same contract for the host-API path (its timed region is host-driven:
    pinned H2D + kernels + D2H, synchronous); wall clock bracketed by syncs."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def cpu_reference_unpack(sample_frames=1, reps=3):
    """The reference's own CPU path on this box's host cores (bounded sample)."""
    import oracle
    from oracle import port, synth
    ncores = os.cpu_count() or 1
    data, pitch = synth.packed_frame(W, H, BPS, seed=2)
    img = port.new_image(W, H)
    if oracle.HAVE_REF:
        ref = oracle.ref
        # (a) as shipped: UncompressedDecompressor is single threaded
        ms1 = min(ref.unpack(data, img, W, 1, (0, 0, W, H), pitch, BPS, port.MSB, reps=1)
                  for _ in range(reps))
        # (b) the reference's best OpenMP shape: rows split into one strip per core,
        #     fanned out by its own AbstractDngDecompressor (compression 1)
        th = (H + ncores - 1) // ncores
        nt = (H + th - 1) // th
        offs = [n * th * pitch for n in range(nt)]
        lens = [min(th, H - n * th) * pitch for n in range(nt)]
        # tile height th: last tile shorter; AbstractDngDecompressor wants full-size
        # tiles in the buffer only for the rows it reads
        msn = min(ref.dng_decompress(data, offs, lens, img, W, 1, W, th, 1, bps=BPS,
                                     nthreads=ncores, reps=1) for _ in range(reps))
        return {"kind": "reference", "cores": ncores,
                "value": PIX / (msn * 1e-3) / 1e6, "unit": "MPixels/s",
                "single_thread_value": PIX / (ms1 * 1e-3) / 1e6,
                "sample": "1 frame 8256x5504 14-bit MSB, best of %d; value = "
                          "AbstractDngDecompressor(compression 1) over %d row strips with %d "
                          "OpenMP threads; single_thread_value = UncompressedDecompressor as "
                          "shipped (no OpenMP)" % (reps, nt, ncores)}
    t0 = time.perf_counter()
    port.unpack(data, img, W, 1, (0, 0, W, H), pitch, BPS, port.MSB)
    ms = (time.perf_counter() - t0) * 1e3
    return {"kind": "port", "cores": 1, "value": PIX / (ms * 1e-3) / 1e6,
            "unit": "MPixels/s", "sample": "1 frame 8256x5504 14-bit MSB, oracle C port"}


# ------------------------------------------------------------------
# LJPEG workloads (BASELINE configs[2] / configs[4])
# ------------------------------------------------------------------
FRAMES_TOTAL = 256      # configs[4]: 256-frame batch, sharded 256/N per GPU (strong scaling)
SEED0 = 12345           # frame i is synth.image_model(W, H, SEED0 + i) (SURVEY 8d C5)


_WTS = {}


def _weights(w=W, h=H):
    """Per-pixel weights of the second checksum (uint64 wrap-around arithmetic)."""
    if (w, h) not in _WTS:
        x = np.arange(w, dtype=np.uint64)[None, :]
        y = np.arange(h, dtype=np.uint64)[:, None]
        _WTS[(w, h)] = ((x * np.uint64(31) + y * np.uint64(17)) & np.uint64(0xFFFF)) | np.uint64(1)
    return _WTS[(w, h)]


def frame_image(w, h, seed):
    """Same pixels as oracle.synth.image_model(w, h, seed) (SURVEY 8d C3: px = (2000 + ((7x+3y)&1023)
    + noise6 - 32) & 0x3FFF), without the full-size coordinate grids (tests/test_bench_synth.py
    pins the equality)."""
    from oracle import synth
    r = synth.lcg_u32(w * h, seed).reshape(h, w)
    x = np.arange(w, dtype=np.uint32)[None, :]
    y = np.arange(h, dtype=np.uint32)[:, None]
    v = (np.uint32(7) * x + np.uint32(3) * y) & np.uint32(1023)
    v += np.uint32(2000 - 32)
    v += r >> np.uint32(26)
    v &= np.uint32(0x3FFF)
    return v.astype(np.uint16)


def _gen_frame(job):
    """Worker (no CUDA): synthesise frame `seed`, encode it as a tiled LJPEG DNG payload, put the
    bytes into the shared block and return the scan descriptors + two checksums of the image."""
    seed, shm_name, off, cap = job
    from multiprocessing import shared_memory
    from oracle import synth
    import rawspeed_b200 as rs
    from helpers import dng_ljpeg_scans
    img, s0, s1 = synth.image_model_c(W, H, seed)
    t = synth.make_dng_ljpeg(img, 256, 256, threads=1)  # (one encoder thread: the pool is the parallelism)
    assert t.blob.size <= cap, (t.blob.size, cap)
    shm = shared_memory.SharedMemory(name=shm_name)
    try:
        np.frombuffer(shm.buf, dtype=np.uint8, count=t.blob.size, offset=off)[:] = t.blob
    finally:
        shm.close()
    tabs, scans = dng_ljpeg_scans(t, rs.image_pitch(W))
    keys = list(tabs.keys.keys())
    return (seed, int(t.blob.size), b"".join(bytes(s_) for s_ in scans), keys, s0, s1,
            [int(o) for o in t.offsets], [int(n) for n in t.lengths])


def _worker_init():
    os.environ["OMP_NUM_THREADS"] = "1"
    os.environ.pop("OMP_PROC_BIND", None)
    os.environ.pop("OMP_PLACES", None)


def gen_frames(seeds, procs):
    """Distinct synthetic frames, generated on the host cores in parallel (before CUDA is
    touched).  Returns (shared block, per-frame capacity, per-frame records)."""
    from multiprocessing import shared_memory, get_context
    cap = align(int(PIX * 1.25) + 4096)  # the synthetic frames compress to ~1.01 byte/pixel
    shm = shared_memory.SharedMemory(create=True, size=max(1, len(seeds)) * cap)
    jobs = [(sd, shm.name, k * cap, cap) for k, sd in enumerate(seeds)]
    if procs > 1 and len(seeds) > 1:
        # one thread per worker: the pool is the parallelism (the oracle library is an OpenMP build)
        with get_context("fork").Pool(min(procs, len(seeds)), initializer=_worker_init) as pool:
            recs = pool.map(_gen_frame, jobs, chunksize=1)
    else:
        recs = [_gen_frame(j) for j in jobs]
    return shm, cap, recs


class LJpegBatch:
    """Frames of one rank laid out in one input / one output buffer + the plan over all tiles."""

    def __init__(self, torch, rs, ctx, shm, cap, recs, pinned=True):
        from helpers import TableSet
        self.n = len(recs)
        self.out_pitch = rs.image_pitch(W)
        self.ob = align(H * self.out_pitch)
        self.in_off = []
        off = 0
        for r in recs:
            self.in_off.append(off)
            off += align(r[1])
        self.in_bytes = off
        self.h_in = torch.empty(self.in_bytes + 64, dtype=torch.uint8, pin_memory=pinned)
        hv = self.h_in.numpy()
        src = np.frombuffer(shm.buf, dtype=np.uint8)
        tabs = TableSet()
        scans = []
        ssz = C_sizeof_scan(rs)
        for k, r in enumerate(recs):
            hv[self.in_off[k]:self.in_off[k] + r[1]] = src[k * cap:k * cap + r[1]]
            tid = [tabs.add(*key) for key in r[3]]
            for j in range(len(r[2]) // ssz):
                s1 = rs.LJpegScan.from_buffer_copy(r[2][j * ssz:(j + 1) * ssz])
                s1.in_offset += self.in_off[k]
                s1.out_offset += k * self.ob
                for c in range(4):
                    s1.table[c] = tid[s1.table[c]] if s1.table[c] < len(tid) else 0
                scans.append(s1)
        del src
        self.recs = recs
        self.tabs = tabs
        self.scans = scans
        self.plan = rs.ljpeg_plan(ctx, tabs.tabs, scans)
        self.d_in = self.h_in.cuda()
        self.out_bytes = self.n * self.ob

    def check(self, torch, d_out, wts, full_frames=()):
        """All frames by two checksums (uint64 wrap-around) against the generator's image; the
        frames listed in full_frames bit for bit against a regenerated image."""
        from oracle import synth
        ok = True
        for k, r in enumerate(self.recs):
            fr = d_out[k * self.ob:k * self.ob + H * self.out_pitch].view(torch.int16).view(H, self.out_pitch // 2)
            v = (fr[:, :W].to(torch.int64) & 0xFFFF)
            s0 = int(v.sum().item()) & 0xFFFFFFFFFFFFFFFF
            s1 = int((v * wts).sum().item()) & 0xFFFFFFFFFFFFFFFF
            ok = ok and s0 == r[4] and s1 == r[5]
        for k in full_frames:
            img = synth.image_model(W, H, self.recs[k][0])  # (the oracle's generator, not the fast copy)
            g = d_out[k * self.ob:k * self.ob + H * self.out_pitch].cpu().numpy().view(np.uint16).reshape(H, self.out_pitch // 2)
            ok = ok and bool(np.array_equal(g[:, :W], img))
        return ok


def dump_outputs(torch, path, batch, d_out, plan, nsample=8 << 20):
    """What the last step of the timed path handed its caller, as .npy files under `path`: every
    frame's pixel sum (exact in float64), a fixed sample of pixels (seed 0: the same positions
    in every run with the same arguments) and every segment's (status, consumed)."""
    os.makedirs(path, exist_ok=True)
    st = plan.results(check=False)
    px = d_out[:batch.out_bytes].view(torch.int16).view(batch.n, batch.ob // 2)
    sums = np.array([float((px[k, :H * batch.out_pitch // 2].view(H, -1)[:, :W].to(torch.int64) & 0xFFFF)
                           .sum().item()) for k in range(batch.n)], dtype=np.float64)
    flat = np.sort(np.random.default_rng(0).integers(0, batch.n * H * W, nsample))
    f, y, x = flat // (H * W), flat % (H * W) // W, flat % W
    at = torch.from_numpy(f * (batch.ob // 2) + y * (batch.out_pitch // 2) + x).cuda()
    sample = (px.view(-1)[at].to(torch.int32) & 0xFFFF).to(torch.float32).cpu().numpy()
    np.save(os.path.join(path, "frame_pixel_sums.npy"), sums)
    np.save(os.path.join(path, "pixel_sample.npy"), sample)
    np.save(os.path.join(path, "segment_status.npy"), np.array([s for s, _ in st], dtype=np.float64))
    np.save(os.path.join(path, "segment_consumed.npy"), np.array([c for _, c in st], dtype=np.float64))


def C_sizeof_scan(rs):
    import ctypes
    return ctypes.sizeof(rs.LJpegScan)


def cpu_reference_ljpeg(shm, cap, recs, reps=5, warm=1):
    """The reference's own CPU path for this workload on the box's host cores:
    AbstractDngDecompressor::decompress() (OpenMP over the tiles) on a bounded sample of frames,
    median of `reps` passes after `warm` warm-up passes."""
    import oracle
    from oracle import port
    ncores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    src = np.frombuffer(shm.buf, dtype=np.uint8)
    frames = [(src[k * cap:k * cap + r[1]].copy(), r[6], r[7]) for k, r in enumerate(recs)]
    del src
    img = port.new_image(W, H)
    if oracle.HAVE_REF:
        def one_pass(nt):
            return sum(oracle.ref.dng_decompress(b, o, l, img, W, 1, 256, 256, 7, nthreads=nt, reps=1)
                       for b, o, l in frames)
        for _ in range(warm):
            one_pass(ncores)
        ts = sorted(one_pass(ncores) for _ in range(reps))
        ms = ts[len(ts) // 2]
        ms1 = oracle.ref.dng_decompress(frames[0][0], frames[0][1], frames[0][2], img, W, 1, 256, 256, 7,
                                        nthreads=1, reps=1)
        return {"kind": "reference", "cores": ncores, "unit": "MPixels/s",
                "value": len(frames) * PIX / (ms * 1e-3) / 1e6,
                "best": len(frames) * PIX / (ts[0] * 1e-3) / 1e6,
                "worst": len(frames) * PIX / (ts[-1] * 1e-3) / 1e6,
                "single_thread_value": PIX / (ms1 * 1e-3) / 1e6,
                "sample": "%d frame(s) 8256x5504 DNG LJPEG (726 tiles each), "
                          "AbstractDngDecompressor::decompress() with %d OpenMP threads "
                          "(OMP_PROC_BIND=close, OMP_PLACES=cores), median of %d passes after %d warm-up; "
                          "single_thread_value = the same with 1 thread" % (len(frames), ncores, reps, warm)}
    t0 = time.perf_counter()
    for b, o, l in frames:
        port.dng_decompress(b, o, l, img, W, 1, 256, 256, 7, nthreads=ncores)
    ms = (time.perf_counter() - t0) * 1e3
    return {"kind": "port", "cores": ncores, "unit": "MPixels/s", "value": len(frames) * PIX / (ms * 1e-3) / 1e6,
            "sample": "%d frame(s), oracle C port with %d OpenMP threads" % (len(frames), ncores)}


def cpu_baseline_children(args):
    """cpu_baseline of the GPU arm = the reference arm itself on a smaller sample (child processes,
    one per CPU placement; this process's OpenMP runtime and affinity are torch's business)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3", "--warmup", "1",
           "--ref-frames", str(max(1, args.cpu_frames))]
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "OMP_NUM_THREADS"):
        env.pop(k, None)
    try:
        os_aff = None
        if hasattr(os, "sched_getaffinity"):
            os_aff = os.sched_getaffinity(0)
            os.sched_setaffinity(0, range(os.cpu_count() or 1))  # children start from the whole box
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
        if os_aff:
            os.sched_setaffinity(0, os_aff)
        return json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
    except Exception as ex:  # noqa: BLE001
        return {"kind": "reference", "error": str(ex)[:200]}


def cpu_reference_c1():
    """BASELINE configs[0]: UncompressedDecompressor 12-bit packed, 4000x3000, CPU only --
    the reference's own accounting (items = pixels, bytes = bps*pixels/8,
    bench/librawspeed/decompressors/UncompressedDecompressorBenchmark.cpp:80-82)."""
    import oracle
    from oracle import port, synth
    if not oracle.HAVE_REF:
        return None
    w, h, bps = 4000, 3000, 12
    out = {}
    for name, order in (("MSB", port.MSB), ("LSB", port.LSB)):
        data, pitch = synth.packed_frame(w, h, bps, seed=1)
        img = port.new_image(w, h)
        ts = sorted(oracle.ref.unpack(data, img, w, 1, (0, 0, w, h), pitch, bps, order, reps=1) for _ in range(7))
        ms = ts[len(ts) // 2]
        out[name] = {"ms": ms, "MPixels/s": w * h / (ms * 1e-3) / 1e6,
                     "input_MB/s": w * h * bps / 8 / (ms * 1e-3) / 1e6}
    out["what"] = ("configs[0]: UncompressedDecompressor::readUncompressedRaw 12-bit 4000x3000 on the host, "
                   "1 thread as shipped, median of 7")
    return out


def numa_cpu_sets():
    """{"all": every CPU, "node0": the CPUs of NUMA node 0} (the latter from sysfs when present)."""
    ncpu = os.cpu_count() or 1
    sets = {"all": list(range(ncpu))}
    try:
        txt = open("/sys/devices/system/node/node0/cpulist").read().strip()
        cpus = []
        for part in txt.split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        if 0 < len(cpus) < ncpu:
            sets["node0"] = cpus
    except Exception:
        pass
    return sets


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the headline workload (DNG LJPEG
    frames through AbstractDngDecompressor::decompress), rank 0 only; one step = a bounded sample
    of the batch.  The OpenMP team is placed when the runtime starts, so every placement is
    measured in a child process of its own (all CPUs of the box / the CPUs of one NUMA node, one
    thread per CPU each) and the line reports the fastest -- the reference at its best on this box --
    with the others beside it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.ref_affinity is None:
        sets = numa_cpu_sets()
        lines = {}
        for name in sets:
            cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--ref-affinity", name,
                   "--steps", str(args.steps), "--warmup", str(args.warmup), "--gpus", str(args.gpus),
                   "--ref-frames", str(args.ref_frames)]
            try:
                r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
                lines[name] = json.loads(r.stdout.strip().splitlines()[-1])
            except Exception as ex:  # noqa: BLE001
                lines[name] = {"error": str(ex)[:200]}
        good = {k: v for k, v in lines.items() if "value" in v}
        if not good:
            print(json.dumps({"impl": "reference", "unavailable": "reference arm failed: %s" % lines}))
            return
        best = max(good, key=lambda k: good[k]["value"])
        line = good[best]
        line["cpu_baseline"]["placements"] = {k: (v.get("value"), v.get("cpu_baseline", {}).get("cores"))
                                              for k, v in lines.items()}
        line["cpu_baseline"]["sample"] += "; placement '%s' (the fastest of %s)" % (best, sorted(lines))
        print(json.dumps(line))
        return
    cpus = numa_cpu_sets().get(args.ref_affinity)
    if cpus:
        try:
            os.sched_setaffinity(0, cpus)
        except Exception:
            pass
        os.environ["OMP_NUM_THREADS"] = str(len(cpus))
    # stable placement of the reference's OpenMP team (set before the runtime starts)
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "threads")
    nsample = max(1, args.ref_frames)
    shm, cap, recs = gen_frames([SEED0 + i for i in range(nsample)], procs=min(nsample, os.cpu_count() or 1))
    try:
        import oracle
        from oracle import port
        ncores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        src = np.frombuffer(shm.buf, dtype=np.uint8)
        frames = [(src[k * cap:k * cap + r[1]].copy(), r[6], r[7]) for k, r in enumerate(recs)]
        del src
        img = port.new_image(W, H)
        dec = oracle.ref.dng_decompress if oracle.HAVE_REF else None

        def step():
            if dec:
                return sum(dec(b, o, l, img, W, 1, 256, 256, 7, nthreads=ncores, reps=1) for b, o, l in frames)
            t0 = time.perf_counter()
            for b, o, l in frames:
                port.dng_decompress(b, o, l, img, W, 1, 256, 256, 7, nthreads=ncores)
            return (time.perf_counter() - t0) * 1e3
        for _ in range(args.warmup):
            step()
        ts = [step() for _ in range(args.steps)]
        ms = float(np.median(ts))
        v = nsample * PIX / (ms * 1e-3) / 1e6
        cb = {"kind": "reference" if dec else "port", "cores": ncores, "value": v, "unit": "MPixels/s",
              "best": nsample * PIX / (min(ts) * 1e-3) / 1e6, "worst": nsample * PIX / (max(ts) * 1e-3) / 1e6,
              "sample": "%d distinct frame(s) 8256x5504 DNG LJPEG per step, AbstractDngDecompressor::decompress() "
                        "with %d OpenMP threads (OMP_PROC_BIND=close, OMP_PLACES=cores); value = median of the "
                        "%d timed steps" % (nsample, ncores, args.steps)}
        line = {
            "impl": "reference", "metric": "MPixels/s decoded (bit-exact)", "value": v,
            "unit": "MPixels/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u16", "data": "synthetic",
            "config": {"workload": "configs[4]: batch of configs[2] frames (DNG lossless-JPEG predictor 1, "
                                   "8256x5504, 726 tiles of 256x256); %d frames per step = a bounded sample "
                                   "of the GPU arm's 256-frame batch" % nsample},
            "cpu_baseline": cb,
            "e2e": {"value": v, "unit": "MPixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
    finally:
        shm.close()
        shm.unlink()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--total-frames", type=int, default=FRAMES_TOTAL,
                    help="frames of the batch over all GPUs (configs[4]: 256)")
    ap.add_argument("--ref-frames", type=int, default=8, help="frames per step of --impl reference")
    ap.add_argument("--ref-affinity", default=None, help="(internal) CPU placement of one reference-arm child")
    ap.add_argument("--cpu-frames", type=int, default=4, help="frames of the cpu_baseline sample")
    ap.add_argument("--gen-procs", type=int, default=0, help="host processes that synthesise the frames")
    ap.add_argument("--frames", type=int, default=8, help="frames per step of the configs[1] unpack leg")
    ap.add_argument("--ljpeg-frames", type=int, default=8)
    ap.add_argument("--ljpeg-big-frames", type=int, default=64)
    ap.add_argument("--sustain-s", type=float, default=1.0,
                    help="seconds of the same step back to back after the timed steps "
                         "(clock sampling + sustained figure)")
    ap.add_argument("--c5", action="store_true", help="(kept for compatibility: the headline IS configs[4] now)")
    ap.add_argument("--all-legs", action="store_true",
                    help="also time every secondary kernel (UncompressedDecompressor forms, vendor codecs, "
                         "post-decode stages): several minutes")
    ap.add_argument("--skip-others", action="store_true")
    ap.add_argument("--skip-single", action="store_true")
    ap.add_argument("--only-unvalidated", action="store_true")
    ap.add_argument("--unvalidated", action="store_true",
                    help="with --all-legs: include the post-decode kernels K9-K12 and Panasonic V4")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0's frames) "
                         "as DIR/<name>.npy, about 35 MB")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    pin_rank_to_numa(local)

    # ---------------- synthetic frames: this rank's share of the 256-frame batch ----------------
    FT = args.total_frames
    per = (FT + world - 1) // world
    mine = list(range(rank * per, min(FT, (rank + 1) * per)))  # contiguous blocks of 256/N frames
    ncpu = os.cpu_count() or 1
    procs = args.gen_procs or max(1, min(len(mine), (ncpu - 2 * world) // world))
    t_gen = time.perf_counter()
    shm, cap, recs = gen_frames([SEED0 + i for i in mine], procs)
    t_gen = time.perf_counter() - t_gen

    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist_
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist_.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_
    torch.cuda.set_device(local)
    import rawspeed_b200 as rs
    from oracle import port, synth  # checker + synthetic inputs only
    ctx = rs.Context(local)
    peak, peak_src = measured_peaks()
    try:
        batch = LJpegBatch(torch, rs, ctx, shm, cap, recs)
        d_out = torch.zeros(batch.out_bytes, dtype=torch.uint8, device="cuda")
        plan = batch.plan
        in_b, out_b, pixels = plan.bytes()
        run = lambda: plan.run((batch.d_in.data_ptr(), batch.in_bytes), d_out)  # noqa: E731

        # parity gate (not timed): every frame by checksum, first / last frame bit for bit
        run()
        st = plan.results()
        wts = torch.from_numpy(_weights().view(np.int64)).cuda()
        bit_exact = all(s == 0 for s, _ in st) and batch.check(torch, d_out, wts, sorted({0, batch.n - 1}))
        if dist is not None:
            t = torch.tensor([1 if bit_exact else 0], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            bit_exact = bool(t.item())
        if not bit_exact:
            if rank == 0:
                print(json.dumps({"error": "GPU output differs from the encoder's input; no number reported"}))
            sys.exit(1)

        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        l0 = ctx.launches
        ms = time_steps(torch, run, args.steps, args.warmup, dist)
        launches = ctx.launches - l0 - args.warmup * plan.launches
        if args.dump_outputs and rank == 0:
            dump_outputs(torch, args.dump_outputs, batch, d_out, plan)
        sus_n, sus_ms = 0, 0.0
        t_pre = time.perf_counter()
        while time.perf_counter() - t_pre < args.sustain_s:
            sus_ms += time_steps(torch, run, 10, 0, None)
            sus_n += 10
        clocks = sampler.stop() if rank == 0 else None
        ms_per_step = ms / args.steps
        total_pixels = FT * PIX
        if dist is not None:
            tp = torch.tensor([pixels], dtype=torch.float64, device="cuda")
            dist.all_reduce(tp)
            total_pixels = float(tp.item())
        value = total_pixels / (ms_per_step * 1e-3) / 1e6
        kern = kernel_name(plan, batch.n)
        ach = (in_b + out_b) / (ms_per_step * 1e-3) / 1e9  # this GPU; one plan run per step
        roofline = {"bound": "hbm", "kernel": kern, "achieved": ach, "peak": peak, "unit": "GB/s",
                    "frac": ach / peak, "traffic": None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": in_b + out_b,
                    "algorithmic_bytes_per_pixel": (in_b + out_b) / pixels,
                    "read_only_frac": (in_b / (ms_per_step * 1e-3) / 1e9) / peak,
                    "launches_per_step": plan.launches,
                    "note": "in+out accounting of SURVEY 8(d): compressed bytes read once + 2 B/pixel written "
                            "once; read_only_frac = compressed bytes only (north_star's wording) -- the 2 B/pixel "
                            "of output cap it at ~0.34 when the in+out fraction is 1"}
        tr = ncu_traffic(kern.split(" ")[0])
        if tr:
            roofline["traffic"] = tr["dram_bytes_per_frame"] * batch.n
            roofline["traffic_source"] = tr["source"]
        sustained = None
        if sus_n:
            sp = sus_ms / sus_n
            sustained = {"ms_per_step": sp, "steps": sus_n, "value_this_gpu": pixels / (sp * 1e-3) / 1e6,
                         "frac": (in_b + out_b) / (sp * 1e-3) / 1e9 / peak,
                         "note": "same step back to back for %.1f s after the timed steps (rank-local)" % args.sustain_s}

        # ---------------- e2e: host buffers through the C-ABI call ----------------
        h_out = torch.empty(batch.out_bytes, dtype=torch.uint8, pin_memory=True)

        def e2e_step():
            plan.run_host(batch.h_in.numpy()[:batch.in_bytes], h_out.numpy())
        e2e_steps = 3
        ms_e = wall_steps(torch, e2e_step, e2e_steps, 1, dist)
        e2e = {"value": total_pixels * e2e_steps / (ms_e * 1e-3) / 1e6, "unit": "MPixels/s",
               "h2d_bytes_per_step": int(batch.in_bytes), "d2h_bytes_per_step": int(batch.out_bytes),
               "steps": e2e_steps, "ms_per_step": ms_e / e2e_steps,
               "api": "rsb200_plan_run_host: pinned host buffers; upload, decode and download of consecutive "
                      "groups of tiles (8-32 MB of pixels) overlap on eight streams"}
        got = d_out.cpu().numpy()
        e2e["bit_exact"] = bool(np.array_equal(h_out.numpy()[:H * batch.out_pitch], got[:H * batch.out_pitch])) and \
            bool(np.array_equal(h_out.numpy()[(batch.n - 1) * batch.ob:(batch.n - 1) * batch.ob + H * batch.out_pitch],
                                got[(batch.n - 1) * batch.ob:(batch.n - 1) * batch.ob + H * batch.out_pitch]))
        del got

        gather = None
        if dist is not None:
            gather = bench_gather_abi(torch, dist, rs, ctx, batch, world, rank, args, total_pixels)
        del h_out

        single = None
        others = {}
        if rank == 0 and not args.skip_single:
            single = bench_single_frame(torch, rs, ctx, port, synth, args, shm, cap, recs, peak, peak_src)
        if not args.skip_others:
            if args.all_legs:
                others = bench_others(torch, rs, ctx, port, synth, args, dist, peak)
            elif rank == 0 or dist is not None:
                others = bench_core_others(torch, rs, ctx, port, synth, args, dist, peak)

        if rank == 0:
            cpu = None
            if not args.skip_cpu:
                cpu = cpu_baseline_children(args)
                c1 = cpu_reference_c1()
                if c1:
                    others["configs[0] 12-bit packed 4000x3000, CPU only"] = c1
            line = {
                "metric": "MPixels/s decoded (bit-exact)", "value": value, "unit": "MPixels/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "u16", "data": "synthetic",
                "config": {"workload": "configs[4]: %d-frame batch of configs[2] frames (DNG lossless-JPEG predictor 1, "
                                       "14-bit 8256x5504 = 45 MP, 726 tiles of 256x256 each, distinct frames "
                                       "seeds %d..%d), sharded %d frames per GPU over %d GPU(s), one plan run per step"
                                       % (FT, SEED0, SEED0 + FT - 1, per, world),
                           "frames_total": FT, "frames_per_gpu": per,
                           "bytes_per_step_per_gpu": in_b + out_b,
                           "compressed_bytes_per_pixel": in_b / pixels,
                           "l2": "inputs+outputs of one step (%.1f GB per GPU) exceed the 126 MB L2; no flush needed"
                                 % ((in_b + out_b) / 1e9),
                           "parallelism": "frames sharded across ranks (contiguous blocks of 256/N), no data-path "
                                          "collective in `value`; the NVLink output gather is `gather`",
                           "frame_synthesis_s": round(t_gen, 1)},
                "bit_exact": bit_exact, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
                "gpu_launches": int(launches), "clocks": clocks, "sustained": sustained,
                "single_frame": single, "others": others,
            }
            if gather:
                line["gather"] = gather
            print(json.dumps(line))
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
    finally:
        shm.close()
        shm.unlink()


def kernel_name(plan, nframes):
    return plan.kernels


def _cpulist(text):
    out = []
    for part in text.strip().split(","):
        if "-" in part:
            a, b = part.split("-")
            out += list(range(int(a), int(b) + 1))
        elif part:
            out.append(int(part))
    return out


def gpu_numa_cpus(local):
    """The CPUs of the NUMA node GPU `local` hangs off: its PCI address from nvidia-smi (the
    CUDA_VISIBLE_DEVICES order is the order nvidia-smi lists the visible GPUs in), the node from
    sysfs.  None when any of that is unavailable."""
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.split()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = local
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if all(v.isdigit() for v in ids) and local < len(ids):
                idx = int(ids[local])
        bus = q[idx].lower()
        if len(bus.split(":")[0]) == 8:      # nvidia-smi prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        return _cpulist(open("/sys/devices/system/node/node%d/cpulist" % node).read())
    except Exception:
        return None


def pin_rank_to_numa(local):
    """Keep this rank's threads, and therefore its pinned staging buffers (first touch), on the cores
    of the NUMA node its GPU hangs off (sysfs; r2_run15: on a 4-GPU allocation GPUs 2 and 3 sit on
    node 1).  Fallback when sysfs / nvidia-smi do not tell: GPUs 0-3 on node 0, 4-7 on node 1 (the
    8-GPU boxes, SCALE_r01.json topology)."""
    try:
        ncpu = os.cpu_count() or 1
        if ncpu < 64 or not hasattr(os, "sched_setaffinity"):
            return
        cores = gpu_numa_cpus(local)
        if not cores:
            half, q = ncpu // 2, ncpu // 4
            node = 0 if local < 4 else 1
            cores = list(range(node * q, (node + 1) * q)) + list(range(half + node * q, half + (node + 1) * q))
        os.sched_setaffinity(0, cores)
    except Exception:
        pass


def bench_gather_abi(torch, dist, rs, ctx, batch, world, rank, args, total_pixels):
    """north_star's NVLink output gather through the C ABI (rsb200_plan_run_gather): the slab of a
    group of tiles travels on the communicator's stream while the next groups decode.  Two
    modes: every rank gets everything / only the consumer GPU (rank 0) does."""
    uid = [rs.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    comm = rs.Comm(ctx, uid[0], world, rank)
    slab = batch.out_bytes
    d_all = torch.zeros(world * slab, dtype=torch.uint8, device="cuda")
    out = {"what": "decode + gather of the uint16 images over NVLink (rsb200_plan_run_gather: per group of "
                   "tiles (or per 512 MB of the slab when the plan is one launch), grouped ncclSend/ncclRecv on a side stream)",
           "gathered_bytes_total": int(world * slab)}
    for name, mode in (("to_all_ranks", rs.GATHER_ALL), ("to_rank0", rs.GATHER_ROOT)):
        def step():
            batch.plan.run_gather(comm, (batch.d_in.data_ptr(), batch.in_bytes), d_all, slab, mode, 0)
        n = 3
        ms = time_steps(torch, step, n, 1, dist) / n
        recv = (world - 1) * slab
        out[name] = {"ms_per_step": ms, "MPixels/s": total_pixels / (ms * 1e-3) / 1e6,
                     "received_bytes_busiest_gpu": int(recv),
                     "ingress_GBps_busiest_gpu": recv / (ms * 1e-3) / 1e9}
    # parity of the gathered data: slab r of rank 0 == what rank r decoded (checksum of the first frame)
    torch.cuda.synchronize()
    mine = d_all[rank * slab:rank * slab + 1024 * 1024].to(torch.int64).sum()
    sums = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(sums, mine)
    ok = True
    if rank == 0:
        for r in range(world):
            ok = ok and int(d_all[r * slab:r * slab + 1024 * 1024].to(torch.int64).sum().item()) == int(sums[r].item())
    out["gathered_matches_the_owners"] = bool(ok)
    out["bound"] = ("the consumer GPU receives (N-1)/N of %.1f GB; at the 900 GB/s per direction of NVLink 5 that "
                    "alone is %.1f ms" % (world * slab / 1e9, (world - 1) * slab / 900e9 * 1e3))
    comm.close()
    del d_all
    return out


def bench_single_frame(torch, rs, ctx, port, synth, args, shm, cap, recs, peak, peak_src):
    """BASELINE configs[2]: ONE 8256x5504 DNG LJPEG frame (726 tiles): device-timed decode,
    roofline, host-buffer runs (pinned / pageable) and the drop-in call of the host mirror."""
    from rawspeed_b200 import host
    b1 = LJpegBatch(torch, rs, ctx, shm, cap, recs[:1])
    d_out = torch.zeros(b1.out_bytes, dtype=torch.uint8, device="cuda")
    plan = b1.plan
    plan.run((b1.d_in.data_ptr(), b1.in_bytes), d_out)
    st = plan.results()
    img = synth.image_model(W, H, recs[0][0])
    got = d_out.cpu().numpy().view(np.uint16).reshape(H, b1.out_pitch // 2)
    exact = bool(np.array_equal(got[:, :W], img)) and all(s == 0 for s, _ in st)
    # the launch is shorter than the L2 flush would be meaningful for: flush L2 between runs by
    # writing a 256 MB buffer (not timed: CUDA events around the decode only)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ts = []
    for i in range(3 + 20):
        flush.fill_(i & 0xFF)
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        plan.run((b1.d_in.data_ptr(), b1.in_bytes), d_out)
        e1.record()
        torch.cuda.synchronize()
        if i >= 3:
            ts.append(e0.elapsed_time(e1))
    ms = float(np.mean(ts))
    ms_warm = time_steps(torch, lambda: plan.run((b1.d_in.data_ptr(), b1.in_bytes), d_out), 20, 3, None) / 20
    in_b, out_b, pixels = plan.bytes()
    ent = {"workload": "configs[2]: DNG lossless-JPEG predictor 1, 8256x5504, 726 tiles 256x256, ONE frame per launch",
           "MPixels/s": pixels / (ms * 1e-3) / 1e6, "ms_per_frame": ms, "bit_exact": exact,
           "timing": "CUDA events around each launch, L2 flushed (256 MB write) between launches, mean of 20",
           "ms_per_frame_back_to_back": ms_warm,
           "kernel": kernel_name(plan, 1), "launches_per_frame": plan.launches,
           "compressed_bytes_per_pixel": in_b / pixels,
           "roofline": {"bound": "hbm", "achieved": (in_b + out_b) / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": (in_b + out_b) / (ms * 1e-3) / 1e9 / peak,
                        "read_only_frac": in_b / (ms * 1e-3) / 1e9 / peak, "peak_source": peak_src,
                        "traffic": None}}
    tr = ncu_traffic(ent["kernel"].split(" ")[0])
    if tr:
        ent["roofline"]["traffic"] = tr["dram_bytes_per_frame"]
        ent["roofline"]["traffic_source"] = tr["source"]
    del flush
    # host buffers through the C ABI: pinned and pageable
    h_out = torch.empty(b1.out_bytes, dtype=torch.uint8, pin_memory=True)
    n = 5
    ms_p = wall_steps(torch, lambda: plan.run_host(b1.h_in.numpy()[:b1.in_bytes], h_out.numpy()), n, 2) / n
    ok_p = bool(np.array_equal(h_out.numpy()[:H * b1.out_pitch].view(np.uint16).reshape(H, -1)[:, :W], img))
    pg_in = np.array(b1.h_in.numpy()[:b1.in_bytes])
    pg_out = np.zeros(b1.out_bytes, dtype=np.uint8)
    ms_g = wall_steps(torch, lambda: plan.run_host(pg_in, pg_out), n, 2) / n
    ent["e2e"] = {"value": pixels / (ms_p * 1e-3) / 1e6, "unit": "MPixels/s", "ms_per_frame": ms_p,
                  "h2d_bytes_per_step": int(b1.in_bytes), "d2h_bytes_per_step": int(b1.out_bytes),
                  "bit_exact": ok_p, "api": "rsb200_plan_run_host, pinned host buffers, pipelined groups",
                  "pageable": {"value": pixels / (ms_g * 1e-3) / 1e6, "ms_per_frame": ms_g}}
    # the drop-in call: the host mirror's AbstractDngDecompressor::decompress() -- marker walk of
    # every tile, table validation, plan, upload, decode, download, per-tile results
    r = recs[0]
    blob = np.array(b1.h_in.numpy()[:r[1]])
    himg = port.new_image(W, H)
    host.dng_decompress(blob, r[6], r[7], himg, W, 1, 256, 256, 7)
    ok_m = bool(np.array_equal(himg[:, :W], img))
    inner = []

    def mirror_call():
        host.dng_decompress(blob, r[6], r[7], himg, W, 1, 256, 256, 7)
        inner.append(host.last_call_ms())
    ms_h = wall_steps(torch, mirror_call, n, 1) / n
    ms_m = float(np.median(inner[1:]))
    ent["e2e_host_mirror"] = {"value": PIX / (ms_m * 1e-3) / 1e6, "unit": "MPixels/s", "ms_per_frame": ms_m,
                              "ms_per_frame_with_test_harness": ms_h, "bit_exact": ok_m,
                              "api": "rawspeed_b200::AbstractDngDecompressor::decompress() (C++ host mirror, pageable "
                                     "RawImage): parse + plan + H2D + decode + D2H + results, per call; timed "
                                     "around the member call (the ctypes harness around it allocates a RawImage "
                                     "and copies the numpy image in and out: ms_per_frame_with_test_harness)"}
    return ent


def bench_core_others(torch, rs, ctx, port, synth, args, dist, peak):
    """The other BASELINE configs, short: configs[1] (14-bit packed unpack, 8 frames per launch)
    and configs[3] (CR2 6720x4480, 3 slices)."""
    out = {}
    F = args.frames
    data, pitch = synth.packed_frame(W, H, BPS, seed=2)
    out_pitch = rs.image_pitch(W)
    in_fb, out_fb = align(pitch * H), align(out_pitch * H)
    d_in = torch.zeros(F * in_fb, dtype=torch.uint8, device="cuda")
    base = torch.from_numpy(data).cuda()
    for f in range(F):
        d_in[f * in_fb:f * in_fb + pitch * H] = torch.roll(base, f * 7919)
    d_out = torch.zeros(F * out_fb, dtype=torch.uint8, device="cuda")
    plan = rs.unpack_plan(ctx, unpack_jobs(rs, F, in_fb, out_fb, pitch, out_pitch, rs.MSB))
    plan.run(d_in, d_out)
    want = port.new_image(W, H)
    port.unpack(data, want, W, 1, (0, 0, W, H), pitch, BPS, port.MSB)
    got = d_out[:out_pitch * H].cpu().numpy().view(np.uint16).reshape(H, out_pitch // 2)
    exact = bool(np.array_equal(got[:, :W], want[:, :W]))
    n = max(5, min(args.steps, 20))
    ms = time_steps(torch, lambda: plan.run(d_in, d_out), n, 3, dist) / n
    in_b, out_b, pixels = plan.bytes()
    out["configs[1] 14-bit packed (MSB) unpack 8256x5504, %d frames per launch" % F] = {
        "MPixels/s": pixels / (ms * 1e-3) / 1e6, "ms_per_step": ms, "bit_exact": exact,
        "kernel": "unpack_fast_kernel<14,MSB>", "achieved_GBps": (in_b + out_b) / (ms * 1e-3) / 1e9,
        "roofline_frac": (in_b + out_b) / (ms * 1e-3) / 1e9 / peak}
    del plan, d_in, d_out, base
    from helpers import TableSet
    from test_gpu_cr2 import cr2_job
    cw, ch = 6720, 4480
    cimg = port.new_image(cw, ch)
    cimg[:, :cw] = synth.image_model(cw, ch, 4)
    hts = synth.default_tables(2)
    fmt, frame = (2, 1, 1), (3360, 4480)
    blob = port.cr2_encode(cimg, cw, fmt, frame, (3, 2240, 2240), 14, hts, [0, 1])
    ts = TableSet()
    job = cr2_job(blob, cw, ch, fmt, (3, 2240, 2240), cimg.shape[1] * 2, ts)
    plan = rs.cr2_plan(ctx, ts.tabs, [job])
    d_in = torch.zeros(blob.size + 64, dtype=torch.uint8, device="cuda")
    d_in[:blob.size] = torch.from_numpy(blob)
    d_out = torch.zeros(cimg.size * 2, dtype=torch.uint8, device="cuda")
    plan.run((d_in.data_ptr(), blob.size), d_out)
    res = plan.results()
    got = d_out.cpu().numpy().view(np.uint16).reshape(cimg.shape)
    exact = bool(np.array_equal(got[:, :cw], cimg[:, :cw])) and res[0][0] == 0
    ms = time_steps(torch, lambda: plan.run((d_in.data_ptr(), blob.size), d_out), 5, 2, dist) / 5
    ent = {"MPixels/s": cw * ch / (ms * 1e-3) / 1e6, "ms_per_frame": ms, "bit_exact": exact,
           "kernels": "k2_range_count/verify/diffs + k3_column/row"}
    if not args.skip_cpu and int(os.environ.get("RANK", "0")) == 0:
        import oracle
        if oracle.HAVE_REF:
            tmp = port.new_image(cw, ch)
            msr = min(oracle.ref.cr2_ljpeg_decode(blob, tmp, cw, (3, 2240, 2240), reps=1) for _ in range(2))
            ent["cpu_reference"] = {"kind": "reference", "cores": 1, "MPixels/s": cw * ch / (msr * 1e-3) / 1e6,
                                    "sample": "Cr2LJpegDecoder::decode (single threaded by design)"}
    out["configs[3] CR2 6720x4480 3 slices <2,1,1>"] = ent
    return out


def bench_gather(torch, dist, d_out, world, rank, plan, d_in, args, frames, out_fb):
    """north_star's NVLink output gather (every rank ends up with all decoded
    frames), timed separately from the decode: rawspeed_b200.shard.gather_frames
    = one NCCL all_gather on the decode stream."""
    from rawspeed_b200 import shard
    local = d_out.view(frames, out_fb)
    gathered = torch.empty((world, frames, out_fb), dtype=torch.uint8, device="cuda")

    def step():
        plan.run(d_in, d_out)
        # copy-free form: preallocated result, the collective's own layout (frame r + k*world at [r, k])
        shard.gather_frames(local, frames * world, dist, out=gathered, reorder=False)
    n = max(2, min(args.steps, 5))
    ms = time_steps(torch, step, n, 1, dist)
    total = frames * world * out_fb
    return {"what": "decode + ncclAllGather of the uint16 outputs over NVLink (all ranks get all frames)",
            "ms_per_step": ms / n, "gathered_bytes_per_rank": int(total),
            "MPixels/s": world * frames * PIX / (ms / n * 1e-3) / 1e6,
            "busbw_GBps": (total * (world - 1) / world) / (ms / n * 1e-3) / 1e9}


def bench_others(torch, rs, ctx, port, synth, args, dist, peak):
    """configs[2] (DNG LJPEG tiles) and configs[3] (CR2): device-timed decode."""
    from helpers import dng_ljpeg_scans, parse_ljpeg, TableSet
    if args.unvalidated and args.only_unvalidated:
        return bench_unvalidated(torch, rs, ctx, port, synth, args, dist, peak)
    out = {}
    steps = max(3, min(args.steps, 10))
    # ---- C3: 8256x5504 DNG, 726 LJPEG tiles of 256x256, 2 components ----
    img = synth.image_model(W, H, 12345)
    t = synth.make_dng_ljpeg(img, 256, 256)
    out_pitch = rs.image_pitch(W)
    tabs, scans = dng_ljpeg_scans(t, out_pitch)
    plan = rs.ljpeg_plan(ctx, tabs.tabs, scans)
    d_in = torch.zeros(t.blob.size + 64, dtype=torch.uint8, device="cuda")
    d_in[:t.blob.size] = torch.from_numpy(t.blob)
    d_out = torch.zeros(H * out_pitch, dtype=torch.uint8, device="cuda")
    plan.run((d_in.data_ptr(), t.blob.size), d_out)
    res = plan.results()
    got = d_out.cpu().numpy().view(np.uint16).reshape(H, out_pitch // 2)
    exact = bool(np.array_equal(got[:, :W], img)) and all(s == 0 for s, _ in res)
    ms = time_steps(torch, lambda: plan.run((d_in.data_ptr(), t.blob.size), d_out), steps, 3, dist)
    in_b, out_b, pixels = plan.bytes()
    per = ms / steps
    c3 = {
        "MPixels/s": pixels / (per * 1e-3) / 1e6, "ms_per_frame": per, "bit_exact": exact,
        "compressed_bytes_per_pixel": t.blob.size / PIX,
        "achieved_GBps": (in_b + out_b) / (per * 1e-3) / 1e9,
        "roofline_frac": (in_b + out_b) / (per * 1e-3) / 1e9 / peak,
        "read_only_roofline_frac": in_b / (per * 1e-3) / 1e9 / peak,
        "kernel": "k2_fused_kernel", "launches_per_frame": plan.launches}
    out["configs[2] DNG LJPEG 8256x5504 (726 tiles 256x256)"] = c3
    del plan, d_out
    # ---- C5-style batches: NB frames of C3 resident in HBM, one plan per batch ----
    # 8 frames stay on the block-per-segment kernel (K2F); from ~22 frames (16384 segments)
    # the plan switches to the one-thread-per-segment path (K2C unstuff pre-pass + K2T).
    world = int(os.environ.get("WORLD_SIZE", "1"))
    fb = (t.blob.size + 255) // 256 * 256
    ob = (H * out_pitch + 255) // 256 * 256
    batches = [max(1, 256 // world)] if args.c5 else sorted({args.ljpeg_frames, args.ljpeg_big_frames})
    for NB in batches:
        d_inb = torch.zeros(NB * fb + 64, dtype=torch.uint8, device="cuda")
        scans_b = []
        for f in range(NB):
            d_inb[f * fb:f * fb + t.blob.size] = d_in[:t.blob.size]
            for s0 in scans:
                s1 = rs.LJpegScan.from_buffer_copy(s0)
                s1.in_offset = s0.in_offset + f * fb
                s1.out_offset = s0.out_offset + f * ob
                scans_b.append(s1)
        planb = rs.ljpeg_plan(ctx, tabs.tabs, scans_b)
        d_outb = torch.zeros(NB * ob, dtype=torch.uint8, device="cuda")
        planb.run((d_inb.data_ptr(), NB * fb), d_outb)
        resb = planb.results()
        exact_b = all(s_ == 0 for s_, _ in resb)
        for f in sorted({0, NB // 2, NB - 1}):
            gb = d_outb[f * ob:f * ob + H * out_pitch].cpu().numpy().view(np.uint16).reshape(H, out_pitch // 2)
            exact_b = exact_b and bool(np.array_equal(gb[:, :W], img))
        nst = max(3, min(steps, 5))
        msb = time_steps(torch, lambda: planb.run((d_inb.data_ptr(), NB * fb), d_outb), nst, 3, dist)
        in_bb, out_bb, pix_b = planb.bytes()
        perb = msb / nst
        kern = "k2_fused_kernel" if planb.launches == 1 else "k2_clean_kernel + k2_thread_kernel"
        label = ("configs[4]: 256-frame LJPEG batch, %d frames per GPU x %d GPUs, one plan per GPU"
                 % (NB, world)) if args.c5 else \
            "configs[4]-style batch: %d LJPEG frames of configs[2] per GPU, one plan" % NB
        entb = {
            "MPixels/s_per_gpu": pix_b / (perb * 1e-3) / 1e6, "ms_per_step": perb, "bit_exact": exact_b,
            "kernels": kern, "launches_per_step": planb.launches,
            "achieved_GBps": (in_bb + out_bb) / (perb * 1e-3) / 1e9,
            "roofline_frac": (in_bb + out_bb) / (perb * 1e-3) / 1e9 / peak,
            "read_only_roofline_frac": in_bb / (perb * 1e-3) / 1e9 / peak}
        if args.c5:
            entb["MPixels/s_all_gpus"] = world * pix_b / (perb * 1e-3) / 1e6
            entb["frames"] = NB * world
            entb["note"] = ("the 256 frames are copies of one synthetic frame (same statistics; generating "
                            "256 distinct frames on the host would take minutes); ms_per_step is the max "
                            "over ranks")
            if dist is not None:
                from rawspeed_b200 import shard
                local = d_outb.view(NB, ob)
                gathered = torch.empty((world, NB, ob), dtype=torch.uint8, device="cuda")

                def step_g():
                    planb.run((d_inb.data_ptr(), NB * fb), d_outb)
                    shard.gather_frames(local, NB * world, dist, out=gathered, reorder=False)
                msg = time_steps(torch, step_g, 3, 1, dist)
                entb["decode_plus_gather_ms"] = msg / 3
                entb["decode_plus_gather_MPixels/s"] = world * pix_b / (msg / 3 * 1e-3) / 1e6
                entb["gather"] = ("one ncclAllGather of the uint16 outputs into a preallocated "
                                  "[world, frames_per_gpu, frame] buffer on every rank (frame r + k*world "
                                  "at [r, k]); %.1f GB received per GPU" % ((world - 1) * NB * ob / 1e9))
                del gathered
        out[label] = entb
        del planb, d_inb, d_outb
    del d_in
    if not args.skip_cpu and int(os.environ.get("RANK", "0")) == 0:
        import oracle
        if oracle.HAVE_REF:
            ncores = os.cpu_count() or 1
            tmp = port.new_image(W, H)
            ms_cpu = min(oracle.ref.dng_decompress(t.blob, t.offsets, t.lengths, tmp, W, 1, 256, 256, 7,
                                                   nthreads=ncores, reps=1) for _ in range(3))
            ms_1 = oracle.ref.dng_decompress(t.blob, t.offsets, t.lengths, tmp, W, 1, 256, 256, 7,
                                             nthreads=1, reps=1)
            c3["cpu_reference"] = {"kind": "reference", "cores": ncores,
                                   "MPixels/s": PIX / (ms_cpu * 1e-3) / 1e6,
                                   "single_thread_MPixels/s": PIX / (ms_1 * 1e-3) / 1e6,
                                   "sample": "AbstractDngDecompressor::decompress() (OpenMP over the 726 "
                                             "tiles), 1 frame, best of 3"}
    # ---- C4: CR2 6720x4480, 3 slices, 2 and 4 components ----
    from test_gpu_cr2 import cr2_job
    cw, ch = 6720, 4480
    cimg = port.new_image(cw, ch)
    cimg[:, :cw] = synth.image_model(cw, ch, 4)
    hts = synth.default_tables(2)
    for fmt, frame in [((2, 1, 1), (3360, 4480)), ((4, 1, 1), (1680, 4480))]:
        blob = port.cr2_encode(cimg, cw, fmt, frame, (3, 2240, 2240), 14, hts, [0, 1, 0, 1][:fmt[0]])
        ts = TableSet()
        job = cr2_job(blob, cw, ch, fmt, (3, 2240, 2240), cimg.shape[1] * 2, ts)
        plan = rs.cr2_plan(ctx, ts.tabs, [job])
        d_in = torch.zeros(blob.size + 64, dtype=torch.uint8, device="cuda")
        d_in[:blob.size] = torch.from_numpy(blob)
        d_out = torch.zeros(cimg.size * 2, dtype=torch.uint8, device="cuda")
        plan.run((d_in.data_ptr(), blob.size), d_out)
        res = plan.results()
        got = d_out.cpu().numpy().view(np.uint16).reshape(cimg.shape)
        exact = bool(np.array_equal(got[:, :cw], cimg[:, :cw])) and res[0][0] == 0
        ms = time_steps(torch, lambda: plan.run((d_in.data_ptr(), blob.size), d_out), 3, 1, dist)
        per = ms / 3
        ent = {"MPixels/s": cw * ch / (per * 1e-3) / 1e6, "ms_per_frame": per, "bit_exact": exact,
               "compressed_bytes_per_pixel": blob.size / (cw * ch),
               "kernels": "k2_range_count/verify/diffs + k3_column/row"}
        if not args.skip_cpu and int(os.environ.get("RANK", "0")) == 0:
            import oracle
            if oracle.HAVE_REF:
                tmp = port.new_image(cw, ch)
                msr = min(oracle.ref.cr2_ljpeg_decode(blob, tmp, cw, (3, 2240, 2240), reps=1)
                          for _ in range(2))
                ent["cpu_reference"] = {"kind": "reference", "cores": 1,
                                        "MPixels/s": cw * ch / (msr * 1e-3) / 1e6,
                                        "sample": "Cr2LJpegDecoder::decode (single threaded by design)"}
        out["configs[3] CR2 6720x4480 3 slices <%d,1,1>" % fmt[0]] = ent
        del plan, d_in, d_out
    out.update(bench_forms(torch, rs, ctx, port, synth, args, dist, peak))
    out.update(bench_codecs(torch, rs, ctx, port, synth, args, dist, peak))
    if args.unvalidated:
        out.update(bench_unvalidated(torch, rs, ctx, port, synth, args, dist, peak))
    return out


def bench_codecs(torch, rs, ctx, port, synth, args, dist, peak):
    """SURVEY 8(f)2/4: Canon sRaw interpolation, the Pentax PEF codec, Sony ARW2; device-timed."""
    out = {}
    steps = max(3, min(args.steps, 10))
    rank0 = int(os.environ.get("RANK", "0")) == 0
    # ---- Cr2sRawInterpolator, 4:2:0 version 2, 5040x3360 RGB output (mRAW class) ----
    num_mcus, rows = 2520, 1680
    rng = np.random.default_rng(5)
    in_w = num_mcus * 6
    pitch = (in_w * 2 + 15) // 16 * 16
    inp = np.zeros((rows, pitch // 2), dtype=np.uint16)
    inp[:, :in_w] = rng.integers(0, 16384, (rows, in_w), dtype=np.uint16)
    out_w, out_h = 2 * num_mcus, 2 * rows
    want = port.new_image(out_w, out_h, 3)
    j = rs.SrawJob()
    j.in_offset, j.in_pitch, j.num_mcus, j.in_rows = 0, pitch, num_mcus, rows
    j.sub_x, j.sub_y, j.version = 2, 2, 2
    j.sraw_coeffs[0], j.sraw_coeffs[1], j.sraw_coeffs[2] = 2000, 1024, 1500
    j.hue, j.out_offset, j.out_pitch = 0, 0, want.shape[1] * 2
    plan = rs.sraw_plan(ctx, [j])
    d_in = torch.from_numpy(inp.view(np.int16)).cuda()
    d_out = torch.from_numpy(want.view(np.int16).copy()).cuda()
    plan.run(d_in, d_out)
    torch.cuda.synchronize()
    port.sraw_interpolate(inp, in_w, want, out_w, (2, 2), (2000, 1024, 1500), 0, 2)
    exact = bool(np.array_equal(d_out.cpu().numpy().view(np.uint16), want))
    ms = time_steps(torch, lambda: plan.run(d_in, d_out), steps, 3, dist)
    in_b, out_b, pixels = plan.bytes()
    per = ms / steps
    ent = {"MPixels/s": pixels / (per * 1e-3) / 1e6, "ms_per_frame": per, "bit_exact": exact,
           "achieved_GBps": (in_b + out_b) / (per * 1e-3) / 1e9,
           "roofline_frac": (in_b + out_b) / (per * 1e-3) / 1e9 / peak, "kernel": "sraw_kernel<2,420>"}
    if not args.skip_cpu and rank0:
        import oracle
        if oracle.HAVE_REF:
            ncores = os.cpu_count() or 1
            tmp = want.copy()
            msr = min(oracle.ref.sraw_interpolate(inp, in_w, tmp, out_w, (2, 2), (2000, 1024, 1500), 0, 2,
                                                  nthreads=ncores) for _ in range(3))
            ent["cpu_reference"] = {"kind": "reference", "cores": ncores,
                                    "MPixels/s": pixels / (msr * 1e-3) / 1e6,
                                    "sample": "Cr2sRawInterpolator::interpolate(2), OpenMP rows, best of 3"}
    out["8(f)2 Cr2sRawInterpolator 4:2:0 -> 5040x3360 RGB"] = ent
    del plan, d_in, d_out
    # ---- PentaxDecompressor, 6016x4000 (K-3 class), legacy table ----
    w, h = 6016, 4000
    table = port.pentax_table(None)
    img = (synth.image_model(w, h, seed=11, bits=12) & 0x0FFF).astype(np.uint16)
    data = synth.make_pentax(img, table)
    got0 = port.new_image(w, h)
    pj = rs.PentaxJob()
    pj.in_offset, pj.in_size, pj.table, pj.width, pj.height = 0, data.size, 0, w, h
    pj.out_offset, pj.out_pitch = 0, got0.shape[1] * 2
    plan = rs.pentax_plan(ctx, [rs.huff_table(table[0], table[1])], [pj])
    d_in = torch.zeros(data.size + 64, dtype=torch.uint8, device="cuda")
    d_in[:data.size] = torch.from_numpy(data)
    d_out = torch.from_numpy(got0.view(np.int16).copy()).cuda()
    plan.run((d_in.data_ptr(), data.size), d_out)
    res = plan.results()
    exact = bool(np.array_equal(d_out.cpu().numpy().view(np.uint16)[:, :w], img)) and res[0][0] == 0
    ms = time_steps(torch, lambda: plan.run((d_in.data_ptr(), data.size), d_out), 3, 1, dist)
    per = ms / 3
    ent = {"MPixels/s": w * h / (per * 1e-3) / 1e6, "ms_per_frame": per, "bit_exact": exact,
           "compressed_bytes_per_pixel": data.size / (w * h),
           "kernels": "k2_range_count/verify/diffs (plain MSB pump) + k3p_column/row"}
    if not args.skip_cpu and rank0:
        import oracle
        if oracle.HAVE_REF:
            tmp = port.new_image(w, h)
            msr = min(oracle.ref.pentax_decompress(tmp, w, data) for _ in range(2))
            ent["cpu_reference"] = {"kind": "reference", "cores": 1,
                                    "MPixels/s": w * h / (msr * 1e-3) / 1e6,
                                    "sample": "PentaxDecompressor::decompress (single threaded by design)"}
    out["8(f)2 PentaxDecompressor 6016x4000"] = ent
    del plan, d_in, d_out
    # ---- NikonDecompressor (no split), 6032x4032 14-bit, curve + dither ----
    w, h = 6032, 4032
    half = 1 << 13
    pup = [half, half + 2, half - 8, half - 2]
    meta = synth.nikon_meta("table", 14, (pup[0], pup[2], pup[1], pup[3]), True)
    su = port.nikon_setup(meta, True, 14, w, h)
    img = (synth.image_model(w, h, seed=7, bits=14) & 0x3FFF).astype(np.uint16)
    data = synth.make_nikon(img, su["huff_select"], pup)
    ncpl, values = port.nikon_tree(su["huff_select"])
    nj = rs.NikonJob()
    nj.in_offset, nj.in_size, nj.table, nj.width, nj.height = 0, data.size, 0, w, h
    nj.out_offset, nj.out_pitch, nj.lut = 0, rs.image_pitch(w), 0
    for k in range(4):
        nj.pup[k] = pup[k]
    plan = rs.nikon_plan(ctx, [rs.huff_table(ncpl, values)], [nj], port.build_table(su["curve"], True))
    d_in = torch.zeros(data.size + 64, dtype=torch.uint8, device="cuda")
    d_in[:data.size] = torch.from_numpy(data)
    d_out = torch.zeros(h * rs.image_pitch(w), dtype=torch.uint8, device="cuda")
    plan.run((d_in.data_ptr(), data.size), d_out)
    res = plan.results()
    want = port.new_image(w, h)
    port.nikon_decompress(want, w, meta, True, 14, data)
    exact = bool(np.array_equal(d_out.cpu().numpy().view(np.uint16).reshape(want.shape), want)) and res[0][0] == 0
    ms = time_steps(torch, lambda: plan.run((d_in.data_ptr(), data.size), d_out), 3, 1, dist)
    per = ms / 3
    ent = {"MPixels/s": w * h / (per * 1e-3) / 1e6, "ms_per_frame": per, "bit_exact": exact,
           "compressed_bytes_per_pixel": data.size / (w * h),
           "kernels": "k2_range_count/verify/diffs (plain MSB pump) + k3n_column/row (curve + dither)"}
    if not args.skip_cpu and rank0:
        import oracle
        if oracle.HAVE_REF:
            tmp = port.new_image(w, h)
            msr = min(oracle.ref.nikon_decompress(tmp, w, meta, True, 14, data) for _ in range(2))
            ent["cpu_reference"] = {"kind": "reference", "cores": 1,
                                    "MPixels/s": w * h / (msr * 1e-3) / 1e6,
                                    "sample": "NikonDecompressor::decompress (single threaded by design)"}
    out["8(f)2 NikonDecompressor 6032x4032 14-bit (curve + dither)"] = ent
    del plan, d_in, d_out
    # ---- PanasonicV5 (14 bit) / V6 (14 bit) / V7, 5184x3888-class frames, 4 frames per launch ----
    for ver, bps, w, h in ((5, 14, 5184, 3888), (6, 14, 5181, 3888), (7, 14, 5184, 3888)):
        npix = (11 if ver == 6 else 128 // bps)
        nunits = w * h // npix
        nbytes = ((nunits + 1023) // 1024) * 0x4000 if ver == 5 else nunits * 16
        data = synth.lcg_bytes(nbytes, 40 + ver)
        opitch = rs.image_pitch(w)
        nf = 4
        fb = (nbytes + 255) // 256 * 256
        ob = (h * opitch + 255) // 256 * 256
        jobs = []
        for f in range(nf):
            pj = rs.PanaJob()
            pj.in_offset, pj.in_size, pj.out_offset, pj.out_pitch = f * fb, nbytes, f * ob, opitch
            pj.width, pj.height, pj.version, pj.bps = w, h, ver, bps
            jobs.append(pj)
        plan = rs.pana_plan(ctx, jobs)
        d_in = torch.zeros(nf * fb + 64, dtype=torch.uint8, device="cuda")
        for f in range(nf):
            d_in[f * fb:f * fb + nbytes] = torch.from_numpy(data)
        d_out = torch.zeros(nf * ob, dtype=torch.uint8, device="cuda")
        plan.run((d_in.data_ptr(), nf * fb), d_out)
        torch.cuda.synchronize()
        want = port.new_image(w, h)
        port.panasonic(ver, want, w, data, bps)
        got = d_out[(nf - 1) * ob:(nf - 1) * ob + h * opitch].cpu().numpy().view(np.uint16).reshape(h, opitch // 2)
        exact = bool(np.array_equal(got[:, :w], want[:, :w]))
        ms = time_steps(torch, lambda: plan.run((d_in.data_ptr(), nf * fb), d_out), steps, 3, dist)
        in_b, out_b, pixels = plan.bytes()
        per = ms / steps
        ent = {"MPixels/s": pixels / (per * 1e-3) / 1e6, "ms_per_step": per, "frames_per_step": nf,
               "bit_exact": exact, "achieved_GBps": (in_b + out_b) / (per * 1e-3) / 1e9,
               "roofline_frac": (in_b + out_b) / (per * 1e-3) / 1e9 / peak,
               "kernel": "pana_kernel<%d,%d>" % (ver, bps)}
        if not args.skip_cpu and rank0:
            import oracle
            if oracle.HAVE_REF:
                ncores = os.cpu_count() or 1
                tmp = port.new_image(w, h)
                msr = min(oracle.ref.panasonic(ver, tmp, w, data, bps, nthreads=ncores) for _ in range(3))
                ent["cpu_reference"] = {"kind": "reference", "cores": ncores,
                                        "MPixels/s": w * h / (msr * 1e-3) / 1e6,
                                        "sample": "PanasonicV%dDecompressor::decompress (OpenMP), 1 frame, best of 3" % ver}
        out["8(f)4 PanasonicV%dDecompressor %dx%d %d-bit" % (ver, w, h, bps)] = ent
        del plan, d_in, d_out
    # ---- PhaseOneDecompressor, 11608x8708 (IQ3 100MP class): group headers per row, pixels in parallel ----
    w, h = 11608, 8708
    rowimg = (synth.image_model(w, 4, seed=31, bits=14)).astype(np.uint16)
    rows4 = [np.frombuffer(synth.phaseone_row(rowimg[k]), dtype=np.uint8) for k in range(4)]
    offs, blobs, pos = [], [], 0
    for r in range(h):   # the four encoded rows repeat down the image (rows are independent streams)
        offs.append((pos, rows4[r % 4].size, r))
        blobs.append(rows4[r % 4])
        pos += rows4[r % 4].size
    blob = np.concatenate(blobs)
    pj = rs.PhaseOneJob()
    pj.out_offset, pj.out_pitch, pj.width, pj.height, pj.first_strip = 0, rs.image_pitch(w), w, h, 0
    pstrips = []
    for off, size, row in offs:
        ps = rs.PhaseOneStrip()
        ps.in_offset, ps.in_size, ps.row = off, size, row
        pstrips.append(ps)
    plan = rs.phaseone_plan(ctx, [pj], pstrips)
    d_in = torch.zeros(blob.size + 64, dtype=torch.uint8, device="cuda")
    d_in[:blob.size] = torch.from_numpy(blob)
    d_out = torch.zeros(h * rs.image_pitch(w), dtype=torch.uint8, device="cuda")
    plan.run((d_in.data_ptr(), blob.size), d_out)
    res = plan.results()
    got = d_out.cpu().numpy().view(np.uint16).reshape(h, rs.image_pitch(w) // 2)
    exact = res[0][0] == 0 and all(bool(np.array_equal(got[k::4, :w], np.broadcast_to(rowimg[k], (len(range(k, h, 4)), w))))
                                   for k in range(4))   # every row of the frame
    ms = time_steps(torch, lambda: plan.run((d_in.data_ptr(), blob.size), d_out), 3, 1, dist)
    per = ms / 3
    ent = {"MPixels/s": w * h / (per * 1e-3) / 1e6, "ms_per_frame": per, "bit_exact": bool(exact),
           "compressed_bytes_per_pixel": blob.size / (w * h),
           "kernel": ("p1_kernel_v2 (one thread per row: 8708 threads, latency bound)"
                      if os.environ.get("RSB200_P1") in ("1", "2") else
                      "p1_walk_kernel (one thread per row reads the group headers) + p1_decode_kernel (one warp "
                      "per row, 32 groups per step, segmented scan of the predictors)")}
    if not args.skip_cpu and rank0:
        import oracle
        if oracle.HAVE_REF:
            ncores = os.cpu_count() or 1
            tmp = port.new_image(w, h)
            msr = min(oracle.ref.phaseone(tmp, w, blob, offs, nthreads=ncores) for _ in range(2))
            ent["cpu_reference"] = {"kind": "reference", "cores": ncores,
                                    "MPixels/s": w * h / (msr * 1e-3) / 1e6,
                                    "sample": "PhaseOneDecompressor::decompress (OpenMP over rows), best of 2"}
    out["8(f)4 PhaseOneDecompressor 11608x8708"] = ent
    del plan, d_in, d_out
    # ---- HasselbladDecompressor, 8272x6200 (H5D-50c class, 51 MP): one MSB32 pair stream per frame ----
    w, h = 8272, 6200
    himg = synth.image_model(w, 200, seed=41, bits=14)
    himg = np.tile(himg, (h // 200, 1))          # (rows restart their predictors: any rows will do)
    hht = port.Huff(synth.DEFAULT_NCPL, synth.DEFAULT_VALUES, full=False)
    hdata = synth.make_hasselblad_fast(himg, hht, 0x8000)
    hj = rs.HasselbladJob()
    hj.in_offset, hj.in_size, hj.width, hj.height = 0, hdata.size, w, h
    hj.out_pitch, hj.out_offset, hj.init_pred, hj.table = rs.image_pitch(w), 0, 0x8000, 0
    plan = rs.hasselblad_plan(ctx, [rs.huff_table(bytes(synth.DEFAULT_NCPL), bytes(synth.DEFAULT_VALUES), False)], [hj])
    d_in = torch.zeros(hdata.size + 64, dtype=torch.uint8, device="cuda")
    d_in[:hdata.size] = torch.from_numpy(hdata)
    d_out = torch.zeros(h * rs.image_pitch(w), dtype=torch.uint8, device="cuda")
    plan.run((d_in.data_ptr(), hdata.size), d_out)
    res = plan.results()
    got = d_out.cpu().numpy().view(np.uint16).reshape(h, rs.image_pitch(w) // 2)
    exact = res[0][0] == 0 and bool(np.array_equal(got[:, :w], himg))
    ms = time_steps(torch, lambda: plan.run((d_in.data_ptr(), hdata.size), d_out), steps, 3, dist)
    per = ms / steps
    ent = {"MPixels/s": w * h / (per * 1e-3) / 1e6, "ms_per_frame": per, "bit_exact": bool(exact),
           "compressed_bytes_per_pixel": hdata.size / (w * h), "launches_per_frame": plan.launches,
           "achieved_GBps": (hdata.size + 2 * w * h) / (per * 1e-3) / 1e9,
           "roofline_frac": (hdata.size + 2 * w * h) / (per * 1e-3) / 1e9 / peak,
           "kernel": "hass_parse/link x6 + scan + hass_decode + hass_rows (one thread per 2 KiB of stream)"}
    if not args.skip_cpu and rank0:
        tmp = port.new_image(w, h)
        t0 = time.perf_counter()
        port.hasselblad_decompress(tmp, w, hht, 0x8000, hdata)
        msr = (time.perf_counter() - t0) * 1e3
        ent["cpu_reference"] = {"kind": "port", "cores": 1, "MPixels/s": w * h / (msr * 1e-3) / 1e6,
                                "sample": "the oracle's HasselbladDecompressor restatement (single threaded by "
                                          "design: one stream), 1 frame"}
    out["8(f)2 HasselbladDecompressor 8272x6200"] = ent
    del plan, d_in, d_out
    # ---- SonyArw2Decompressor, 9568x6376 (61 MP, A7R IV class), dithered curve, 4 frames ----
    w, h, nf = 9568, 6376, 4
    data = synth.arw2_frame(w, h, seed=21)
    curve = synth.sony_curve()
    table = port.build_table(curve, True)
    opitch = rs.image_pitch(w)
    fb = (data.size + 255) // 256 * 256
    ob = (h * opitch + 255) // 256 * 256
    jobs = []
    for f in range(nf):
        aj = rs.Arw2Job()
        aj.in_offset, aj.out_offset, aj.out_pitch = f * fb, f * ob, opitch
        aj.width, aj.height, aj.table = w, h, 0
        jobs.append(aj)
    plan = rs.arw2_plan(ctx, jobs, table, True)
    d_in = torch.zeros(nf * fb + 64, dtype=torch.uint8, device="cuda")
    for f in range(nf):
        d_in[f * fb:f * fb + data.size] = torch.from_numpy(data)
    d_out = torch.zeros(nf * ob, dtype=torch.uint8, device="cuda")
    plan.run((d_in.data_ptr(), nf * fb), d_out)
    res = plan.results()
    want = port.new_image(w, h)
    port.sony_arw2(want, w, data, table, True)
    got = d_out[(nf - 1) * ob:(nf - 1) * ob + h * opitch].cpu().numpy().view(np.uint16).reshape(h, opitch // 2)
    exact = bool(np.array_equal(got, want)) and all(s_ == 0 for s_, _ in res)
    ms = time_steps(torch, lambda: plan.run((d_in.data_ptr(), nf * fb), d_out), steps, 3, dist)
    in_b, out_b, pixels = plan.bytes()
    per = ms / steps
    ent = {"MPixels/s": pixels / (per * 1e-3) / 1e6, "ms_per_step": per, "frames_per_step": nf,
           "bit_exact": exact, "achieved_GBps": (in_b + out_b) / (per * 1e-3) / 1e9,
           "roofline_frac": (in_b + out_b) / (per * 1e-3) / 1e9 / peak,
           "algorithmic_bytes_per_pixel": 3.0, "kernel": "arw2_kernel<dither>"}
    if not args.skip_cpu and rank0:
        import oracle
        if oracle.HAVE_REF:
            ncores = os.cpu_count() or 1
            tmp = port.new_image(w, h)
            msr = min(oracle.ref.sony_arw2(tmp, w, data, curve, True, nthreads=ncores) for _ in range(3))
            ms1 = oracle.ref.sony_arw2(tmp, w, data, curve, True, nthreads=1)
            ent["cpu_reference"] = {"kind": "reference", "cores": ncores,
                                    "MPixels/s": w * h / (msr * 1e-3) / 1e6,
                                    "single_thread_MPixels/s": w * h / (ms1 * 1e-3) / 1e6,
                                    "sample": "SonyArw2Decompressor::decompress (OpenMP over rows), 1 frame, best of 3"}
    out["8(f)4 SonyArw2Decompressor 9568x6376 (dithered curve)"] = ent
    del plan, d_in, d_out
    return out


def bench_unvalidated(torch, rs, ctx, port, synth, args, dist, peak):
    """SURVEY 8(f)3 (+ Panasonic V4): kernels written after round 1's GPU budget was spent.  Off by
    default (--unvalidated); every leg first checks the result against the oracle."""
    out = {}
    steps = max(3, min(args.steps, 10))
    W, H = 8256, 5504
    pitch = rs.image_pitch(W)
    rng = np.random.default_rng(9)
    base = port.new_image(W, H)
    base[:, :] = rng.integers(0, 16384, size=base.shape, dtype=np.uint16)

    rank0 = int(os.environ.get("RANK", "0")) == 0
    ncores = os.cpu_count() or 1

    def leg(name, plan, want, kernel, restore=True, cpu=None, cpu_threads=None):
        d = torch.from_numpy(base.view(np.int16).copy()).cuda()
        src = d.clone()
        plan.run(None, d)
        torch.cuda.synchronize()
        exact = bool(np.array_equal(d.cpu().numpy().view(np.uint16), want))

        def step():
            if restore:
                d.copy_(src)        # in-place kernels: every timed run starts from the same pixels
            plan.run(None, d)
        ms = time_steps(torch, step, steps, 3, dist)
        ms_copy = time_steps(torch, lambda: d.copy_(src), steps, 3, dist) if restore else 0.0
        in_b, out_b, pixels = plan.bytes()
        per = (ms - ms_copy) / steps
        out[name] = {"MPixels/s": pixels / (per * 1e-3) / 1e6, "ms_per_frame": per, "bit_exact": exact,
                     "achieved_GBps": (in_b + out_b) / (per * 1e-3) / 1e9,
                     "roofline_frac": (in_b + out_b) / (per * 1e-3) / 1e9 / peak, "kernel": kernel,
                     "timing": "in-place kernel + restoring copy, minus the copy alone"}
        if cpu is not None and not args.skip_cpu and rank0:
            import oracle
            if oracle.HAVE_REF:
                best = 1e30
                for _ in range(3):
                    cpu(base.copy())
                    best = min(best, oracle.ref.last_ms())
                out[name]["cpu_reference"] = {"kind": "reference", "cores": cpu_threads or ncores,
                                              "MPixels/s": W * H / (best * 1e-3) / 1e6, "ms": best,
                                              "sample": "the reference's own member on 1 frame, best of 3 (driver copies excluded)"}

    # K9: black / white scaling, both loops
    for label, black, white in (("SSE2 loop", (1008, 1010, 1009, 1011), 16383), ("plain loop", (64,) * 4, 1000)):
        j = rs.ScaleJob()
        j.offset, j.pitch, j.width, j.height, j.cpp = 0, pitch, W, H, 1
        j.crop_x, j.crop_y, j.crop_w, j.crop_h = 8, 8, W - 16, H - 16
        for i in range(4):
            j.black_separate[i] = black[i]
        j.white_point, j.dither, j.path = white, 1, 0
        want = base.copy()
        port.scale_values(want, W, (8, 8, W - 16, H - 16), black, white)
        leg("8(f)3 scaleBlackWhite 8256x5504 (%s, dither)" % label, rs.scale_plan(ctx, [j]), want,
            "scale_kernel<%d>" % (0 if "SSE2" in label else 1),
            cpu=lambda im, black=black, white=white: __import__("oracle").ref.scale_values(
                im, W, (8, 8, W - 16, H - 16), black, white, nthreads=ncores))
    # K12: whole-image table lookup, Sony curve, plain and dithered
    for dither in (False, True):
        lj = rs.LookupJob()
        lj.offset, lj.pitch, lj.width, lj.height, lj.cpp, lj.table = 0, pitch, W, H, 1, 0
        t = port.build_table(synth.sony_curve(), dither)
        want = base.copy()
        port.sixteen_bit_lookup(want, W, 1, t, dither)
        leg("8(f)3 sixteenBitLookup 8256x5504 (%s)" % ("dithered" if dither else "plain"),
            rs.lookup_plan(ctx, [lj], t, dither), want, "lookup_kernel<%s>" % ("true" if dither else "false"),
            cpu=lambda im, dither=dither: __import__("oracle").ref.sixteen_bit_lookup(
                im, W, 1, [0, 0, W, H], synth.sony_curve(), dither, nthreads=ncores))
    # K10: eight opcodes in one pass
    from rawspeed_b200 import host
    area = synth.dng_pixel_area((0, 0, H, W))
    blob = synth.dng_opcode_list([
        synth.dng_delta(12, area, rng.random(H, dtype=np.float32) + 0.5),
        synth.dng_delta(13, synth.dng_pixel_area((0, 0, H, W), 0, 1, 1, 2), rng.random(W // 2, dtype=np.float32) + 0.5),
        synth.dng_delta(10, synth.dng_pixel_area((1, 1, H, W), 0, 1, 2, 2), (rng.random(H // 2, dtype=np.float32) - 0.5) * 0.01),
        synth.dng_delta(11, area, (rng.random(W, dtype=np.float32) - 0.5) * 0.01),
        synth.dng_map_polynomial(area, [0.0, 0.8, 0.3, -0.1]),
        synth.dng_map_table(synth.dng_pixel_area((0, 1, H, W), 0, 1, 2, 2), (np.arange(65536) ^ 1).astype(np.uint16)),
        synth.dng_delta(13, synth.dng_pixel_area((8, 8, H - 8, W - 8), 0, 1, 1, 16), rng.random((W - 16 + 15) // 16, dtype=np.float32) + 0.25),
        synth.dng_delta(12, synth.dng_pixel_area((0, 0, H, W), 0, 1, 4, 1), rng.random(H // 4, dtype=np.float32) + 0.75)])
    low = host.dngop_lower(base, W, 1, [0, 0, W, H], blob)
    dj = rs.DngOpJob()
    dj.offset, dj.pitch, dj.width, dj.height, dj.cpp, dj.is_f32 = 0, pitch, W, H, 1, 0
    dj.first_op, dj.num_ops = 0, len(low["ops"])
    want = base.copy()
    port.dng_opcodes(want, W, 1, [0, 0, W, H], blob)
    leg("8(f)3 DngOpcodes 8256x5504, 8 opcodes in one pass", rs.dngop_plan(ctx, [dj], low["ops"], low["tables"], low["deltas"]),
        want, "dngop_kernel", cpu=lambda im: __import__("oracle").ref.dng_opcodes(im, W, 1, [0, 0, W, H], blob),
        cpu_threads=1)   # applyOpCodes is single threaded in the reference
    # K11: 20 000 defects
    n = 20000
    p = ((rng.integers(0, H, n).astype(np.uint32) << 16) | rng.integers(0, W, n).astype(np.uint32))
    bj = rs.BadPixJob()
    bj.offset, bj.pitch, bj.width, bj.height, bj.is_cfa = 0, pitch, W, H, 1
    bj.first_position, bj.num_positions, bj.prior_map = 0, n, None
    want = base.copy()
    port.fix_bad_pixels(want, W, 1, p, True)
    leg("8(f)3 fixBadPixels 8256x5504, 20000 defects", rs.badpix_plan(ctx, [bj], p), want, "badpix_kernel",
        restore=False,     # idempotent: good pixels are never written
        cpu=lambda im: __import__("oracle").ref.fix_bad_pixels(im, W, 1, p, True, nthreads=ncores))
    # Panasonic V4, 4592x3448-class frames, 4 per launch
    w, h, split = 4592 // 14 * 14, 3448, 0x2008
    nbytes = (w * h // 14 * 16 + 0x3FFF) // 0x4000 * 0x4000
    data = synth.lcg_bytes(nbytes, 44)
    opitch = rs.image_pitch(w)
    nf, fb, ob = 4, (nbytes + 255) // 256 * 256, (h * opitch + 255) // 256 * 256
    jobs = []
    for f in range(nf):
        pj = rs.PanaJob()
        pj.in_offset, pj.in_size, pj.out_offset, pj.out_pitch = f * fb, nbytes, f * ob, opitch
        pj.width, pj.height, pj.version, pj.bps = w, h, 4, 12
        pj.zero_is_not_bad, pj.section_split_offset = 0, split
        jobs.append(pj)
    plan = rs.pana_plan(ctx, jobs)
    d_in = torch.zeros(nf * fb + 64, dtype=torch.uint8, device="cuda")
    for f in range(nf):
        d_in[f * fb:f * fb + nbytes] = torch.from_numpy(data)
    d_out = torch.zeros(nf * ob, dtype=torch.uint8, device="cuda")
    plan.run((d_in.data_ptr(), nf * fb), d_out)
    torch.cuda.synchronize()
    want = port.new_image(w, h)
    zwant = port.panasonic_v4(want, w, data, False, split, cap=1 << 22)
    got = d_out[(nf - 1) * ob:(nf - 1) * ob + h * opitch].cpu().numpy().view(np.uint16).reshape(h, opitch // 2)
    nz, zl = plan.bad_pixels(nf - 1, cap=1 << 22)
    exact = bool(np.array_equal(got[:, :w], want[:, :w])) and sorted(zl) == zwant
    ms = time_steps(torch, lambda: plan.run((d_in.data_ptr(), nf * fb), d_out), steps, 3, dist)
    in_b, out_b, pixels = plan.bytes()
    per = ms / steps
    out["8(f)4 PanasonicV4Decompressor %dx%d" % (w, h)] = {
        "MPixels/s": pixels / (per * 1e-3) / 1e6, "ms_per_step": per, "frames_per_step": nf, "bit_exact": exact,
        "achieved_GBps": (in_b + out_b) / (per * 1e-3) / 1e9,
        "roofline_frac": (in_b + out_b) / (per * 1e-3) / 1e9 / peak, "kernel": "pana_kernel<4,12>"}
    return out


def bench_forms(torch, rs, ctx, port, synth, args, dist, peak):
    """SURVEY 8(f)1: the fixed-layout UncompressedDecompressor forms, one 8256x5504
    frame each, device-timed like the headline (inputs resident in HBM)."""
    from rawspeed_b200 import formats as F
    out = {}
    steps = max(3, min(args.steps, 10))
    cases = [("decode12BitRawWithControl<big>", F.RAW_12BIT_CONTROL_BE, 12 * W // 8 + (W + 2) // 10,
              port.FORM_12BIT_CONTROL_BE, 12, port.MSB, False),
             ("decode12BitRawUnpackedLeftAligned<little>", F.RAW_12BIT_LEFT_LE, 2 * W,
              port.FORM_12BIT_LEFT_LE, 16, port.LSB, False),
             ("decode8BitRaw<uncorrected>", F.RAW_8BIT, W, port.FORM_8BIT_UNCORRECTED, 8, port.LSB, False),
             ("decodePackedFP<MSB, binary16> -> float", F.RAW_FP16_MSB, 2 * W, port.FORM_READ, 16,
              port.MSB, True)]
    for name, fmt, pitch, form, bps, order, f32 in cases:
        data = synth.lcg_bytes(pitch * H, seed=7)
        want = port.new_image_f32(W, H) if f32 else port.new_image(W, H)
        got0 = want.copy()
        j = rs.RawJob()
        j.in_offset, j.in_size, j.out_offset = 0, data.size, 0
        j.out_pitch = want.shape[1] * want.itemsize
        j.row0, j.rows, j.samples, j.out_col0 = 0, H, W, 0
        j.in_pitch, j.format, j.table = pitch, fmt, 0
        plan = rs.raw_plan(ctx, [j])
        d_in = torch.zeros(data.size + 64, dtype=torch.uint8, device="cuda")
        d_in[:data.size] = torch.from_numpy(data.copy())
        d_out = torch.from_numpy(got0.view(np.uint8).reshape(-1).copy()).cuda()
        plan.run((d_in.data_ptr(), data.size), d_out)
        torch.cuda.synchronize()
        port.unpack_form(data, want, W, 1, (0, 0, W, H), pitch, bps, order, form)
        exact = bool(np.array_equal(d_out.cpu().numpy().view(want.dtype).reshape(want.shape), want))
        ms = time_steps(torch, lambda: plan.run((d_in.data_ptr(), data.size), d_out), steps, 3, dist)
        in_b, out_b, pixels = plan.bytes()
        per = ms / steps
        ent = {"MPixels/s": pixels / (per * 1e-3) / 1e6, "ms_per_frame": per, "bit_exact": exact,
               "achieved_GBps": (in_b + out_b) / (per * 1e-3) / 1e9,
               "roofline_frac": (in_b + out_b) / (per * 1e-3) / 1e9 / peak,
               "kernel": "rawform_kernel<%d>" % fmt,
               "note": "single 45 MP frame per launch (%.0f MB moved): a short launch, below "
                       "the batch figure" % ((in_b + out_b) / 1e6)}
        if not args.skip_cpu and int(os.environ.get("RANK", "0")) == 0:
            import oracle
            if oracle.HAVE_REF:
                tmp = want.copy()
                msr = min(oracle.ref.unpack_form(data, tmp, W, 1, (0, 0, W, H), pitch, bps, order,
                                                 form, reps=1) for _ in range(2))
                ent["cpu_reference"] = {"kind": "reference", "cores": 1,
                                        "MPixels/s": PIX / (msr * 1e-3) / 1e6,
                                        "sample": "1 frame, best of 2 (single threaded by design)"}
        out["8(f)1 " + name + " 8256x5504"] = ent
        del plan, d_in, d_out
    return out


if __name__ == "__main__":
    main()
