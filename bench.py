#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native scan->pointcloud path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--only k1|k2|sweep]
                    [--dump-outputs DIR]

ONE JSON line (the last line of stdout).  Top level = BASELINE.json's metric on configs[1]:
Mpoints/s of 128x2048 dual-return range->XYZ (+ destaggered range) through the fused K1 kernel, with
`roofline`, `cpu_baseline`, `e2e`, `clocks`.  The same line carries

  "k2"          configs[2]: synthetic RNG19 dual-return packet stream -> ScanBatcher decode -> LidarScan
                -> fused destagger + cartesian (the path north_star's >= 70 % target is written on),
  "k2_streams8" configs[3] semantics: 8 independent sensor streams per GPU (64 at N=8), own LUT each,
  "sweep"       configs[4]: 32x512 .. 128x2048, single + dual return, K1 and K2, next to the CPU figure,
  "pcie"        pinned-memory H2D / D2H copy rates measured in this run (the e2e figures sit on them).

A "step" is one pass of the hot path over one batch of `frames_per_step` synthetic frames (K1: 128 frames
= 67 Mpoints and 1.35 GB of DRAM traffic per step; K2: 32 frames, 0.57 GB -- far beyond the 126 MB L2, so
consecutive steps cannot be served from cache).  --steps sets the number of timed steps of every record.

--dump-outputs DIR writes what the last timed K1 and K2 steps computed (rank 0) as DIR/<name>.npy: XYZ and
destaggered range of K1; the fields, XYZ, destaggered ranges and column headers of K2.  Each is a fixed,
seeded sample of the output (float32, or float64 where float32 would round), and the inputs are seeded, so
two builds run with the same arguments can be compared array for array.

  value : device-resident inputs/outputs, one fused launch per step, CUDA-event timed.
  e2e   : the same batch through the C ABI with HOST (pinned) buffers: H2D of the inputs and D2H of
          the outputs are inside the timed region.
  --impl reference : the reference's CPU algorithm for the same config, driven from C
          (oracle/orc_bench.c; the reference itself cannot be compiled here -- needs Eigen3): as shipped
          (one thread), its opt-in OpenMP mode, one thread per stream; value = the best of them.

Multi-GPU (torchrun, one rank per GPU): independent sensor streams shard across ranks with no
data-path collective (weak scaling); the LUT is broadcast once from rank 0 over NCCL before the timed
region.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# The CPU arm drives OpenMP code (oracle/orc_bench.c).  libgomp's default busy-wait between parallel
# regions is ruinous on a 128-thread host (measured on the GPU box: 4 Mpoints/s vs 3 400 with passive
# waiting for the reference's -DOUSTER_OMP mode), so the wait policy is pinned before any OpenMP
# runtime is loaded (torch brings its own copy).
os.environ.setdefault("OMP_WAIT_POLICY", "passive")

import bench_common as bc  # noqa: E402

H, W, R = 128, 2048, 2                 # OS1-128 2048x128 dual return (BASELINE configs[1])
POINTS_PER_FRAME = H * W * R
SHIFTS = np.tile(np.array([48, 32, 16, 0], np.int32), H // 4)  # OS1-128 1024-mode shifts x2 (SURVEY 8d)
K1_WORKLOAD = "OS1-128 2048x128 dual-return fused destagger+cartesian (K1), LUT tiles staged in smem via TMA"
METRIC = "Mpoints/s 128x2048 dual-return range->XYZ"
DUMP_K1_POINTS = 1 << 20               # --dump-outputs: 20 MB of K1 points (XYZ + destaggered range)

# kept for tools/ that import them
K1_BYTES_PER_FRAME_F32 = 16_777_216     # SURVEY 8(d) algorithmic: 64 B/px = 8 (range) + 24 (LUT) + 24 (xyz) + 8 (rd)
measured_peaks = bc.measured_peaks
ClockSampler = bc.ClockSampler


def synth_pool(n_frames, seed=42, h=H, w=W, returns=R):
    """Range images as the reference's benchmark generator draws them
    (tests/benchmarks/benchmark_utils.h:93-110): ~50 % zeros (RANGE2 80 %), valid returns uniform
    in [1, 2^19-1] (19-bit RNG19 field)."""
    rs = np.random.default_rng(seed)
    rng = rs.integers(1, 1 << 19, size=(n_frames, returns, h, w), dtype=np.uint32)
    rng[:, 0][rs.random((n_frames, h, w)) < 0.5] = 0
    if returns > 1:
        rng[:, 1][rs.random((n_frames, h, w)) < 0.8] = 0
    return rng


def synth_lut(seed=43, h=H, w=W):
    """Random LUT as tests/benchmarks/benchmark_utils.h:112-126 (dir U(0.5,1.5), off U(0,0.01))."""
    rs = np.random.default_rng(seed)
    d = (rs.random((h * w, 3)) + 0.5).astype(np.float32)
    o = (rs.random((h * w, 3)) * 0.01).astype(np.float32)
    return d, o


def cpu_modes_k1(orc, rng, d, o, shifts, budget_s=8.0):
    """The reference's CPU path for K1 (destagger<u32>() + cartesian() per return, per-call result
    allocation) driven from C in its three modes, float and (reference default) double LUT.
    Returns ({mode_dtype: Mpoints/s}, description)."""
    F, returns, h, w = rng.shape
    ppf = h * w * returns
    cores = os.cpu_count() or 1
    d64, o64 = d.astype(np.float64), o.astype(np.float64)
    res = {}
    orc.bench_k1("thread_per_stream", rng[:min(F, cores)], shifts, d, o, reps=1)   # OpenMP team warm-up

    thread_counts = sorted({cores, max(1, cores // 2)})   # all hardware threads / one per physical core (2-way SMT)

    def best(mode, sample, dd, oo, reps, tries=2):
        if mode == "as_shipped":
            return min(orc.bench_k1(mode, sample, shifts, dd, oo, reps=reps) / reps for _ in range(tries))
        return min(orc.bench_k1(mode, sample, shifts, dd, oo, threads=t, reps=reps) / reps
                   for t in thread_counts for _ in range(tries))

    n1, nomp = min(F, 4), min(F, 16)
    for nm, dd, oo in (("f32", d, o), ("f64", d64, o64)):
        res[f"as_shipped_1thread_{nm}"] = n1 * ppf / best("as_shipped", rng[:n1], dd, oo, 1) / 1e6
        res[f"ouster_omp_{nm}"] = nomp * ppf / best("ouster_omp", rng[:nomp], dd, oo, 1) / 1e6
        t1 = orc.bench_k1("thread_per_stream", rng, shifts, dd, oo, reps=1)
        reps = int(max(1, min(20, budget_s / 6 / max(t1, 1e-4))))
        res[f"thread_per_stream_{nm}"] = F * ppf / best("thread_per_stream", rng, dd, oo, reps) / 1e6
    what = (f"{F} frames {h}x{w}x{returns}: destagger<u32>() + cartesian() per return with the reference's per-call "
            f"result allocation, driven from C (oracle/orc_bench.c), best of {thread_counts} host threads "
            "(OMP_WAIT_POLICY=passive); modes: as shipped (1 thread), -DOUSTER_OMP (impl/cartesian.h:15-23,50-52), "
            "one thread per stream")
    return res, what


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm for configs[1] on the host cores of this box.
    Same workload string and frames/step as the b200 arm; value = best of the three modes (float LUT,
    the arm's dtype); the as-shipped double-LUT figures are reported beside it."""
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    cores = os.cpu_count() or 1
    F = args.frames
    rng = synth_pool(F)
    d, o = synth_lut()
    for _ in range(max(1, min(args.warmup, 2))):
        orc.bench_k1("thread_per_stream", rng, SHIFTS, d, o, reps=1)
    modes, what = cpu_modes_k1(orc, rng, d, o, SHIFTS, budget_s=6.0)
    f32 = {k: v for k, v in modes.items() if k.endswith("f32")}
    best = max(f32, key=f32.get)
    mode = "_".join(best.split("_")[:-1])
    mode = {"as_shipped_1thread": "as_shipped"}.get(mode, mode)
    tc = sorted({cores, max(1, cores // 2)})
    probe = {t: min(orc.bench_k1(mode, rng, SHIFTS, d, o, threads=t, reps=1) for _ in range(2)) for t in tc}
    nthreads = min(probe, key=probe.get)
    ts = [orc.bench_k1(mode, rng, SHIFTS, d, o, threads=nthreads, reps=1) for _ in range(args.steps)]
    t = float(np.sum(ts))
    val = F * POINTS_PER_FRAME * args.steps / t / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": val,
        "unit": "Mpoints/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": K1_WORKLOAD, "frames_per_step_per_gpu": F, "points_per_frame": POINTS_PER_FRAME},
        "cpu_baseline": {"value": val, "unit": "Mpoints/s", "cores": nthreads, "kind": "port", "mode": mode,
                         "host_threads_available": cores, "modes": modes, "sample": what},
        "e2e": {"value": val, "unit": "Mpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa(local_rank):
    """Multi-GPU runs: pin this rank to the CPU cores NVML reports as local to its GPU, before any
    page-locked buffer is allocated, so the e2e staging memory is NUMA-local to the PCIe root of the
    GPU.  Best effort; returns the number of cores bound to (0 = left alone)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, w in enumerate(mask) for b in range(64) if (w >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def measure_k1(args, ob, torch, dist, rank, local_rank, world, pcie, dump=None):
    """configs[1]: the top-level record.  With a `dump` dict, rank 0 adds to it a seeded sample of the
    points its last timed step computed."""
    dev = torch.device("cuda", local_rank)
    F = args.frames
    # ---- inputs: each rank owns F independent frames (one "sensor stream shard") ----
    rng_host = synth_pool(F, seed=42 + rank)
    d, o = synth_lut()
    # the only collective: one LUT broadcast from rank 0, outside the timed region
    t_dir, t_off = ob.sharding.broadcast_lut(d, o, dist, src=0, device=dev)
    lut = ob.XYZLutT.from_arrays(t_dir, t_off, H, W, device=local_rank)
    t_rng = torch.from_numpy(rng_host.view(np.int32)).to(dev)
    t_xyz = torch.empty((F, R, H * W, 3), dtype=torch.float32, device=dev)
    t_rd = torch.empty((F, R, H, W), dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream()
    obs = ob.Stream(local_rank, cuda_stream=stream.cuda_stream)

    # the call is marshalled once; a step is one launch of the plan (ob_scan_to_cloud through the C ABI)
    step = ob.plan_scan_to_cloud(lut, SHIFTS, t_rng, xyz=t_xyz, range_destaggered=t_rd, stream=obs)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    bc.gpu_spin(torch, dev)                 # clocks up after the host-only set-up
    sampler = bc.ClockSampler(local_rank)   # NVML polling thread: warm-up and timed region, marked below
    sampler.start()
    for _ in range(args.warmup):
        step()
    barrier()
    l0 = ob.kernel_launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    sampler.mark()
    ev[0].record(stream)
    for i in range(args.steps):
        step()
        ev[i + 1].record(stream)
    barrier()
    sampler.mark()
    launches = ob.kernel_launch_count() - l0
    clocks = sampler.stop()
    if dump is not None and rank == 0:
        idx = bc.dump_index(torch, dev, F * R * H * W, DUMP_K1_POINTS, seed=1)
        dump["k1_xyz"] = bc.dump_array(t_xyz.view(-1, 3)[idx], np.float32)
        dump["k1_range_destaggered"] = bc.dump_array(t_rd.view(-1)[idx], np.uint32)
    ms_total = ev[0].elapsed_time(ev[-1])
    per_launch_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    ms_total_max = bc.max_over_ranks(torch, dist, dev, ms_total)
    value = world * F * POINTS_PER_FRAME * args.steps / (ms_total_max * 1e-3) / 1e6
    avg_launch_s = float(np.mean(per_launch_ms)) * 1e-3
    alg, comp = bc.k1_bytes(H, W, R, F)

    if args.kernel_only:
        return {"value": value, "ms_per_step": ms_total_max / args.steps,
                "frac": comp / avg_launch_s / 1e9 / bc.measured_peaks()[0],
                "frac_algorithmic": alg / avg_launch_s / 1e9 / bc.measured_peaks()[0], "clocks": clocks}

    # ---- parity over ALL frames of the timed launch against the CPU oracle (every rank its own pool) ----
    from oracle import oracle as orc   # test infrastructure: the checker, never the thing measured
    ref_xyz, ref_rd = orc.pool_k1(rng_host, SHIFTS, d, o)
    dev_xyz = t_xyz.cpu().numpy()
    dev_rd = t_rd.cpu().numpy().view(np.uint32)
    ok = bool(np.array_equal(dev_xyz, ref_xyz)) and bool(np.array_equal(dev_rd, ref_rd))
    parity = bc.all_ok(torch, dist, dev, ok)
    del dev_xyz, dev_rd

    # ---- e2e: host (pinned) buffers through the C ABI, copies inside the timed region ----
    CH = 8                                   # frames per call
    n_chunks = F // CH
    NS = 3                                   # streams in flight: H2D / kernel / D2H overlap
    h_rng = ob.pinned_empty((F, R, H, W), np.uint32)
    h_rng[...] = rng_host
    h_xyz = ob.pinned_empty((F, R, H * W, 3), np.float32)
    h_rd = ob.pinned_empty((F, R, H, W), np.uint32)
    tstreams = [torch.cuda.Stream(device=dev) for _ in range(NS)]
    ostreams = [ob.Stream(local_rank, cuda_stream=s.cuda_stream) for s in tstreams]

    def e2e_step():
        for c in range(n_chunks):
            sl = slice(c * CH, (c + 1) * CH)
            ob.scan_to_cloud(lut, SHIFTS, h_rng[sl], xyz=h_xyz[sl], range_destaggered=h_rd[sl],
                             stream=ostreams[c % NS])

    e2e_steps = args.steps
    for _ in range(2):
        e2e_step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for s in tstreams:
        s.wait_stream(stream)
    for _ in range(e2e_steps):
        e2e_step()
    for s in tstreams:
        stream.wait_stream(s)
    e1.record(stream)
    barrier()
    e2e_ms = bc.max_over_ranks(torch, dist, dev, e0.elapsed_time(e1))
    e2e_val = world * F * POINTS_PER_FRAME * e2e_steps / (e2e_ms * 1e-3) / 1e6
    e2e_ok = bc.all_ok(torch, dist, dev, bool(np.array_equal(h_xyz, ref_xyz)) and bool(np.array_equal(h_rd, ref_rd)))
    h2d_b, d2h_b = int(F * R * H * W * 4), int(F * R * H * W * (12 + 4))
    del ref_xyz, ref_rd

    # ---- the reference's default XYZLut is double: same launch with a float64 LUT, for the record ----
    f64 = None
    if rank == 0:
        try:
            lut64 = ob.XYZLutT.from_arrays(t_dir.double(), t_off.double(), H, W, device=local_rank)
            t_xyz64 = torch.empty((F, R, H * W, 3), dtype=torch.float64, device=dev)
            for _ in range(3):
                ob.scan_to_cloud(lut64, SHIFTS, t_rng, xyz=t_xyz64, range_destaggered=t_rd, stream=obs)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a0.record(stream)
            for _ in range(5):
                ob.scan_to_cloud(lut64, SHIFTS, t_rng, xyz=t_xyz64, range_destaggered=t_rd, stream=obs)
            a1.record(stream)
            torch.cuda.synchronize()
            s64 = a0.elapsed_time(a1) / 5 * 1e-3
            a64, c64 = bc.k1_bytes(H, W, R, F, esz=8)
            peak = bc.measured_peaks()[0]
            f64 = {"value_mpoints_s": F * POINTS_PER_FRAME / s64 / 1e6, "frac": c64 / s64 / 1e9 / peak,
                   "frac_algorithmic": a64 / s64 / 1e9 / peak}
            del t_xyz64, lut64
        except Exception as ex:  # supplementary figure only
            f64 = {"error": str(ex)}

    # ---- CPU baseline in the same run: the reference's loops driven from C, bounded sample ----
    cpu = None
    if not args.no_cpu_baseline and world == 1 and rank == 0:
        modes, what = cpu_modes_k1(orc, rng_host, d, o, SHIFTS)
        f32 = {k: v for k, v in modes.items() if k.endswith("f32")}
        best = max(f32, key=f32.get)
        cpu = {"value": f32[best], "unit": "Mpoints/s", "cores": os.cpu_count() or 1, "kind": "port",
               "mode": best, "modes": modes, "sample": what,
               "as_shipped_double_1thread": modes["as_shipped_1thread_f64"]}

    return {
        "metric": METRIC, "value": value, "unit": "Mpoints/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total_max / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": K1_WORKLOAD,
                   "frames_per_step_per_gpu": F, "points_per_frame": POINTS_PER_FRAME,
                   "l2_policy": f"compulsory DRAM traffic per step {comp / 1e6:.0f} MB > 126 MB L2",
                   "parallelism": f"{world} independent stream shards, LUT broadcast only",
                   "numa_bound_cores_per_rank": args.numa_cores},
        "roofline": bc.roofline(alg, comp, avg_launch_s, "cloud_tma_kernel<float,2>", "k1_traffic.json", bc.K1_SOURCES),
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_val, "unit": "Mpoints/s", "h2d_bytes_per_step": h2d_b, "d2h_bytes_per_step": d2h_b,
                "frames_per_call": CH, "streams": NS, "matches_oracle_all_frames": e2e_ok,
                "pcie_frac": bc.pcie_fraction(pcie, h2d_b, d2h_b, e2e_ms * 1e-3 / e2e_steps) if pcie else None},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "parity_vs_oracle": {"ok": parity, "frames_checked": F * world,
                             "what": "XYZ + destaggered range of every frame and return of the timed launch vs "
                                     "oracle cartesianT<float> / destagger<u32>, bit-exact"},
        "f64_lut": f64,
    }


def measure_lut_free(args, ob, torch, dist, rank, local_rank, world):
    """SURVEY 8d's LUT-free variant, reported beside the LUT path: the same K1 / K2 launches with a LUT
    built from the OS1-128 intrinsics and switched to the analytic projection (ob_lut_set_analytic).
    Opt-in mode: XYZ agrees with the oracle's float LUT path to 1e-5 norm-wise (checked here on every
    frame), it is not bit-exact."""
    import bench_k2
    dev = torch.device("cuda", local_rank)
    meta = json.load(open(os.path.join(ROOT, "tests", "golden", "OS-1-128_767798045_1024x10_20230712_120049.json")))
    args_i = (W, H, 0.001, meta["beam_to_lidar_transform"], meta["lidar_to_sensor_transform"],
              meta["beam_azimuth_angles"], meta["beam_altitude_angles"])
    lut = ob.XYZLutT.from_intrinsics(*args_i, dtype=np.float32, device=local_rank)
    d, o = lut.direction.copy(), lut.offset.copy()          # the float LUT the analytic mode replaces
    lut.set_analytic(True)
    stream = torch.cuda.current_stream()
    obs = ob.Stream(local_rank, cuda_stream=stream.cuda_stream)
    peak, _ = bc.measured_peaks()
    out = {}

    def timed(step, warmup=3):
        bc.gpu_spin(torch, dev)
        for _ in range(warmup):
            step()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            step()
        e1.record(stream)
        torch.cuda.synchronize()
        return bc.max_over_ranks(torch, dist, dev, e0.elapsed_time(e1) / args.steps * 1e-3)

    def normwise_ok(got, ref):
        err = np.linalg.norm(got.astype(np.float64) - ref.astype(np.float64), axis=-1)
        return bool(np.all(err <= 1e-5 * np.linalg.norm(ref.astype(np.float64), axis=-1) + 1e-7))

    from oracle import oracle as orc   # checker only
    # ---- K1 ----
    for returns in (2, 1):
        F = 64
        rng_host = synth_pool(F, seed=142 + rank, returns=returns)
        t_rng = torch.from_numpy(rng_host.view(np.int32)).to(dev)
        t_xyz = torch.empty((F, returns, H * W, 3), dtype=torch.float32, device=dev)
        t_rd = torch.empty((F, returns, H, W), dtype=torch.int32, device=dev)
        s = timed(ob.plan_scan_to_cloud(lut, SHIFTS, t_rng, xyz=t_xyz, range_destaggered=t_rd, stream=obs))
        ref_xyz, ref_rd = orc.pool_k1(rng_host, SHIFTS, d, o)
        got = t_xyz.cpu().numpy()
        ok = normwise_ok(got, ref_xyz) and bool(np.array_equal(t_rd.cpu().numpy().view(np.uint32), ref_rd))
        ok = ok and bool(np.all(got[rng_host.reshape(F, returns, -1) == 0] == 0.0))
        n = H * W
        dram = F * n * returns * (4 + 12 + 4)          # range in + XYZ + destaggered range out; no LUT stream
        out[f"k1_{'dual' if returns == 2 else 'single'}"] = {
            "value": world * F * n * returns / s / 1e6, "unit": "Mpoints/s", "ms_per_step": s * 1e3,
            "frac": dram / s / 1e9 / peak, "within_1e-5_of_oracle_lut_path": bc.all_ok(torch, dist, dev, ok)}
        del t_rng, t_xyz, t_rd
    # ---- K2 ----
    st = bench_k2.K2State(args, ob, torch, dist, rank, local_rank, world)
    F = st.F
    plan = st.dec.prepare_batch(F, st.t_pk, st.n_slots, st.psz, st.n_slots * st.psz, st.fields, lut=lut,
                                pixel_shift_by_row=SHIFTS, xyz=st.xyz, range_destaggered=st.rd, timestamp=st.t_ts,
                                measurement_id=st.t_mid, status=st.t_st, stream=st.obs)
    lp0 = ob.kernel_launch_count("decode_pipe")
    s = timed(plan)
    piped = ob.kernel_launch_count("decode_pipe") > lp0
    opf, oframes = st.oracle_frames(orc)
    ok = True
    dev_xyz = [t.cpu().numpy() for t in st.xyz]
    for i in range(F):
        of = oframes[i % st.ND]
        ok &= bool(np.array_equal(st.fields["RANGE"][i].cpu().numpy().view(np.uint32), of.field("RANGE")))
        for r, nm in enumerate(("RANGE", "RANGE2")):
            if i < st.ND:
                ok &= normwise_ok(dev_xyz[r][i], orc.cartesian(of.field(nm), d, o))
            else:
                ok &= bool(np.array_equal(dev_xyz[r][i], dev_xyz[r][i % st.ND]))
    _, comp = bc.k2_bytes(H, W, R, F, st.psz, bench_k2.CPP, st.field_bytes_px, n_luts=0)
    out["k2_dual"] = {"value": world * F * POINTS_PER_FRAME / s / 1e6, "unit": "Mpoints/s", "ms_per_step": s * 1e3,
                      "frac": comp / s / 1e9 / peak, "pipelined_kernel": bool(piped),
                      "within_1e-5_of_oracle_lut_path": bc.all_ok(torch, dist, dev, ok)}
    out["note"] = ("opt-in LUT-free projection (ob_lut_set_analytic): direction/offset rebuilt in-kernel from per-row / "
                   "per-column tables of a LUT made from intrinsics; frac = compulsory DRAM bytes without any LUT stream")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--only", default="all", choices=["all", "k1", "k2", "sweep"],
                    help="restrict the run to one part (tuning / profiling aid); default: everything")
    ap.add_argument("--workload", default=None, choices=["k1", "k2"], help="alias of --only (kept for tools)")
    ap.add_argument("--frames", type=int, default=128, help="K1 frames per step (per GPU)")
    ap.add_argument("--k2-frames", type=int, default=32, help="K2 frames per step (per GPU)")
    ap.add_argument("--streams-per-gpu", type=int, default=1,
                    help="with --only k2: independent sensor streams (own LUT each) per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--kernel-only", action="store_true", help="tuning aid: device-resident timing only")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed seeded sample of what the last K1 and K2 steps "
                         "computed to DIR/<name>.npy (float32 / float64, under 64 MB; rank 0 only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.workload:
        args.only = args.workload

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    args.numa_cores = bind_to_gpu_numa(local_rank) if world > 1 else 0
    import torch
    import __graft_entry__ as graft
    graft.build()
    ob = graft.load_package()
    if ob.device_count() <= 0:
        raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the caller set it (its lines go to stdout); the JSON is the LAST line
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    line = None
    dump = {} if args.dump_outputs else None
    if args.kernel_only:
        import bench_k2
        out = {}
        if args.only in ("all", "k1"):
            out["k1"] = measure_k1(args, ob, torch, dist, rank, local_rank, world, None, dump)
        if args.only in ("all", "k2"):
            st = bench_k2.K2State(args, ob, torch, dist, rank, local_rank, world)
            rec = bench_k2.measure_k2(st, args, args.streams_per_gpu, None, with_e2e=False, with_cpu=False,
                                      dump=dump)
            out["k2"] = {"value": rec["value"], "ms_per_step": rec["ms_per_step"], "frac": rec["roofline"]["frac"],
                         "frac_algorithmic": rec["roofline"]["frac_algorithmic"], "parity": rec["parity_vs_oracle"]["ok"],
                         "pipe_launches": rec["pipelined_kernel_launches"], "clocks": rec["clocks"]}
        out["env"] = {k: v for k, v in os.environ.items() if k.startswith("OB_")}
        line = out
    else:
        pcie_all = None
        pcie = bc.measure_pcie(torch, ob, dev, dist)
        g = bc.gather_floats(torch, dist, dev, [pcie[k] for k in ("h2d_gbs", "d2h_gbs", "bidir_h2d_gbs", "bidir_d2h_gbs")])
        pcie_all = {"per_rank_concurrent": [dict(zip(("h2d_gbs", "d2h_gbs", "bidir_h2d_gbs", "bidir_d2h_gbs"), r)) for r in g],
                    "rank0": pcie,
                    "note": "pinned 256 MB copies; with N ranks all ranks copy at the same time, so the figures "
                            "include the contention for each socket's host memory / PCIe root"}
        if args.only in ("all", "k1"):
            line = measure_k1(args, ob, torch, dist, rank, local_rank, world, pcie, dump)
        else:
            line = {"metric": METRIC, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "partial": args.only}
        line["pcie"] = pcie_all
        if args.only in ("all", "k2"):
            import bench_k2
            st = bench_k2.K2State(args, ob, torch, dist, rank, local_rank, world)
            line["k2"] = bench_k2.measure_k2(st, args, 1, pcie, dump=dump)
            line["k2_streams8"] = bench_k2.measure_k2(st, args, 8, pcie, with_e2e=False, with_cpu=False)
            del st
        if args.only == "all":
            line["lut_free"] = measure_lut_free(args, ob, torch, dist, rank, local_rank, world)
        if args.only in ("all", "sweep") and not args.no_sweep:
            import bench_sweep
            line["sweep"] = bench_sweep.run_sweep(args, ob, torch, dist, rank, local_rank, world)

    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
        # NCCL_DEBUG output (left as the caller set it) also arrives from library finalisers at process
        # exit.  The JSON must be the LAST stdout line: the other ranks leave first and without running
        # finalisers, rank 0 prints after they are gone and leaves the same way.
        sys.stdout.flush()
        sys.stderr.flush()
        if rank != 0:
            os._exit(0)
        time.sleep(1.0)
    if rank == 0:
        if dump is not None:
            bc.write_dumps(args.dump_outputs, dump)
        sys.stdout.flush()
        print(json.dumps(line), flush=True)
        if dist is not None:
            os._exit(0)


if __name__ == "__main__":
    main()
