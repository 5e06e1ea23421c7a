"""configs[4] of BASELINE.json: frame-size sweep 32x512 .. 128x2048, single + dual return, K1 (range ->
destagger + XYZ) and K2 (packets -> fields + destagger + XYZ): Mpoints/s and the HBM roofline fraction,
next to the CPU baseline (the reference's loops driven from C, one thread per stream) at N = 1.

Every entry: device-resident inputs, one fused launch per step, CUDA events, max over ranks; the DRAM
traffic of a step (compulsory bytes) exceeds the 126 MB L2 for every shape (the frame count is scaled:
~1.2 GB per K1 step like the headline launch, ~0.4 GB per K2 step)."""
import os

import numpy as np

import bench_common as bc

SHAPES = [(32, 512), (32, 1024), (64, 1024), (64, 2048), (128, 1024), (128, 2048)]
PROFILES = {1: "RNG19_RFL8_SIG16_NIR16", 2: "RNG19_RFL8_SIG16_NIR16_DUAL"}
TARGET_BYTES = 400e6      # K2: DRAM traffic per step
TARGET_BYTES_K1 = 1.2e9   # K1: as many bytes per step as the headline's 128-frame launch moves


def _time(torch, stream, step, steps, warmup):
    bc.gpu_spin(torch, torch.device("cuda", torch.cuda.current_device()))   # clocks up after the host-only gap
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps * 1e-3


def run_sweep(args, ob, torch, dist, rank, local_rank, world):
    import bench
    import bench_k2
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.current_stream()
    obs = ob.Stream(local_rank, cuda_stream=stream.cuda_stream)
    peak, _ = bc.measured_peaks()
    cores = os.cpu_count() or 1
    with_cpu = world == 1 and rank == 0 and not args.no_cpu_baseline
    orc = None
    if with_cpu:
        from oracle import oracle as orc   # CPU baseline leg only
    steps, warmup = args.steps, 5
    tdt = {1: torch.uint8, 2: torch.int16, 4: torch.int32}
    out = []
    for (h, w) in SHAPES:
        shifts = np.tile(np.array([3 * (w // 128), 2 * (w // 128), w // 128, 0], np.int32), h // 4)
        d, o = bench.synth_lut(seed=43, h=h, w=w)
        t_dir, t_off = torch.from_numpy(d).to(dev), torch.from_numpy(o).to(dev)
        lut = ob.XYZLutT.from_arrays(t_dir, t_off, h, w, device=local_rank)
        for returns in (1, 2):
            ppf = h * w * returns
            # ---------------- K1 ----------------
            _, c1 = bc.k1_bytes(h, w, returns, 1)
            F = int(max(8, min(2048, TARGET_BYTES_K1 // c1)))
            pool = bench.synth_pool(min(F, 16), seed=7 + rank, h=h, w=w, returns=returns)
            t_rng = torch.from_numpy(np.concatenate([pool] * ((F + len(pool) - 1) // len(pool)))[:F].view(np.int32)).to(dev)
            t_xyz = torch.empty((F, returns, h * w, 3), dtype=torch.float32, device=dev)
            t_rd = torch.empty((F, returns, h, w), dtype=torch.int32, device=dev)
            if dist is not None:
                dist.barrier()
            s = _time(torch, stream, lambda: ob.scan_to_cloud(lut, shifts, t_rng, xyz=t_xyz, range_destaggered=t_rd,
                                                               stream=obs), steps, warmup)
            s = bc.max_over_ranks(torch, dist, dev, s)
            alg, comp = bc.k1_bytes(h, w, returns, F)
            e = {"shape": f"{h}x{w}", "returns": returns, "kernel": "k1", "frames_per_step_per_gpu": F,
                 "value": world * F * ppf / s / 1e6, "unit": "Mpoints/s", "ms_per_step": s * 1e3,
                 "hbm_gbs": comp / s / 1e9, "frac": comp / s / 1e9 / peak, "frac_algorithmic": alg / s / 1e9 / peak}
            if with_cpu:
                nf = min(len(pool), max(4, cores // 8))
                sample = np.concatenate([pool] * ((cores + len(pool) - 1) // len(pool)))[:max(cores, nf)]
                orc.bench_k1("thread_per_stream", sample, shifts, d, o, reps=1)
                reps = 2
                t = min(orc.bench_k1("thread_per_stream", sample, shifts, d, o, threads=tn, reps=reps) / reps
                        for tn in (cores, max(1, cores // 2)))
                e["cpu_mpoints_s"] = sample.shape[0] * ppf / t / 1e6
            out.append(e)
            del t_rng, t_xyz, t_rd
            # ---------------- K2 ----------------
            si, pk, src = bench_k2.synth_packets(ob, 2, seed=(0xdeadbeef + h * 7 + w) & 0x7fffffff, profile=PROFILES[returns],
                                                 h=h, w=w, shifts=shifts)
            n_slots, psz = pk.shape[1], pk.shape[2]
            dec = ob.Decoder.from_sensor(si, src[0], device=local_rank)
            fbytes = sum(f["elem_size"] for f in dec.fields)
            _, c2 = bc.k2_bytes(h, w, returns, 1, psz, bench_k2.CPP, fbytes)
            F2 = int(max(8, min(1024, TARGET_BYTES // c2)))
            t_pk = torch.from_numpy(np.stack([pk[i % 2] for i in range(F2)])).to(dev)
            fields = {f["name"]: torch.empty((F2, h, w), dtype=tdt[f["elem_size"]], device=dev) for f in dec.fields}
            xyz = [torch.empty((F2, h * w, 3), dtype=torch.float32, device=dev) for _ in range(returns)]
            rd = [torch.empty((F2, h, w), dtype=torch.int32, device=dev) for _ in range(returns)]
            t_ts = torch.empty((F2, w), dtype=torch.int64, device=dev)
            t_mid = torch.empty((F2, w), dtype=torch.int16, device=dev)
            t_st = torch.empty((F2, w), dtype=torch.int32, device=dev)
            if dist is not None:
                dist.barrier()
            lp0 = ob.kernel_launch_count("decode_pipe")
            plan = dec.prepare_batch(F2, t_pk, n_slots, psz, n_slots * psz, fields, lut=lut,
                                     pixel_shift_by_row=shifts, xyz=xyz, range_destaggered=rd, timestamp=t_ts,
                                     measurement_id=t_mid, status=t_st, stream=obs)
            s = _time(torch, stream, plan, steps, warmup)
            piped = ob.kernel_launch_count("decode_pipe") > lp0
            s = bc.max_over_ranks(torch, dist, dev, s)
            # round trip of frame 0 and the last frame (encode -> decode == source)
            ok = True
            for i in (0, F2 - 1):
                for f in dec.fields:
                    ok &= bool(np.array_equal(fields[f["name"]][i].cpu().numpy().view(src[i % 2].field(f["name"]).dtype),
                                              src[i % 2].field(f["name"])))
            alg, comp = bc.k2_bytes(h, w, returns, F2, psz, bench_k2.CPP, fbytes)
            e = {"shape": f"{h}x{w}", "returns": returns, "kernel": "k2", "frames_per_step_per_gpu": F2,
                 "value": world * F2 * ppf / s / 1e6, "unit": "Mpoints/s", "ms_per_step": s * 1e3,
                 "hbm_gbs": comp / s / 1e9, "frac": comp / s / 1e9 / peak, "frac_algorithmic": alg / s / 1e9 / peak,
                 "pipelined_kernel": bool(piped), "roundtrip_ok": bc.all_ok(torch, dist, dev, ok)}
            if with_cpu:
                from tests.helpers import oracle_pf
                opf = oracle_pf(PROFILES[returns], h, w)
                nfr = max(8, min(cores, 128))
                sample = np.stack([pk[i % 2] for i in range(nfr)])
                orc.bench_k2("thread_per_stream", opf, sample, shifts, d, o, reps=1)
                t = min(orc.bench_k2("thread_per_stream", opf, sample, shifts, d, o, threads=tn, reps=1)
                        for tn in (cores, max(1, cores // 2)))
                e["cpu_mpoints_s"] = nfr * ppf / t / 1e6
            out.append(e)
            del t_pk, fields, xyz, rd, dec
        del lut
    return {"entries": out,
            "note": "frac = compulsory DRAM bytes / event time / measured copy peak (LUT once per launch); "
                    "frac_algorithmic = SURVEY 8d bytes (LUT once per frame); cpu_mpoints_s = reference loops from C, "
                    "one thread per stream on all host cores (N = 1 only)",
            "steps": steps, "warmup": warmup}
