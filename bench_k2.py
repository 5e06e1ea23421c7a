"""K2 records of bench.py (BASELINE configs[2] and configs[3]): synthetic RNG19 dual-return packet stream
-> ScanBatcher decode -> LidarScan fields -> fused destagger + cartesian, 128x2048.

  value : device-resident packets, one fused decode launch per step over `frames` frames
          (ob_decode_batch_run): all 10 channel fields + column headers + XYZ x2 + destaggered range x2.
  e2e   : host packets through the product FrameBatcher (per-packet host state machine, pinned
          staging, H2D of the wire bytes, fused launch, D2H of every decoded field + XYZ + rd).
  streams_per_gpu = 1 is configs[2]; 8 (x 8 GPUs = 64 streams, stream i on GPU i mod G, own LUT per
  stream, all frames of a GPU in one launch) is configs[3].
"""
import os
import time

import numpy as np

import bench_common as bc

H, W, R, CPP = 128, 2048, 2, 16
POINTS_PER_FRAME = H * W * R
SHIFTS = np.tile(np.array([48, 32, 16, 0], np.int32), H // 4)
PROFILE = "RNG19_RFL8_SIG16_NIR16_DUAL"
K2_BYTES_PER_FRAME_F32 = 23_917_696   # SURVEY 8(d) algorithmic bytes (tools/)
DUMP_K2_PIXELS = 1 << 18              # --dump-outputs: ~24 MB of K2 pixels (10 fields, XYZ and destaggered range x2)
DUMP_K2_COLUMNS = 1 << 16             # and 1.3 MB of column headers


def synth_packets(ob, n_distinct, seed=0xdeadbeef, profile=PROFILE, h=H, w=W, shifts=None):
    """Random frames encoded with the product's frame_to_packets, the way the reference's tests
    synthesise packet streams (tests/packet_format_test.cpp:246-266): every profile field drawn
    within its value mask, headers iota, status 1."""
    shifts = SHIFTS if shifts is None else shifts
    si = ob.SensorInfo(profile, h, w, CPP, fw_rev="v3.2.1", pixel_shift_by_row=shifts)
    masks = {f[0]: f[6] for f in si.fields()}
    out, frames = [], []
    for k in range(n_distinct):
        rs = np.random.default_rng((seed + k) % (1 << 32))
        fr = ob.LidarFrame(si)
        for name in fr.fields:
            a = fr.field(name)
            a[...] = (rs.integers(0, 1 << 32, size=a.shape, dtype=np.uint64) & np.uint64(masks[name])).astype(a.dtype)
        # ~50 % / 80 % empty returns like the reference's benchmark inputs (benchmark_utils.h:102-107)
        fr.field("RANGE")[rs.random((h, w)) < 0.5] = 0
        if "RANGE2" in fr.fields:
            fr.field("RANGE2")[rs.random((h, w)) < 0.8] = 0
        fr.measurement_id[:] = np.arange(w)
        fr.timestamp[:] = 1000 + np.arange(w)
        fr.status[:] = 1
        fr.packet_timestamp[:] = 10 + np.arange(w // CPP)
        fr.frame_id = 700 + k
        pk, ts = ob.frame_to_packets(fr, si, init_id=0, prod_sn=0)
        assert pk.shape[0] == w // CPP
        out.append(pk)
        frames.append(fr)
    return si, np.stack(out), frames


def oracle_decode(orc, opf, packets):
    """FrameBatcher decode of one frame's packets on the CPU oracle -> oracle frame."""
    fr = orc.Frame(opf, with_window=True)
    b = orc.Batcher(opf)
    for k, p in enumerate(packets):
        b.batch(p, 10 + k, fr)
    return fr


class K2State:
    """Device-resident inputs/outputs shared by the configs[2] and configs[3] measurements."""

    def __init__(self, args, ob, torch, dist, rank, local_rank, world):
        self.ob, self.torch, self.dist, self.rank, self.local_rank, self.world = ob, torch, dist, rank, local_rank, world
        self.dev = dev = torch.device("cuda", local_rank)
        self.F = F = max(4, int(getattr(args, 'k2_frames', 32)))
        self.ND = ND = 4
        self.si, pk, self.src_frames = synth_packets(ob, ND, seed=0xdeadbeef ^ rank)
        self.n_slots, self.psz = pk.shape[1], pk.shape[2]
        self.pk = pk
        self.pool = np.stack([pk[i % ND] for i in range(F)])            # [F, 128, 33024]
        self.t_pk = torch.from_numpy(self.pool).to(dev)
        rs = np.random.default_rng(43)
        self.d = (rs.random((H * W, 3)) + 0.5).astype(np.float32)
        self.o = (rs.random((H * W, 3)) * 0.01).astype(np.float32)
        # the only collective: one LUT broadcast from rank 0, outside the timed region
        self.t_dir, self.t_off = ob.sharding.broadcast_lut(self.d, self.o, dist, src=0, device=dev)
        self.dec = ob.Decoder.from_sensor(self.si, self.src_frames[0], device=local_rank)
        tdt = {1: torch.uint8, 2: torch.int16, 4: torch.int32}
        self.fields = {f["name"]: torch.empty((F, H, W), dtype=tdt[f["elem_size"]], device=dev)
                       for f in self.dec.fields}
        self.xyz = [torch.empty((F, H * W, 3), dtype=torch.float32, device=dev) for _ in range(R)]
        self.rd = [torch.empty((F, H, W), dtype=torch.int32, device=dev) for _ in range(R)]
        self.t_ts = torch.empty((F, W), dtype=torch.int64, device=dev)
        self.t_mid = torch.empty((F, W), dtype=torch.int16, device=dev)
        self.t_st = torch.empty((F, W), dtype=torch.int32, device=dev)
        self.stream = torch.cuda.current_stream()
        self.obs = ob.Stream(local_rank, cuda_stream=self.stream.cuda_stream)
        self.field_bytes_px = sum(f["elem_size"] for f in self.dec.fields)
        self._oracle = None

    def luts_for(self, streams_per_gpu):
        """stream i lives on GPU i mod G: this rank owns streams rank, rank+G, ...; each has its own LUT
        (scaled copies of the broadcast table, so that they are distinct data)."""
        ob = self.ob
        sids = [self.rank + self.world * i for i in range(streams_per_gpu)]
        luts = [ob.XYZLutT.from_arrays(self.t_dir * (1.0 + 1e-3 * sid), self.t_off * (1.0 + 1e-3 * sid), H, W,
                                       device=self.local_rank) for sid in sids]
        return sids, luts

    def oracle_frames(self, orc):
        """The ND distinct frames decoded by the CPU oracle's FrameBatcher (cached)."""
        if self._oracle is None:
            from tests.helpers import oracle_pf
            opf = oracle_pf(PROFILE, H, W)
            self._oracle = (opf, [oracle_decode(orc, opf, self.pk[i]) for i in range(self.ND)])
        return self._oracle

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()


def measure_k2(st, args, streams_per_gpu, pcie, with_e2e=True, with_cpu=True, dump=None):
    """One K2 record (dict).  Every rank calls this; the record is complete on rank 0.  With a `dump` dict,
    rank 0 adds to it a seeded sample of the pixels and columns its last timed step decoded."""
    ob, torch, dist, dev = st.ob, st.torch, st.dist, st.dev
    F, world, rank = st.F, st.world, st.rank
    S = max(1, min(int(streams_per_gpu), F))
    sids, stream_luts = st.luts_for(S)
    frame_luts = [stream_luts[i % S] for i in range(F)]

    # the launch descriptor is marshalled once (Decoder.prepare_batch); a step is one call of the plan
    step = st.dec.prepare_batch(F, st.t_pk, st.n_slots, st.psz, st.n_slots * st.psz, st.fields, lut=None,
                                pixel_shift_by_row=SHIFTS, xyz=st.xyz, range_destaggered=st.rd, timestamp=st.t_ts,
                                measurement_id=st.t_mid, status=st.t_st, stream=st.obs, frame_luts=frame_luts)

    bc.gpu_spin(torch, dev)
    sampler = bc.ClockSampler(st.local_rank)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    st.barrier()
    l0, lp0 = ob.kernel_launch_count(), ob.kernel_launch_count("decode_pipe")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    st.barrier()
    sampler.mark()
    ev[0].record(st.stream)
    for i in range(args.steps):
        step()
        ev[i + 1].record(st.stream)
    st.barrier()
    sampler.mark()
    launches = ob.kernel_launch_count() - l0
    pipe_launches = ob.kernel_launch_count("decode_pipe") - lp0
    clocks = sampler.stop()
    if dump is not None and rank == 0:
        px = bc.dump_index(torch, dev, F * H * W, DUMP_K2_PIXELS, seed=2)
        for f in st.dec.fields:
            dump["k2_" + f["name"]] = bc.dump_array(st.fields[f["name"]].view(-1)[px],
                                                    st.src_frames[0].field(f["name"]).dtype)
        for r in range(R):
            dump[f"k2_xyz{r}"] = bc.dump_array(st.xyz[r].view(-1, 3)[px], np.float32)
            dump[f"k2_range_destaggered{r}"] = bc.dump_array(st.rd[r].view(-1)[px], np.uint32)
        col = bc.dump_index(torch, dev, F * W, DUMP_K2_COLUMNS, seed=3)
        dump["k2_timestamp"] = bc.dump_array(st.t_ts.view(-1)[col], np.uint64)
        dump["k2_measurement_id"] = bc.dump_array(st.t_mid.view(-1)[col], np.uint16)
        dump["k2_status"] = bc.dump_array(st.t_st.view(-1)[col], np.uint32)
    ms_total = ev[0].elapsed_time(ev[-1])
    per_launch_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    ms_max = bc.max_over_ranks(torch, dist, dev, ms_total)
    value = world * F * POINTS_PER_FRAME * args.steps / (ms_max * 1e-3) / 1e6
    avg = float(np.mean(per_launch_ms)) * 1e-3
    alg, comp = bc.k2_bytes(H, W, R, F, st.psz, CPP, st.field_bytes_px, n_luts=S)

    # ---- parity over ALL frames of the timed launch: fields + headers vs the CPU oracle's FrameBatcher,
    #      XYZ / destaggered range vs the oracle's cartesianT<float> / destagger on the decoded ranges ----
    from oracle import oracle as orc   # test infrastructure: the checker, never the thing measured
    opf, oframes = st.oracle_frames(orc)
    ok = True
    xyz_ref = {}
    dev_fields = {n: t.cpu().numpy() for n, t in st.fields.items()}
    dev_xyz = [t.cpu().numpy() for t in st.xyz]
    dev_rd = [t.cpu().numpy().view(np.uint32) for t in st.rd]
    dev_ts = st.t_ts.cpu().numpy().view(np.uint64)
    for i in range(F):
        of = oframes[i % st.ND]
        for f in st.dec.fields:
            ref = of.field(f["name"])
            ok &= bool(np.array_equal(dev_fields[f["name"]][i].view(ref.dtype), ref))
        ok &= bool(np.array_equal(dev_ts[i], of.timestamp))
        key = (i % st.ND, i % S)
        if key not in xyz_ref:
            lut = frame_luts[i]
            xyz_ref[key] = [(orc.cartesian(of.field(nm), lut.direction, lut.offset), orc.destagger(of.field(nm), SHIFTS))
                            for nm in ("RANGE", "RANGE2")]
        for r in range(R):
            ok &= bool(np.array_equal(dev_xyz[r][i], xyz_ref[key][r][0]))
            ok &= bool(np.array_equal(dev_rd[r][i], xyz_ref[key][r][1]))
    parity = bc.all_ok(torch, dist, dev, ok)

    rec = {
        "metric": "Mpoints/s 128x2048 dual-return packets->fields+destagger+XYZ", "value": value,
        "unit": "Mpoints/s", "ms_per_step": ms_max / args.steps,
        "dtype": "u8/u16/u32 decode + f32 xyz",
        "config": {"workload": ("synthetic RNG19 dual-return packet stream -> ScanBatcher decode -> LidarScan -> "
                                "fused cartesian (K2), 128x2048" if S == 1 else
                                f"{S * world} concurrent 2048x128 synthetic streams batched and sharded across "
                                f"{world} GPU(s), own LUT per stream"),
                   "frames_per_step_per_gpu": F, "points_per_frame": POINTS_PER_FRAME,
                   "streams_per_gpu": S, "streams_total": S * world,
                   "frames_per_stream_per_step": F // S,
                   "parallelism": f"{S * world} independent sensor streams, stream i -> GPU i mod {world}, "
                                  "one fused launch per GPU per step, no data-path collective",
                   "l2_policy": f"{comp / 1e6:.0f} MB of DRAM traffic per step > 126 MB L2"},
        "roofline": bc.roofline(alg, comp, avg, "decode_pipe_kernel<float>" if pipe_launches else "decode_kernel<float>",
                                "k2_traffic.json" if S == 1 else "k2_streams8_traffic.json", bc.K2_SOURCES),
        "gpu_launches": int(launches), "pipelined_kernel_launches": int(pipe_launches),
        "clocks": clocks,
        "parity_vs_oracle": {"ok": parity, "frames_checked": F * world,
                             "what": "every field + timestamps vs the oracle FrameBatcher, XYZ + destaggered "
                                     "range vs oracle cartesianT<float>/destagger, all frames of the timed launch"},
    }
    if not with_e2e:
        return rec

    # ---- e2e: page-locked host packets -> product FramePipeline (FrameBatcher host state machine,
    #      3 frames in flight) -> host LidarFrame fields + fused cloud, every frame H2D + D2H ----
    ob.set_device(st.local_rank)
    pipe = ob.FramePipeline(st.si, depth=3, lut=frame_luts[0], pixel_shift_by_row=SHIFTS)
    e2e_frames = 2 * F
    pin_pool = ob.pinned_empty((e2e_frames,) + st.pool.shape[1:], np.uint8)
    pin_pool[:F] = st.pool
    pin_pool[F:] = st.pool
    host_ts = 10 + np.arange(st.n_slots, dtype=np.uint64)

    def stamp_ids(base):   # distinct, increasing frame ids so that no packet is dropped as "old frame"
        for i in range(e2e_frames):
            fid = base + i
            pin_pool[i, :, 2] = fid & 0xff
            pin_pool[i, :, 3] = (fid >> 8) & 0xff

    ref0 = xyz_ref[(0, 0)]

    def e2e_step(check=False):
        n_done, good = 0, True

        def retire(slot):
            nonlocal n_done, good
            if check:   # every frame: fields == oracle decode, cloud == oracle projection with stream 0's LUT
                of = oframes[n_done % st.ND]
                for f in st.dec.fields:
                    good &= bool(np.array_equal(slot.frame.field(f["name"]), of.field(f["name"])))
                if n_done % st.ND == 0:
                    for r in range(R):
                        good &= bool(np.array_equal(slot.xyz[r].reshape(-1, 3), ref0[r][0]))
                        good &= bool(np.array_equal(slot.range_destaggered[r], ref0[r][1]))
            n_done += 1
        for i in range(e2e_frames):
            used, slot = pipe.push_burst(pin_pool[i], host_ts)   # 128 packets -> 1 frame
            if slot is not None:
                retire(slot)
        while (slot := pipe.drain()) is not None:
            retire(slot)
        return n_done, good

    stamp_ids(1000)
    _, e2e_ok = e2e_step(check=True)
    stamp_ids(3000)
    st.barrier()
    st0 = pipe.stats()
    t0 = time.perf_counter()
    done, _ = e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    st1 = pipe.stats()
    host_ms = {k[:-2] + "_ms_per_frame": (st1[k] - st0[k]) * 1e3 / e2e_frames
               for k in ("burst_s", "upload_wait_s", "submit_s", "wait_s")}
    host_ms["total_ms_per_frame"] = e2e_s * 1e3 / e2e_frames
    e2e_max = bc.max_over_ranks(torch, dist, dev, e2e_s)
    e2e_val = world * e2e_frames * POINTS_PER_FRAME / e2e_max / 1e6
    field_bytes = st.field_bytes_px * H * W
    h2d = int(e2e_frames * st.n_slots * st.psz)
    d2h = int(e2e_frames * (field_bytes + R * H * W * 16))
    rec["e2e"] = {"value": e2e_val, "unit": "Mpoints/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                  "frames": e2e_frames, "frames_completed": int(done),
                  "matches_oracle": bc.all_ok(torch, dist, dev, e2e_ok),
                  "pcie_frac": bc.pcie_fraction(pcie, h2d, d2h, e2e_max) if pcie else None,
                  "host_thread": host_ms,
                  "path": "FramePipeline.push_burst (FrameBatcher host state machine per packet, zero-copy "
                          "upload from page-locked bursts, 3 frames in flight) + one fused launch per frame"}
    del pipe

    if with_cpu and world == 1 and rank == 0 and not args.no_cpu_baseline:
        rec["cpu_baseline"] = cpu_baseline_k2(orc, opf, st.pool, frame_luts[0].direction, frame_luts[0].offset)
    return rec


def cpu_baseline_k2(orc, opf, pool, d, o, budget_s=6.0):
    """The reference's CPU path for K2 driven from C (oracle/orc_bench.c): FrameBatcher decode +
    destagger<u32> + cartesianT<float> per return, three ways; value = the best of them."""
    cores = os.cpu_count() or 1
    nf = max(8, min(cores, 128))
    sample = np.stack([pool[i % pool.shape[0]] for i in range(nf)])
    res = {}
    orc.bench_k2("thread_per_stream", opf, sample[:min(nf, cores)], SHIFTS, d, o, reps=1)   # thread team warm-up
    t1 = orc.bench_k2("as_shipped", opf, sample[:2], SHIFTS, d, o, reps=1)
    res["as_shipped_1thread_f32"] = 2 * POINTS_PER_FRAME / t1 / 1e6
    t64 = orc.bench_k2("as_shipped", opf, sample[:2], SHIFTS, d.astype(np.float64), o.astype(np.float64), reps=1)
    res["as_shipped_1thread_f64"] = 2 * POINTS_PER_FRAME / t64 / 1e6
    orc.bench_k2("ouster_omp", opf, sample[:1], SHIFTS, d, o, reps=1)
    tomp = orc.bench_k2("ouster_omp", opf, sample[:4], SHIFTS, d, o, reps=1)
    res["ouster_omp_f32"] = 4 * POINTS_PER_FRAME / tomp / 1e6
    reps = max(1, int(budget_s / max(1e-3, nf * t1 / 2 / min(cores, nf))) // 4)
    reps = min(reps, 8)
    tN = min(orc.bench_k2("thread_per_stream", opf, sample, SHIFTS, d, o, threads=t, reps=reps) / reps
             for t in sorted({cores, max(1, cores // 2)}) for _ in range(2))
    res["thread_per_stream_f32"] = nf * POINTS_PER_FRAME / tN / 1e6
    best = max(res, key=res.get)
    return {"value": res[best], "unit": "Mpoints/s", "cores": cores, "kind": "port", "mode": best, "modes": res,
            "sample": f"{nf} frames x {reps} passes: FrameBatcher decode + destagger<u32> + cartesianT<float> per "
                      f"return, driven from C (oracle/orc_bench.c); value = best of the modes"}
