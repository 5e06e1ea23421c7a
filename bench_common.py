"""Shared pieces of bench.py / bench_k2.py / bench_sweep.py: measured peaks, clock sampling, PCIe
peaks, byte accounting (SURVEY 8d algorithmic bytes and compulsory DRAM bytes), ncu traffic records."""
import hashlib
import json
import os
import subprocess
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


_SPIN = {}


def gpu_spin(torch, dev, ms=40.0):
    """Part of the warm-up: keep the GPU busy for `ms` milliseconds right before a measurement.  The bench
    alternates GPU measurements with seconds of host-only work (oracle parity checks, the CPU baseline legs);
    after such a gap the first launches run while the clocks are still ramping, and three 60-microsecond warm-up
    launches do not cover the ramp (the same K2 launch measured 0.058 ms back to back and 0.080 ms after a CPU
    leg).  The spin kernel is a plain torch elementwise op on a private buffer; nothing of it is timed."""
    key = str(dev)
    if key not in _SPIN:
        _SPIN[key] = torch.zeros(16 << 20, dtype=torch.float32, device=dev)
    x = _SPIN[key]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(2000):
        for _ in range(20):
            x.add_(1.0)
        e1.record()
        e1.synchronize()
        if e0.elapsed_time(e1) >= ms:
            break


class ClockSampler:
    """SM clock and clock-event (throttle) reasons sampled DURING the timed region: an NVML polling thread
    (a timed region is a few milliseconds -- `nvidia-smi -lms` often delivers its first line after it),
    with `nvidia-smi` as the fallback when NVML cannot be loaded.  `mark()` stamps the start / end of the
    timed region; samples outside it (taken under the same load during the warm-up steps in front of it)
    are only used when none fell inside, and the result says so."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.samples, self.marks, self._stop, self.t, self.nv = [], [], False, None, None

    def _visible_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if self.index < len(ids) and ids[self.index].isdigit():
                return int(ids[self.index])
        return self.index

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._visible_index())
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nv = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self._visible_index())], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def mark(self):
        self.marks.append(time.perf_counter())

    def _poll(self):
        nv = self.nv
        rs, i = 0, 0
        while not self._stop:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                if i % 4 == 0:  # the reasons bitmask is the slower query: every 4th sample (sticky bits are OR-ed)
                    try:
                        rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                    except Exception:
                        rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((time.perf_counter(), sm, rs))
                i += 1
            except Exception:
                pass
            time.sleep(0.0002)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nv is not None:
            self._stop = True
            self.t.join(timeout=1)
            inside = self.samples
            window = "timed_region"
            if len(self.marks) >= 2:
                inside = [x for x in self.samples if self.marks[0] <= x[0] <= self.marks[-1]]
                if not inside:
                    inside, window = self.samples, "warmup_and_timed_region"
            bits = 0
            for x in inside:
                bits |= x[2]
            sm = [x[1] for x in inside]
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_sm,
                    "reasons": [n for n, b in self.REASONS if bits & b], "samples": len(sm), "window": window,
                    "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names)
                   if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": "nvidia-smi"}


# ---------------------------------------------------------------------------------------------
# byte accounting
# ---------------------------------------------------------------------------------------------
def k1_bytes(h, w, returns, frames, n_luts=1, esz=4):
    """(algorithmic, compulsory) bytes of one K1 launch over `frames` frames.
    algorithmic (SURVEY 8d): per pixel read 4R + 6T, write 3T*R + 4R -- the LUT counted once per FRAME.
    compulsory DRAM: range in + XYZ out + destaggered range out per frame, each distinct LUT once per
    LAUNCH (it is L2-resident across the frames of a launch)."""
    n = h * w
    per_frame = n * (4 * returns + 3 * esz * returns + 4 * returns)
    lut = n * 6 * esz
    return frames * (per_frame + lut), frames * per_frame + n_luts * lut


def k2_bytes(h, w, returns, frames, packet_size, cols_per_packet, field_bytes_per_px, n_luts=1, esz=4):
    """(algorithmic, compulsory) bytes of one K2 launch: wire bytes + staggered fields + XYZ +
    destaggered range + column/packet headers (14 B per column + 9 B per packet, SURVEY 8d)."""
    n = h * w
    n_pk = w // cols_per_packet
    per_frame = (n_pk * packet_size + field_bytes_per_px * n + 3 * esz * returns * n + 4 * returns * n
                 + 14 * w + 9 * n_pk)
    lut = n * 6 * esz
    return frames * (per_frame + lut), frames * per_frame + n_luts * lut


def roofline(alg_bytes, comp_bytes, launch_s, kernel, traffic_file, sources):
    """The `roofline` object of a bench line.  `frac` is the physical figure: compulsory DRAM bytes per
    launch / CUDA-event launch time / measured copy peak; the SURVEY 8d figure is `frac_algorithmic`."""
    peak, kind = measured_peaks()
    tr = read_traffic(traffic_file, sources)
    return {"bound": "hbm", "achieved": comp_bytes / launch_s / 1e9, "peak": peak, "unit": "GB/s",
            "frac": comp_bytes / launch_s / 1e9 / peak, "peak_kind": kind,
            "frac_algorithmic": alg_bytes / launch_s / 1e9 / peak,
            "achieved_algorithmic": alg_bytes / launch_s / 1e9,
            "traffic": tr.get("dram_bytes_per_launch"), "traffic_record": tr.get("record"),
            "kernel": kernel, "compulsory_bytes_per_launch": int(comp_bytes),
            "algorithmic_bytes_per_launch": int(alg_bytes), "avg_launch_ms": launch_s * 1e3,
            "note": "frac = compulsory DRAM bytes (inputs + outputs once, each distinct LUT once per launch) / "
                    "event time / measured copy peak; frac_algorithmic counts the LUT once per frame "
                    "(SURVEY 8d) although it is L2-resident across a launch"}


def source_sha(sources):
    h = hashlib.sha256()
    for s in sources:
        with open(os.path.join(ROOT, s), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def read_traffic(name, sources):
    """ncu-measured DRAM bytes per launch (tools/capture_traffic.py).  Only reported when the kernel
    sources are byte-identical to those of the capture; otherwise traffic is null and says why."""
    p = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(p):
        return {"record": "none"}
    rec = json.load(open(p))
    if rec.get("source_sha") != source_sha(sources):
        return {"record": f"stale: {name} was captured for other kernel sources ({rec.get('source_sha')})"}
    return {"dram_bytes_per_launch": rec.get("dram_bytes_per_launch"),
            "record": f"{name}: ncu dram__bytes_read.sum + dram__bytes_write.sum of `{rec.get('cmd')}`"}


K1_SOURCES = ["ouster-sdk_b200/csrc/ob_cloud.cu", "ouster-sdk_b200/csrc/ob_ptx.cuh"]
K2_SOURCES = ["ouster-sdk_b200/csrc/ob_decode_pipe.cu", "ouster-sdk_b200/csrc/ob_decode_tile.cuh",
              "ouster-sdk_b200/csrc/ob_decode.cu", "ouster-sdk_b200/csrc/ob_ptx.cuh"]


# ---------------------------------------------------------------------------------------------
# PCIe peaks (pinned host <-> device memcpy), measured in the run so that e2e carries a PCIe fraction
# ---------------------------------------------------------------------------------------------
def measure_pcie(torch, ob, dev, dist=None, mb=256):
    """Pinned-memory copy rates of this rank's GPU: H2D alone, D2H alone and both at once (GB/s per
    direction).  With several ranks all of them measure at the same time (barrier first), so the
    figures include the contention for the host memory system / the socket's PCIe root."""
    n = mb << 20
    h_a = torch.from_numpy(ob.pinned_empty((n,), np.uint8))
    h_b = torch.from_numpy(ob.pinned_empty((n,), np.uint8))
    d_a = torch.empty(n, dtype=torch.uint8, device=dev)
    d_b = torch.empty(n, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def timed(up, down, reps=3):
        best = None
        for _ in range(reps + 1):
            if dist is not None:
                dist.barrier()
            torch.cuda.synchronize()
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            if up:
                with torch.cuda.stream(s1):
                    e[0].record()
                    d_a.copy_(h_a, non_blocking=True)
                    e[1].record()
            if down:
                with torch.cuda.stream(s2):
                    e[2].record()
                    h_b.copy_(d_b, non_blocking=True)
                    e[3].record()
            torch.cuda.synchronize()
            r = (n / (e[0].elapsed_time(e[1]) * 1e-3) / 1e9 if up else None,
                 n / (e[2].elapsed_time(e[3]) * 1e-3) / 1e9 if down else None)
            if best is None or sum(x or 0 for x in r) > sum(x or 0 for x in best):
                best = r
        return best

    h2d = timed(True, False)[0]
    d2h = timed(False, True)[1]
    bi = timed(True, True)
    out = {"h2d_gbs": h2d, "d2h_gbs": d2h, "bidir_h2d_gbs": bi[0], "bidir_d2h_gbs": bi[1],
           "buffer_mb": mb}
    del d_a, d_b
    return out


def pcie_fraction(pcie, h2d_bytes, d2h_bytes, seconds):
    """Fraction of the measured PCIe capability an e2e step used: the time the slower direction needs
    at its measured rate with both directions busy, over the measured step time."""
    t_up = h2d_bytes / (pcie["bidir_h2d_gbs"] * 1e9) if h2d_bytes else 0.0
    t_down = d2h_bytes / (pcie["bidir_d2h_gbs"] * 1e9) if d2h_bytes else 0.0
    return max(t_up, t_down) / seconds if seconds > 0 else None


def gather_floats(torch, dist, dev, vals):
    """vals (list of floats) from every rank -> [world][len(vals)] (rank 0 order)."""
    if dist is None:
        return [list(vals)]
    t = torch.tensor(vals, dtype=torch.float64, device=dev)
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return [o.cpu().tolist() for o in out]


def max_over_ranks(torch, dist, dev, v):
    if dist is None:
        return float(v)
    t = torch.tensor([v], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def all_ok(torch, dist, dev, ok):
    if dist is None:
        return bool(ok)
    t = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item())


# ---------------------------------------------------------------------------------------------
# --dump-outputs: what the timed launches computed, as .npy files, so that two builds can be compared
# ---------------------------------------------------------------------------------------------
DUMP_MAX_BYTES = 64_000_000


def dump_index(torch, dev, n, k, seed):
    """Sorted flat indices (a device tensor) of a fixed, seeded sample of k of n elements; all n when k >= n."""
    idx = np.arange(n) if k >= n else np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))
    return torch.from_numpy(idx).to(dev)


def dump_array(t, dtype):
    """Host copy of a device output holding `dtype` values (the tensors carry unsigned fields in signed
    types of the same width), as float32 for floats and integers of up to 16 bits, float64 otherwise:
    exact for every integer below 2**53."""
    a = t.cpu().numpy().view(dtype)
    if a.dtype.kind == "f" or a.dtype.itemsize <= 2:
        return a.astype(np.float32)
    return a.astype(np.float64)


def write_dumps(directory, arrays):
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte budget")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)
