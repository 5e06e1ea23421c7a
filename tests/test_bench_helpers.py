"""CPU checks of the bench plumbing (bench_common): byte accounting of the roofline objects, the traffic
record's source hash, the clock sampler's behaviour on a machine without NVML / nvidia-smi, and the
--dump-outputs helpers."""
import json
import os

import numpy as np
import pytest

import bench_common as bc


def test_k1_byte_accounting_matches_survey_8d():
    # dual return, float: 64 B per pixel algorithmic; compulsory = 40 B per pixel per frame + the LUT once
    h, w, r, f = 128, 2048, 2, 64
    alg, comp = bc.k1_bytes(h, w, r, f)
    assert alg == f * h * w * 64 == 1073741824
    assert comp == f * h * w * 40 + h * w * 24 == 677380096
    # per-stream LUTs are each counted once
    assert bc.k1_bytes(h, w, r, f, n_luts=8)[1] == f * h * w * 40 + 8 * h * w * 24


def test_k2_byte_accounting_matches_design():
    h, w, r, f = 128, 2048, 2, 32
    psz, cpp, fbytes = 33024, 16, 19
    alg, comp = bc.k2_bytes(h, w, r, f, psz, cpp, fbytes)
    per_frame = (w // cpp) * psz + fbytes * h * w + 24 * h * w + 8 * h * w + 14 * w + 9 * (w // cpp)
    assert per_frame == 17626240
    assert comp == f * per_frame + h * w * 24 == 570331136
    assert alg == f * (per_frame + h * w * 24) == 765366272


def test_traffic_record_is_only_quoted_for_identical_sources():
    """The committed ncu traffic records carry the hash of the kernel sources they were captured for; bench.py
    quotes `roofline.traffic` only while that hash matches (a record for other sources reads as stale)."""
    sha = bc.source_sha(bc.K1_SOURCES)
    assert len(sha) >= 16 and sha == bc.source_sha(bc.K1_SOURCES) and sha != bc.source_sha(bc.K2_SOURCES)
    for name, src in (("k1_traffic.json", bc.K1_SOURCES), ("k2_traffic.json", bc.K2_SOURCES),
                      ("k2_streams8_traffic.json", bc.K2_SOURCES)):
        path = os.path.join(bc.ROOT, "profiles", name)
        if not os.path.exists(path):
            continue
        rec = json.load(open(path))
        got = bc.read_traffic(name, src)
        if rec.get("source_sha") == bc.source_sha(src):
            assert got["dram_bytes_per_launch"] == rec["dram_bytes_per_launch"]
        else:
            assert "dram_bytes_per_launch" not in got and got["record"].startswith("stale")
    assert bc.read_traffic("no_such_record.json", bc.K1_SOURCES) == {"record": "none"}


def test_clock_sampler_without_gpu_reports_unavailable_or_samples():
    s = bc.ClockSampler(0)
    s.start()
    s.mark()
    s.mark()
    out = s.stop()
    assert "sm_mhz" in out and "reasons" in out
    if out["sm_mhz"] is None:
        assert out.get("samples", 0) == 0 or out["reasons"] == ["unavailable"] or out.get("source") in ("nvml", "nvidia-smi")


def test_dump_helpers_sample_reproducibly_and_convert_exactly(tmp_path):
    """--dump-outputs: the sample is fixed by its seed, and values the device tensors carry in signed types
    come out as the unsigned values they are, in a float type that holds them exactly."""
    torch = pytest.importorskip("torch")
    a, b = bc.dump_index(torch, "cpu", 1000, 100, seed=1), bc.dump_index(torch, "cpu", 1000, 100, seed=1)
    assert torch.equal(a, b) and len(torch.unique(a)) == 100 and bool((a[1:] > a[:-1]).all())
    assert torch.equal(bc.dump_index(torch, "cpu", 10, 100, seed=1), torch.arange(10))
    u16 = bc.dump_array(torch.tensor([-1, 7], dtype=torch.int16), np.uint16)
    u32 = bc.dump_array(torch.tensor([-1, 7], dtype=torch.int32), np.uint32)
    assert u16.dtype == np.float32 and u16.tolist() == [65535.0, 7.0]
    assert u32.dtype == np.float64 and u32.tolist() == [4294967295.0, 7.0]
    assert bc.dump_array(torch.tensor([0.1], dtype=torch.float32), np.float32).dtype == np.float32
    bc.write_dumps(str(tmp_path / "d"), {"x": u32})
    assert np.array_equal(np.load(tmp_path / "d" / "x.npy"), u32)
    with pytest.raises(SystemExit):
        bc.write_dumps(str(tmp_path / "e"), {"big": np.zeros(bc.DUMP_MAX_BYTES // 8 + 1)})
