"""Host-side logic added in round 2 (no GPU): the BASELINE workloads as data, the channel sampler of the parity checks, the strong-scaling
shard plan of config 5, the NUMA helper's parsing, and bench.py's reference arm on a bounded sample."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_workload_shapes(msdr, K):
    w3, w4, w5 = (msdr.workloads.get(n, K) for n in ("c3", "c4", "c5"))
    assert (w3.channels, w3.blocks, w3.blocks_per_update, w3.scaling) == (4096, 3446, 1024, "weak")      # 10 s at 44.1 kHz
    assert (w4.channels, w4.blocks, w4.max_taps, w4.fs) == (16384, 1500, 256, 192000.0)                  # 1 s at 192 kHz
    assert (w5.channels, w5.blocks, w5.blocks_per_update, w5.scaling, w5.stream_seconds) == (1 << 20, 128, 32, "strong", 60.0)
    assert w3.modes(8, ch0=2) == [msdr.capi.MODE_LSB, msdr.capi.MODE_CW, msdr.capi.MODE_AM, msdr.capi.MODE_USB] * 2
    for md, (cI, cQ) in w4.tables.items():   # 255 designed taps + the zero arm_fir_init_q15 asks for (arm_fir_init_q15.c:55-64)
        assert cI.size == cQ.size == 256 and cI[-1] == 0 and cQ[-1] == 0 and cI.dtype == np.int16
        if md != msdr.capi.MODE_AM:
            assert np.array_equal(cQ[:255], cI[:255][::-1])   # the relation of the sketch's +-45 degree tables (Minimal-SDR.ino:119-128)
    assert int(np.abs(w4.tables[msdr.capi.MODE_AM][0]).sum()) > 30000
    assert w3.tables_for(msdr.capi.MODE_SYNCAM)[0] is w3.tables_for(msdr.capi.MODE_AM)[0]   # init_FIR binds the AM table for SYNCAM (.ino:904-929)


def test_configure_uses_one_call_per_mode(msdr, K):
    """Workload.configure on a recording stand-in: AM for everything, then ONE list call per other mode (2^20 channels stay cheap)."""
    calls = []

    class Rec:
        n_channels = 1000

        def __getattr__(self, name):
            return lambda *a, **k: calls.append((name, a))

    w = msdr.workloads.get("c5", K)
    modes = w.configure(Rec(), ch0=3)
    names = [c[0] for c in calls]
    assert names.count("set_mode_list") == 3 and names.count("fir_init_list") == 3 and names.count("set_mode") == 1 and names.count("fir_init") == 1
    for name, a in calls:
        if name == "set_mode_list":
            md, ch = a
            assert all(modes[c] == md for c in ch) and len(ch) == sum(1 for m_ in modes if m_ == md)


def test_sample_channels(msdr):
    for C in (1, 5, 48, 203, 4096, 1 << 20):
        s = msdr.workloads.sample_channels(C)
        assert s == sorted(set(s)) and len(s) == min(48, C) and s[0] == 0 and s[-1] == C - 1
        if C >= 4096:
            assert {31, 32, 33, 127, 128, C - 33, C - 32}.issubset(s)   # group and tile edges
    assert msdr.workloads.sample_channels(4096) == msdr.workloads.sample_channels(4096)   # seeded


def test_c5_strong_scaling_plan(msdr):
    for world in (1, 2, 4, 8):
        sh = msdr.shard.plan(1 << 20, world)
        assert [s.n for s in sh] == [(1 << 20) // world] * world and all(s.ch0 % 128 == 0 for s in sh)


def test_numa_helper_parsing(msdr):
    assert msdr.shard._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert msdr.shard._parse_cpulist("") == set()
    info = msdr.shard.bind_to_gpu_numa(0)   # no GPU here: reports why it did nothing, never raises
    assert info["bound"] is False


def test_dump_sample_is_the_last_step_in_stream_order(msdr, monkeypatch):
    """bench.py --dump-outputs: sampled rows of every update's output buffer, in stream order, within DUMP_BYTES as float32."""
    import torch
    import bench
    C, ups = 300, [4, 4, 2]
    L = sum(ups) * 128
    ys = [torch.randint(-32768, 32768, (C, nb * 128 + 128), dtype=torch.int16) for nb in ups]  # a buffer may outsize its update
    calls = [(None, y, nb, y.stride(0)) for y, nb in zip(ys, ups)]
    full = torch.cat([y[:, :nb * 128] for y, nb in zip(ys, ups)], dim=1)
    shapes = []
    for budget in (64_000_000, 4 * L * 40, 4 * L * 2):  # every channel; 40 whole rows; the fixed edge channels, leading samples only
        monkeypatch.setattr(bench, "DUMP_BYTES", budget)
        got, chans = bench.output_sample(msdr, calls, C, L)
        assert chans == msdr.workloads.sample_channels(C, want=max(1, budget // (4 * L)))
        assert 4 * got.numel() <= budget and torch.equal(got, full[chans, :got.shape[1]])
        shapes.append(tuple(got.shape))
    assert shapes[0] == (C, L) and shapes[1] == (40, L) and 20 < shapes[2][0] < 40 and shapes[2][1] < L


def test_reference_arm_line_says_what_ran():
    import oracle_lib as ol
    # the reference's own sources where they were built (oracle/_ref), else the oracle port of them
    build, kind = ("gcc -O2", "reference") if ol.have_ref() else ("gcc -O2 (oracle port)", "port")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--config", "c4"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["value"] > 0 and d["config"]["config"] == "c4"
    assert "reference arm:" in d["config"]["ran"] and "256-tap" in d["config"]["ran"]
    assert set(d["cpu_baseline"]["builds"]) >= {build} and d["cpu_baseline"]["kind"] == kind and d["e2e"]["h2d_bytes_per_step"] == 0
