#!/usr/bin/env python3
"""Snapshots of a whole C5 chain on one GPU: how fast a checkpoint is taken and restored, against plain copies of the same bytes and
against the per-channel state calls.

  python tools/bench_snapshot.py [--channels 1048576] [--rounds 5] [--loop-channels 4096] [--out FILE]

Two configurations of workloads.get("c5"): 2^20 channels, mixed modes, 102-tap maximum; then the same with ANR 2 on the first eighth of
the channels and the front end enabled.  Each chain first runs one update, so the state is not the initial one.  Timed, in this process:

  snapshot / restore           msdr_chain_snapshot / msdr_chain_restore on a pinned host buffer (host clock; both calls return when done)
  pinned_d2h / pinned_h2d      a plain cudaMemcpyAsync of the same byte count between a device buffer and the same pinned buffer
  snapshot_device / restore_device   on a device buffer, to the chain's stream being synchronised, as GB/s of snapshot bytes
  per_channel_loop             get_state (+ get_anr_state, get_frontend_state) and the matching setters over `--loop-channels`
                               channels; `extrapolated_to_all_channels_s` scales that linearly and is not a measurement

The restored chain's own snapshot must equal the one it was restored from, byte for byte.  Prints one JSON line (and writes it to --out).
There is no CPU fallback: without a GPU the script fails.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        vals = [v.strip() for v in r.stdout.strip().split(",")]
        return dict(zip(q.split(","), vals))
    except Exception as e:  # the line still says what was not read
        return {"error": str(e)}


def timed(fn, rounds):
    ts = []
    for _ in range(rounds):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return {"min_s": round(min(ts), 6), "median_s": round(statistics.median(ts), 6)}


def run_config(m, torch, K, C, label, anr_fe, rounds, loop_n):
    wl = m.workloads.get("c5", K)
    nb = 4

    def chain():
        g = m.ReceiveChain(C, max_taps=wl.max_taps)
        wl.configure(g)
        if anr_fe:
            g.set_anr(2, 0, C // 8)
            g.enable_frontend()
        return g
    g = chain()
    x = m.synth.torch_batch(C, nb * 128, "cuda")
    y = torch.empty_like(x)
    torch.cuda.synchronize()
    g.update_device(x.data_ptr(), y.data_ptr(), nb, x.stride(0))
    g.synchronize()
    del x, y
    nbytes = g.snapshot_bytes()
    host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    hview = host.numpy()
    dev = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    dev2 = torch.empty_like(dev)
    r = m.ReceiveChain(C, max_taps=wl.max_taps)  # bare: the first restore configures it

    res = {"config": label, "channels": C, "snapshot_bytes": nbytes, "bytes_per_channel": round(nbytes / C, 2)}
    # warm-up of every path, and the parity check
    g.snapshot(out=hview)
    r.restore(hview)
    check = np.empty(nbytes, np.uint8)
    r.snapshot(out=check)
    res["restored_snapshot_equal"] = bool(np.array_equal(check, hview))
    del check
    g.snapshot_device(0, C, dev)
    r.restore_device(dev, 0, 0, C)
    r.synchronize()
    g.synchronize()

    def d2h():
        host.copy_(dev, non_blocking=True)
        torch.cuda.synchronize()

    def h2d():
        dev2.copy_(host, non_blocking=True)
        torch.cuda.synchronize()

    def d2d():
        dev2.copy_(dev, non_blocking=True)
        torch.cuda.synchronize()

    def snap_dev():
        g.snapshot_device(0, C, dev)
        g.synchronize()

    def rest_dev():
        r.restore_device(dev, 0, 0, C)
        r.synchronize()

    t = {}
    for _ in range(rounds):  # arms alternate round by round
        for name, fn in (("snapshot", lambda: g.snapshot(out=hview)), ("pinned_d2h", d2h), ("restore", lambda: r.restore(hview)),
                         ("pinned_h2d", h2d), ("snapshot_device", snap_dev), ("restore_device", rest_dev), ("plain_d2d", d2d)):
            t.setdefault(name, []).append(timed(fn, 1)["min_s"])
    for name, ts in t.items():
        res[name] = {"min_s": min(ts), "median_s": statistics.median(ts), "gb_per_s": round(nbytes / min(ts) / 1e9, 2)}
    res["snapshot_over_pinned_d2h"] = round(res["snapshot"]["min_s"] / res["pinned_d2h"]["min_s"], 3)
    res["restore_over_pinned_h2d"] = round(res["restore"]["min_s"] / res["pinned_h2d"]["min_s"], 3)

    # the per-channel calls on a slice
    states = []
    t0 = time.perf_counter()
    for c in range(loop_n):
        s = (g.get_state(c), g.get_anr_state(c) if anr_fe else None, g.get_frontend_state(c) if anr_fe else None)
        states.append(s)
    t_get = time.perf_counter() - t0
    t0 = time.perf_counter()
    for c, (s, a, f) in enumerate(states):
        r.set_state(c, s)
        if anr_fe:
            r.set_anr_state(c, a)
            r.set_frontend_state(c, f)
    r.synchronize()
    t_set = time.perf_counter() - t0
    res["per_channel_loop"] = {"channels": loop_n, "get_s": round(t_get, 4), "set_s": round(t_set, 4),
                               "extrapolated_to_all_channels_s": {"get": round(t_get * C / loop_n, 2), "set": round(t_set * C / loop_n, 2)}}
    del host, dev, dev2
    g.close()
    r.close()
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=1 << 20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--loop-channels", type=int, default=4096)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_snapshot.py: no CUDA device (this library has no CPU fallback)")
    import minimal_sdr_b200 as m
    K = m.load_ref_constants()
    info_before = gpu_info()
    results = [run_config(m, torch, K, args.channels, "c5", False, args.rounds, args.loop_channels),
               run_config(m, torch, K, args.channels, "c5 + ANR on 1/8 + front end", True, args.rounds, args.loop_channels)]
    line = json.dumps({"bench": "chain_snapshot", "gpu": info_before, "gpu_after": gpu_info(), "results": results})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
