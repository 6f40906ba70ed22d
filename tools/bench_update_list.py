#!/usr/bin/env python3
"""Channel-list updates against range updates on one GPU, device-resident, C5 modes and tables, 32 blocks per update.  Every arm
has its own chain; the arms run in one process on the same seeded inputs, alternating round by round.

  row-block case, a 2^20-channel chain:
    list_random   msdr_chain_update_list_device over 131 072 seeded random channels in random order
    list_runs     the same call over 64 runs of 2048 channels (a list of the same size)
    ranges_64     those 64 runs as 64 msdr_chain_update_range_device calls, as callers do without lists (each run keeps its
                  cached plan: the most favourable case for range calls)
    range         one range of 131 072 contiguous channels, the ceiling
  few-channel case, a 65 536-channel chain: a list of 4096 scattered channels against a 4096-channel range (both time-folded)
  middle case, the same chain size: a list of 8192 scattered channels (row-block kernel) against an 8192-channel range (chain
                  kernel v4, which has no list form)

  python tools/bench_update_list.py [--rounds 5] [--reps 3] [--cases rowblock,few,middle]
  MSDR_PROF=1 python tools/bench_update_list.py --prof     # one update of list_random and range each, role counters on stderr

Before the timed rounds every arm runs one update on fresh chains and 48 sampled rows of it are compared byte for byte with the CPU
oracle (oracle/msdr_oracle.c); a mismatch ends the script with an error before anything is timed.  Prints the card name, power
limit and SM clock with one JSON line.  There is no CPU fallback: without a GPU the script fails.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

BLOCK, NB = 128, 32


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        vals = [v.strip() for v in r.stdout.strip().split(",")]
        return dict(zip(q.split(","), vals))
    except Exception as e:  # the line still says what was not read
        return {"error": str(e)}


def make_chain(m, wl, C):
    g = m.ReceiveChain(C, max_taps=wl.max_taps)
    wl.configure(g)
    g.set_stream(0)  # torch's stream, where the events are recorded
    return g


def oracle(orc, wl, modes, chans):
    o = orc.chain(len(chans))
    for i, c in enumerate(chans):
        o.set_mode(i, 1, modes[c])
        assert o.fir_init(i, 1, *wl.tables_for(modes[c])) == 0
    o.biquad_set_coefficients(0, 0, len(chans), 0, wl.biquad1)
    o.biquad_set_coefficients(1, 0, len(chans), 0, wl.biquad2)
    return o


def arms_for(case, rng):
    """{arm: (chain channels, [(kind, channels)])}: kind 'list' = one list call over `channels`, 'range' = one range call over
    channels[0] .. channels[-1]; the calls of an arm together take rows 0 .. n of the input in order."""
    if case == "rowblock":
        C, n, run = 1 << 20, 131072, 2048
        scattered = rng.permutation(C)[:n]
        starts = rng.permutation(C // run)[:n // run] * run
        runs = [np.arange(s, s + run) for s in starts]
        return C, {
            "list_random": [("list", scattered)],
            "list_runs": [("list", np.concatenate(runs))],
            "ranges_64": [("range", r) for r in runs],
            "range": [("range", np.arange(n))],
        }
    C = 65536
    n = 4096 if case == "few" else 8192
    return C, {"list": [("list", rng.permutation(C)[:n])], "range": [("range", np.arange(n))]}


def run_case(m, torch, orc, wl, case, rounds, reps, prof=False):
    rng = np.random.default_rng(7)
    C, spec = arms_for(case, rng)
    n = sum(len(ch) for _, ch in next(iter(spec.values())))
    L = NB * BLOCK
    x = m.synth.torch_batch(n, L, "cuda")  # row r of every arm's input is the r-th channel it updates
    s = x.stride(0)
    modes = wl.modes(C)
    torch.cuda.synchronize()
    arms = {}
    for a, calls in spec.items():
        g = make_chain(m, wl, C)
        y = torch.empty_like(x)
        steps, r0 = [], 0
        for kind, ch in calls:
            pin, pout = x[r0:].data_ptr(), y[r0:].data_ptr()
            if kind == "list":
                chl = np.ascontiguousarray(ch, np.uint32)
                steps.append(lambda g=g, chl=chl, pin=pin, pout=pout: g.update_list_device(chl, pin, pout, NB, s))
            else:
                steps.append(lambda g=g, c0=int(ch[0]), k=len(ch), pin=pin, pout=pout: g.update_range_device(c0, k, pin, pout, NB, s))
            r0 += len(ch)
        order = np.concatenate([ch for _, ch in calls])
        arms[a] = (steps, g, y, order)
        if prof and a not in ("list_random", "range"):
            del arms[a]

    # parity: one update of every arm on its fresh chain, 48 sampled rows against the CPU oracle
    rows = m.workloads.sample_channels(n)
    xs = np.ascontiguousarray(x[rows].cpu().numpy())
    mism, kernels = {}, {}
    for a, (steps, g, y, order) in arms.items():
        for f in steps:
            f()
        g.synchronize()
        kernels[a] = g.last_kernel()
        ref = oracle(orc, wl, modes, [int(order[r]) for r in rows]).run(xs)[0]
        mism[a] = int((y[rows].cpu().numpy() != ref).sum())
    if any(mism.values()):  # a rate of wrong outputs is no rate
        raise SystemExit(f"bench_update_list.py: {case}: sampled rows differ from the oracle: {mism}; kernels {kernels}")
    if prof:
        return {"case": case, "last_kernel": kernels, "parity_mismatches": mism}

    times = {a: [] for a in arms}
    for a, (steps, g, y, order) in arms.items():  # warm-up: every plan is cached, every kernel loaded
        for f in steps:
            f()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for a, (steps, g, y, order) in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps):
                for f in steps:
                    f()
            e1.record()
            e1.synchronize()
            times[a].append(e0.elapsed_time(e1) / 1e3)
    samples = n * L * reps
    gs = {a: samples / min(t) / 1e9 for a, t in times.items()}
    ceiling = gs["range"]
    out = {
        "case": case, "chain_channels": C, "rows_per_update": n, "blocks_per_update": NB, "updates_per_measurement": reps, "rounds": rounds,
        "gsamples_per_s": {a: round(v, 2) for a, v in gs.items()},
        "over_range": {a: round(v / ceiling, 4) for a, v in gs.items()},
        "spread_max_over_min": {a: round((max(t) - min(t)) / min(t), 4) for a, t in times.items()},
        "seconds": {a: [round(v, 6) for v in t] for a, t in times.items()},
        "last_kernel": kernels,
        "parity": {"rows": len(rows), "mismatches": mism},
    }
    del arms
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="rowblock,few,middle")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--prof", action="store_true", help="one untimed update of list_random and range (run with MSDR_PROF=1)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_update_list.py: no CUDA device (this library has no CPU fallback)")
    import minimal_sdr_b200 as m
    import oracle_lib as ol
    K = m.load_ref_constants()
    wl = m.workloads.get("c5", K)
    orc = ol.CheckerLib("orc")
    info = gpu_info()
    print(f"# {info.get('name')}, power limit {info.get('power.limit')}, SM clock {info.get('clocks.sm')} (max {info.get('clocks.max.sm')})",
          file=sys.stderr)
    if args.prof:
        print(json.dumps(run_case(m, torch, orc, wl, "rowblock", 1, 1, prof=True)))
        return
    results = [run_case(m, torch, orc, wl, c, args.rounds, args.reps) for c in args.cases.split(",")]
    print(json.dumps({"bench": "update_list", "gpu": info, "gpu_after": gpu_info(), "results": results}))


if __name__ == "__main__":
    main()
