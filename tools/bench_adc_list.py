#!/usr/bin/env python3
"""Channel-list updates from raw ADC codes on one GPU, device-resident, C5 modes and tables, 32 blocks per update.  Every arm has
its own chain; the arms run in one process on the same seeded codes, alternating round by round.

  row-block case, a 2^20-channel chain with the front end enabled:
    adc_list      msdr_chain_update_adc_list_device over 131 072 seeded random channels in random order (the front-end kernel with
                  the list as its state map, then the int16 list kernel)
    adc_range     msdr_chain_update_adc_range_device over 131 072 contiguous channels (front end fused, v5)
    composition   a stand-alone msdr_frontend over the list's rows, then msdr_chain_update_list_device (two objects, IF samples
                  through HBM), as tools/bench_adc.py composes for ranges
    int16_list    msdr_chain_update_list_device over the same channels on int16 IF samples
  few-channel case, a 65 536-channel chain: an ADC list of 4096 scattered channels (the front-end kernel, then the time-folded
                  list kernel) against a 4096-channel ADC range

  python tools/bench_adc_list.py [--rounds 5] [--reps 3] [--cases rowblock,few]

Before the timed rounds every arm runs one update on fresh chains and 48 sampled rows of it are compared byte for byte with the
CPU front-end oracle followed by the CPU chain oracle (the int16 arm with the chain oracle alone); a mismatch ends the script with
an error before anything is timed.  Prints the card name, power limit and SM clock with one JSON line.  There is no CPU fallback:
without a GPU the script fails.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

from bench_update_list import gpu_info, make_chain, oracle  # noqa: E402

BLOCK, NB = 128, 32


def run_case(m, torch, orc, forc, wl, case, rounds, reps):
    rng = np.random.default_rng(7)
    C, n = (1 << 20, 131072) if case == "rowblock" else (65536, 4096)
    chans = np.ascontiguousarray(rng.permutation(C)[:n], np.uint32)
    L = NB * BLOCK
    x = m.synth.torch_batch(n, L, "cuda")                          # row r of every arm's input is the r-th channel it updates
    codes = ((x.to(torch.int32) >> 4) + 2048).to(torch.int16)    # 12-bit ADC codes, the same bits as uint16
    s = x.stride(0)
    modes = wl.modes(C)
    torch.cuda.synchronize()

    def chain(frontend):
        g = make_chain(m, wl, C)
        if frontend:
            g.enable_frontend()
        return g

    arms = {}
    g = chain(True)
    y = torch.empty_like(x)
    arms["adc_list"] = (lambda g=g, y=y: g.update_adc_list_device(chans, codes.data_ptr(), y.data_ptr(), NB, s), g, y, chans)
    g = chain(True)
    y = torch.empty_like(x)
    arms["adc_range"] = (lambda g=g, y=y: g.update_adc_range_device(0, n, codes.data_ptr(), y.data_ptr(), NB, s), g, y, np.arange(n))
    if case == "rowblock":
        g = chain(False)
        y, xif = torch.empty_like(x), torch.empty_like(x)
        fe = m.Frontend(n)
        fe.set_stream(0)
        arms["composition"] = (lambda g=g, y=y, fe=fe, xif=xif: (fe.update_device(codes.data_ptr(), xif.data_ptr(), NB, s),
                                                                    g.update_list_device(chans, xif.data_ptr(), y.data_ptr(), NB, s)), g, y, chans)
        g = chain(False)
        y = torch.empty_like(x)
        arms["int16_list"] = (lambda g=g, y=y: g.update_list_device(chans, x.data_ptr(), y.data_ptr(), NB, s), g, y, chans)

    # parity: one update of every arm on its fresh chain, 48 sampled rows against the front-end oracle and the chain oracle
    rows = m.workloads.sample_channels(n)
    xs = np.ascontiguousarray(x[rows].cpu().numpy())
    cs = np.ascontiguousarray(codes[rows].cpu().numpy().view(np.uint16))
    if_rows = forc.frontend(len(rows)).run(cs)  # every sampled row is a distinct channel from its initial front-end state
    mism, kernels = {}, {}
    for a, (f, g, y, order) in arms.items():
        f()
        g.synchronize()
        torch.cuda.synchronize()
        kernels[a] = g.last_kernel()
        ref = oracle(orc, wl, modes, [int(order[r]) for r in rows]).run(xs if a == "int16_list" else if_rows)[0]
        mism[a] = int((y[rows].cpu().numpy() != ref).sum())
    if any(mism.values()):  # a rate of wrong outputs is no rate
        raise SystemExit(f"bench_adc_list.py: {case}: sampled rows differ from the oracles: {mism}; kernels {kernels}")

    times = {a: [] for a in arms}
    for f, *_ in arms.values():  # warm-up: every plan is cached, every kernel loaded
        f()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for a, (f, *_) in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps):
                f()
            e1.record()
            e1.synchronize()
            times[a].append(e0.elapsed_time(e1) / 1e3)
    samples = n * L * reps
    gs = {a: samples / min(t) / 1e9 for a, t in times.items()}
    med = {a: samples / float(np.median(t)) / 1e9 for a, t in times.items()}
    out = {
        "case": case, "chain_channels": C, "rows_per_update": n, "blocks_per_update": NB, "updates_per_measurement": reps, "rounds": rounds,
        "gsamples_per_s": {a: round(v, 2) for a, v in gs.items()},
        "gsamples_per_s_median_round": {a: round(v, 2) for a, v in med.items()},
        "over_adc_range": {a: round(v / gs["adc_range"], 4) for a, v in gs.items()},
        "spread_max_over_min": {a: round((max(t) - min(t)) / min(t), 4) for a, t in times.items()},
        "seconds": {a: [round(v, 6) for v in t] for a, t in times.items()},
        "last_kernel": kernels,
        "parity": {"rows": len(rows), "mismatches": mism},
    }
    if "composition" in gs:
        out["adc_list_over_composition"] = round(gs["adc_list"] / gs["composition"], 4)
    del arms
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="rowblock,few")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_adc_list.py: no CUDA device (this library has no CPU fallback)")
    import minimal_sdr_b200 as m
    import frontend_lib as fl
    import oracle_lib as ol
    K = m.load_ref_constants()
    wl = m.workloads.get("c5", K)
    orc, forc = ol.CheckerLib("orc"), fl.Orc()
    info = gpu_info()
    print(f"# {info.get('name')}, power limit {info.get('power.limit')}, SM clock {info.get('clocks.sm')} (max {info.get('clocks.max.sm')})",
          file=sys.stderr)
    results = [run_case(m, torch, orc, forc, wl, c, args.rounds, args.reps) for c in args.cases.split(",")]
    print(json.dumps({"bench": "update_adc_list", "gpu": info, "gpu_after": gpu_info(), "results": results}))


if __name__ == "__main__":
    main()
