#!/usr/bin/env python3
"""Receive chain from raw ADC codes on one GPU, device-resident: three arms timed in the same process on the same seeded inputs,
alternating round by round.

  int16        msdr_chain_update_device on conditioned int16 IF samples (the chain alone)
  composition  msdr_frontend_update_device + msdr_chain_update_device on one stream (two objects, IF samples through HBM)
  fused        msdr_chain_update_adc_device (one object; the front end inside the row-block converters where they run)

  python tools/bench_adc.py [--shapes c5:131072,c5:1048576,c4,c3] [--rounds 5] [--reps 4]

Codes are 12-bit, (x >> 4) + 2048 of synth.torch_batch, generated on the device.  Before the timed rounds every arm runs one update on
fresh chains and 48 sampled channels (workloads.sample_channels) are compared with the CPU oracles (oracle/msdr_oracle.c), front end
then chain.  Prints one JSON line.  There is no CPU fallback: without a GPU the script fails.
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

BLOCK = 128


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        vals = [v.strip() for v in r.stdout.strip().split(",")]
        return dict(zip(q.split(","), vals))
    except Exception as e:  # the line still says what was not read
        return {"error": str(e)}


def shape_list(s, K, m):
    out = []
    for item in s.split(","):
        name, _, nch = item.partition(":")
        wl = m.workloads.get(name, K)
        C = int(nch) if nch else wl.channels
        out.append((f"{name}:{C}", wl, C, wl.blocks_per_update))
    return out


def make_chain(m, wl, C, frontend=False):
    g = m.ReceiveChain(C, max_taps=wl.max_taps)
    wl.configure(g)
    if frontend:
        g.enable_frontend()
    return g


def oracle_pair(orc, forc, wl, modes, chans):
    o = orc.chain(len(chans))
    for i, c in enumerate(chans):
        o.set_mode(i, 1, modes[c])
        assert o.fir_init(i, 1, *wl.tables_for(modes[c])) == 0
    o.biquad_set_coefficients(0, 0, len(chans), 0, wl.biquad1)
    o.biquad_set_coefficients(1, 0, len(chans), 0, wl.biquad2)
    return o, forc.frontend(len(chans))


def run_shape(m, torch, orc, forc, label, wl, C, nb, rounds, reps):
    L = nb * BLOCK
    x = m.synth.torch_batch(C, L, "cuda")                         # int16 IF samples (the int16 arm's input)
    codes = ((x.to(torch.int32) >> 4) + 2048).to(torch.int16)    # 12-bit ADC codes, the same bits as uint16
    y = {a: torch.empty_like(x) for a in ("int16", "composition", "fused")}
    xif = torch.empty_like(x)
    torch.cuda.synchronize()

    def arms():
        g16 = make_chain(m, wl, C)
        gc = make_chain(m, wl, C)
        fe = m.Frontend(C)
        gf = make_chain(m, wl, C, frontend=True)
        for obj in (g16, gc, fe, gf):  # one stream (torch's, where the events are recorded): the composition's two kernels in order
            obj.set_stream(0)
        s = x.stride(0)
        return {
            "int16": (lambda: g16.update_device(x.data_ptr(), y["int16"].data_ptr(), nb, s), g16),
            "composition": (lambda: (fe.update_device(codes.data_ptr(), xif.data_ptr(), nb, s),
                                     gc.update_device(xif.data_ptr(), y["composition"].data_ptr(), nb, s)), gc),
            "fused": (lambda: gf.update_adc_device(codes.data_ptr(), y["fused"].data_ptr(), nb, s), gf),
        }

    # parity: one update of every arm on fresh chains, sampled channels against the CPU oracles
    A = arms()
    for a, (fn, g) in A.items():
        fn()
        torch.cuda.synchronize()
        g.synchronize()
    chans = m.workloads.sample_channels(C)
    modes = wl.modes(C)
    o16, _ = oracle_pair(orc, forc, wl, modes, chans)
    o_fe, fo = oracle_pair(orc, forc, wl, modes, chans)
    ref16 = o16.run(np.ascontiguousarray(x[chans].cpu().numpy()))[0]
    ref_adc = o_fe.run(fo.run(np.ascontiguousarray(codes[chans].cpu().numpy().view(np.uint16))))[0]
    mism = {a: int((y[a][chans].cpu().numpy() != (ref16 if a == "int16" else ref_adc)).sum()) for a in y}
    fused_eq_comp = bool(torch.equal(y["fused"], y["composition"]))
    kernels = {a: g.last_kernel() for a, (fn, g) in A.items()}

    # timed rounds: the arms alternate; each measurement is `reps` consecutive updates between CUDA events (state carries)
    times = {a: [] for a in A}
    for a, (fn, g) in A.items():  # warm-up of every shape and plan
        fn()
    torch.cuda.synchronize()
    for r in range(rounds):
        for a, (fn, g) in A.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps):
                fn()
            g.synchronize()
            e1.record()
            e1.synchronize()
            times[a].append(e0.elapsed_time(e1) / 1e3)
    samples = C * L * reps
    gs = {a: samples / min(t) / 1e9 for a, t in times.items()}
    spread = {a: (max(t) - min(t)) / min(t) for a, t in times.items()}
    del A
    torch.cuda.empty_cache()
    return {
        "shape": label, "channels": C, "blocks_per_update": nb, "updates_per_measurement": reps, "rounds": rounds,
        "gsamples_per_s": {a: round(v, 2) for a, v in gs.items()},
        "spread_max_over_min": {a: round(v, 4) for a, v in spread.items()},
        "fused_over_int16": round(gs["fused"] / gs["int16"], 4),
        "fused_over_composition": round(gs["fused"] / gs["composition"], 4),
        "last_kernel": kernels,
        "parity": {"channels": len(chans), "mismatches": mism, "fused_equals_composition": fused_eq_comp},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="c5:131072,c5:1048576,c4,c3")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=4)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_adc.py: no CUDA device (this library has no CPU fallback)")
    import frontend_lib as fl
    import minimal_sdr_b200 as m
    import oracle_lib as ol
    K = m.load_ref_constants()
    orc, forc = ol.CheckerLib("orc"), fl.Orc()
    info_before = gpu_info()
    results = [run_shape(m, torch, orc, forc, *s, args.rounds, args.reps) for s in shape_list(args.shapes, K, m)]
    print(json.dumps({"bench": "chain_adc", "gpu": info_before, "gpu_after": gpu_info(), "results": results}))


if __name__ == "__main__":
    main()
