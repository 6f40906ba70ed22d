#!/usr/bin/env python3
"""Benchmark of the receive DSP chain (fs/4 mix -> FIR pair -> SSB/AM demod -> biquad cascade), BASELINE.json metric:
demodulated Msamples/s summed over all channels, and % of the HBM roofline.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference ...                     (the reference's own C chain on the host cores)
  python bench.py --config c3|c4|c5 ...                    (default c3, the single-GPU configuration BASELINE names)
  python bench.py ... --dump-outputs DIR                   (also write the last timed step's audio, sampled, to DIR/audio.npy)

Workloads (minimal-sdr_b200/workloads.py):
  c3  4096 channels x 10 s at 44.1 kHz per GPU (3446 blocks of 128 samples), mode = {AM, USB, LSB, CW}[c mod 4], the sketch's FIR
      tables and live biquad cascade; N GPUs = N independent shards of that size (weak scaling)
  c4  16 384 channels, 255(+1)-tap FIR pair, 192 kHz, 1 s per GPU, through the fused chain (weak scaling)
  c5  2^20 channels in total, split over the N GPUs of the job (strong scaling), streamed in updates of 32 blocks with state
      carried; a step is 128 blocks (0.37 s) of the 60 s stream, `stream` in the JSON line scales it to the whole stream
One "step" is one pass over the step's signal, fed in updates of --blocks-per-update blocks.  No collective on the data path.
After the timed regions a fresh chain re-runs the first two updates (and the end-to-end call) and sampled channels are compared
with the CPU checker (oracle/_ref when it travelled): `parity_checked`.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

BLOCK = 128
ALGO_BYTES_PER_SAMPLE = 4  # 2 B int16 IF in + 2 B int16 audio out (SURVEY.md 8d)
DUMP_BYTES = 64_000_000  # --dump-outputs: upper bound of the float32 sample it writes
LATENCY_BOUND_CYCLES = 18.0  # loop-carried latency of one biquad stage: IMAD.HI 9 + SHF 4 + I2IP 4 (+1), profiles/r01_microbench_lat.txt
ISSUE_BOUND_CYCLES = 43.5    # a whole stage in one warp, isolated (tools/microbench/bqstep2.cu)


def ncu_traffic(config):
    """DRAM bytes per launch of the chain kernel from the committed `ncu --set full` capture of this configuration (newest round), with
    the algorithmic bytes of THAT launch, so the two are comparable.  (None, None, None) when there is no capture."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", f"r*_{config}_chain_kernel_ncu_metrics.json")))
    if not files and config == "c3":
        files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_chain_kernel_ncu_metrics.json")))
    if not files:
        return None, None, None
    try:
        with open(files[-1]) as f:
            d = json.load(f)
        algo = d.get("algorithmic_bytes_per_launch")
        if algo is None and os.path.basename(files[-1]).startswith("r01_"):
            algo = 4096 * 1024 * BLOCK * ALGO_BYTES_PER_SAMPLE  # the round-1 capture: one launch of 4096 channels x 1024 blocks
        return float(d["dram_bytes_per_launch"]), (float(algo) if algo else None), os.path.basename(files[-1])
    except Exception:
        return None, None, None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled under the bench load (B200_PROFILING.md recipe).  The sampler runs from before
    the warm-up; samples are time-stamped and the ones inside the timed region are reported.  A default run's timed region is
    ~0.1 s (a few sampler periods), so when fewer than 3 samples fall inside it the samples of the identical load right before
    and after it (warm-up steps, untimed cool-down steps) are used as well and `window` says so."""

    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None
        self.t_load0 = self.t0 = self.t1 = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "window": None}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []
        try:
            for line in open(self.path):
                f = [t.strip() for t in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rows.append((ts, float(f[1]), float(f[2]), [v.lower().startswith("active") for v in f[5:9]]))
                except ValueError:
                    continue
            os.unlink(self.path)
        except Exception:
            pass
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        inside = [r for r in rows if self.t0 is not None and self.t0 <= r[0] <= self.t1]
        window = "timed region"
        if len(inside) < 3:
            inside = [r for r in rows if self.t_load0 is not None and r[0] >= self.t_load0]
            window = "timed region plus the identical untimed load around it (warm-up, cool-down): the region is shorter than 3 sampler periods"
        if inside:
            reasons = sorted({n for r in inside for n, a in zip(names, r[3]) if a})
            out.update(sm_mhz=float(np.median([r[1] for r in inside])), sm_max_mhz=float(max(r[2] for r in inside)), reasons=reasons,
                       samples=len(inside), window=window)
        return out


# ---- CPU side: the reference's own C chain on the host cores ---------------------------------------------------------------------

def cpu_chain(lib, w, modes):
    o = lib.chain(len(modes))
    for c, md in enumerate(modes):
        o.set_mode(c, 1, md)
        o.fir_init(c, 1, *w.tables_for(md))
    o.biquad_set_coefficients(0, 0, len(modes), 0, w.biquad1)
    o.biquad_set_coefficients(1, 0, len(modes), 0, w.biquad2)
    return o


def cpu_libs():
    """[(label, CheckerLib, kind)]: every build of the reference sources that travelled (oracle/Makefile: -O2, -O3 -march=x86-64-v3),
    else the oracle port."""
    import oracle_lib as ol
    out = []
    avx2 = False
    try:
        avx2 = " avx2 " in open("/proc/cpuinfo").read()
    except Exception:
        pass
    if ol.have_ref():
        out.append(("gcc -O2", ol.CheckerLib("ref"), "reference"))
        p = ol.REF_VARIANTS["O3-x86-64-v3"]
        if avx2 and os.path.exists(p):
            out.append(("gcc -O3 -march=x86-64-v3", ol.CheckerLib("ref", path=p), "reference"))
    if not out:
        out.append(("gcc -O2 (oracle port)", ol.CheckerLib("orc"), "port"))
    return out


def time_cpu_one(m, w, lib, target_s, n_threads):
    n_ch = max(4, 4 * n_threads)
    modes = w.modes(n_ch)
    x = np.stack([m.synth.channel_stream(c % 16, modes[c], 64 * BLOCK, w.fs) for c in range(n_ch)])
    o = cpu_chain(lib, w, modes)
    t0 = time.perf_counter()
    _, used = o.run(x, n_threads)
    cal = time.perf_counter() - t0  # calibration pass (also warms the threads)
    reps = int(max(1, min(target_s / max(cal, 1e-4), (1 << 28) / x.size)))  # <= 512 MB of input
    xx = np.ascontiguousarray(np.tile(x, (1, reps)))
    runs, t0 = 0, time.perf_counter()
    while True:
        o.run(xx, n_threads)  # state carries on: one long stream per channel
        runs += 1
        dt = time.perf_counter() - t0
        if dt >= target_s or runs >= 64:
            break
    o.close()
    samples = xx.size * runs
    return {"value": samples / dt / 1e6, "cores": int(used), "seconds": dt, "samples": samples, "channels": n_ch, "blocks": reps * 64 * runs}


def time_cpu(m, w, target_s=8.0, n_threads=0):
    """Reference C chain on the host cores over a bounded sample of the workload, every available build; the fastest is `value`."""
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 1
    n_threads = n_threads or cores  # explicit: torchrun exports OMP_NUM_THREADS=1, which would silently serialise the baseline
    libs = cpu_libs()
    res = {label: (time_cpu_one(m, w, lib, target_s / len(libs), n_threads), kind) for label, lib, kind in libs}
    best = max(res, key=lambda k: res[k][0]["value"])
    r, kind = res[best]
    return {"value": r["value"], "unit": "Msamples/s", "cores": r["cores"], "kind": kind, "build": best,
            "builds": {k: round(v[0]["value"], 2) for k, v in res.items()},
            "sample": f"{r['channels']} channels x {r['blocks']} blocks ({r['samples'] / 1e6:.1f} Msamples in {r['seconds']:.1f} s) of the {w.name.upper()} mode mix "
                      f"({w.max_taps if w.name == 'c4' else '102/86'}-tap tables, 16 distinct streams tiled), "
                      f"{'oracle/_ref: the reference CMSIS/Teensy sources' if kind == 'reference' else 'oracle/msdr_oracle.c port'}, {best}, OpenMP over the channels",
            "seconds": r["seconds"], "samples": r["samples"]}


def run_reference(args, rank, world):
    import minimal_sdr_b200 as m
    if rank != 0:
        return
    w = m.workloads.get(args.config, m.load_ref_constants())
    vals, info = [], None
    for i in range(args.warmup + args.steps):
        info = time_cpu(m, w, target_s=max(1.0, min(10.0, 60.0 / max(1, args.steps + args.warmup))))
        if i >= args.warmup:
            vals.append(info)
    tot_s = sum(v["seconds"] for v in vals)
    tot_n = sum(v["samples"] for v in vals)
    value = tot_n / tot_s / 1e6
    cb = {k: info[k] for k in ("unit", "cores", "kind", "build", "builds", "sample")}
    cb["value"] = value
    cfg = workload_config(args, w, None, world)
    cfg["ran"] = "reference arm: " + info["sample"]  # what this arm actually executed (a bounded, per-sample-linear sample of the workload)
    line = {"impl": "reference", "metric": "demodulated Msamples/s (all channels)", "value": value, "unit": "Msamples/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / max(1, len(vals)),
            "higher_is_better": True, "scaling": w.scaling, "vs_baseline": None, "dtype": "q15/q31 fixed point (int16 data, int32 accumulate)",
            "data": "synthetic", "config": cfg, "cpu_baseline": cb,
            "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(args, w, C, world):
    nb = w.blocks
    cfg = {"workload": w.describe, "config": w.name, "blocks_per_channel_per_step": nb, "blocks_per_update": min(args.blocks_per_update or w.blocks_per_update, nb),
           "fs_hz": w.fs, "modes": "{AM,USB,LSB,CW}[c mod 4]",
           "fir": ("255-tap Kaiser designs from the sketch's designer + the zero arm_fir_init_q15 asks for (256): AM low-pass, SSB/CW band-pass with Q = reverse(I)"
                   if w.name == "c4" else "sketch tables: AM 102 taps (bw 2800 @ 24 kHz design, used as-is), SSB/CW 86 taps"),
           "biquads": "biquad1 low-pass (0.9*IF, Q 0.54) + biquad2 notch (fs/8, Q 15), integer Q2.30",
           "l2": "inputs and outputs of a step are GBs, far beyond the 126 MB L2; no explicit flush",
           "sharding": ("2^20 channels split into contiguous ranges over the GPUs (strong scaling)" if w.scaling == "strong"
                        else "independent channel shards of the same size per GPU (weak scaling)"),
           "layout": getattr(args, "layout", "updates")}
    if C is not None:
        cfg["channels_per_gpu"] = C
        cfg["channels_total"] = w.channels if w.scaling == "strong" else C * world
    if getattr(args, "with_frontend", False):
        cfg["with_frontend"] = ("raw 12-bit ADC codes through msdr_frontend_update_device (DC-block, amplifier, AGC) before every chain update; where the chain "
                                "leaves SMs free the front end of batch k+1 runs on them beside the chain of batch k (two streams), else the kernels alternate")
    return cfg


def parity_check(m, w, make_chain, C, ch0, dev_calls, n_updates=2):
    """Outside every timed region: a FRESH chain runs the first `n_updates` device-resident updates of the step (the benchmarked launch
    shape, state carried from the first into the second) and the sampled channels are compared bit for bit with the CPU checker fed the
    same input rows."""
    import torch
    import oracle_lib as ol
    lib = ol.CheckerLib("ref") if ol.have_ref() else ol.CheckerLib("orc")
    chans = m.workloads.sample_channels(C)
    g2 = make_chain()
    mism, n_samples = 0, 0
    modes = w.modes(C, ch0)
    o = cpu_chain(lib, w, [modes[c] for c in chans])
    idx = torch.tensor(chans, device="cuda")
    for (xin, yout, nb, stride) in dev_calls[:n_updates]:
        g2.update_device(xin.data_ptr(), yout.data_ptr(), nb, stride)
        g2.synchronize()
        torch.cuda.synchronize()
        xs = xin[idx, :nb * BLOCK].cpu().numpy()
        ys = yout[idx, :nb * BLOCK].cpu().numpy()
        want = o.run(np.ascontiguousarray(xs))[0]
        mism += int((want != ys).sum())
        n_samples += ys.size
    o.close()
    g2.close()
    return {"channels": len(chans), "updates": min(n_updates, len(dev_calls)), "blocks_per_update": int(dev_calls[0][2]), "samples": n_samples,
            "mismatches": mism, "checker": "oracle/_ref (reference sources)" if lib.prefix == "ref" else "oracle port"}


def output_sample(m, dev_calls, C, L):
    """The audio the timed path left in its output buffers (the last step, every update in stream order) for a fixed, seeded set of
    channels, gathered on the device right after the timed steps: (int16 [channels, samples] on the device, channel indices).
    It takes as many whole channels as fit in DUMP_BYTES as float32. If even the fixed edge channels of sample_channels do not fit,
    it keeps only their leading samples."""
    import torch
    chans = m.workloads.sample_channels(C, want=max(1, DUMP_BYTES // (4 * L)))
    cols = min(L, DUMP_BYTES // (4 * len(chans)))
    idx = torch.tensor(chans, device=dev_calls[0][1].device)
    y = torch.cat([yout[idx, :nb * BLOCK] for _, yout, nb, _ in dev_calls], dim=1)
    return y[:, :cols].clone(), chans


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c3", choices=["c3", "c4", "c5"])
    ap.add_argument("--channels", type=int, default=0, help="override the workload's channel count (per GPU for c3/c4, total for c5)")
    ap.add_argument("--blocks-per-update", type=int, default=0,
                    help="128-sample blocks per msdr_chain_update_device call (state is carried from call to call); default per workload: c3 1024 = 2.97 s of signal")
    ap.add_argument("--seconds", type=float, default=0.0, help="override the signal length of a step")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the sampled-channel comparison with the CPU checker after the timed regions")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to the NUMA node of its GPU")
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--with-frontend", action="store_true",
                    help="study: feed raw 12-bit ADC codes through the front-end conditioning kernel (DC-block, amplifier, AGC; SURVEY 8f rank 1) "
                         "in front of every chain update; the default line measures the north-star path only")
    ap.add_argument("--frontend-serial", action="store_true", help="with --with-frontend: front end and chain alternate on one stream (no overlap)")
    ap.add_argument("--layout", choices=["updates", "rows"], default="updates",
                    help="device-resident input layout: 'updates' = one contiguous [channels][samples] batch per update (how a streaming "
                         "receiver holds its block batches), 'rows' = one row per channel for the whole step, updates are column windows of it")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the audio the last timed step computed as DIR/audio.npy (float32 [channels, samples]: a fixed, "
                         "seeded sample of rank 0's channels, at most 64 MB) so that two builds can be compared output for output. Where a step "
                         "alternates two output batches over more updates (c5), every update gets its own output buffer instead, so that the "
                         "whole step survives: more device memory, and the JSON line's dump_outputs entry says how much")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import minimal_sdr_b200 as m

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    numa = None if args.no_numa else m.shard.bind_to_gpu_numa(local_rank)  # before any pinned allocation: first touch lands on the GPU's node
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # keep stdout to the single JSON line: NCCL writes its version banner / warnings to stdout unless told otherwise
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)

    K = m.load_ref_constants()
    w = m.workloads.get(args.config, K)
    if args.channels:
        w.channels = args.channels
    if args.seconds:
        w.seconds = args.seconds
    if w.scaling == "strong":
        shard = m.shard.plan(w.channels, world, rank)
    else:
        shard = m.shard.weak_scaling_shard(w.channels, world, rank)  # this rank's slice of the global channel space
    C, ch0 = shard.n, shard.ch0
    nb_total = w.blocks
    L = nb_total * BLOCK
    bpu = max(1, min(args.blocks_per_update or w.blocks_per_update, nb_total))

    def make_chain():
        c = m.ReceiveChain(C, device=local_rank, max_taps=w.max_taps)
        c.set_option("variant", args.variant)
        w.configure(c, ch0)
        return c

    g = make_chain()
    updates = [(b0, min(bpu, nb_total - b0)) for b0 in range(0, nb_total, bpu)]
    # distinct input batches: all of them, except for the streaming workload, where two alternate (what is timed does not depend on
    # the content; the parity check runs on the first two, which are consecutive in time)
    n_bufs = len(updates) if w.name != "c5" else min(2, len(updates))
    stream = torch.cuda.Stream(device=dev)  # a real (non-NULL) stream: kernels and timing events share it
    assert stream.cuda_stream != 0
    g.set_stream(stream.cuda_stream)
    if args.layout == "rows":
        x = m.synth.torch_batch(C, L, dev, w.fs, ch0=ch0)
        y = torch.empty_like(x)
        dev_calls = [(x[:, b0 * BLOCK:], y[:, b0 * BLOCK:], nb, x.stride(0)) for b0, nb in updates]
        dump_buffers = {"output_buffers": 1, "without_dump": 1, "extra_bytes": 0}
    else:  # one contiguous batch per update; same samples, same order of processing
        xs = [m.synth.torch_batch(C, nb * BLOCK, dev, w.fs, ch0=ch0, n0=b0 * BLOCK) for b0, nb in updates[:n_bufs]]
        n_out = len(updates) if args.dump_outputs else n_bufs  # the dump needs every update's audio of the last step
        ys = [torch.empty_like(xs[i % n_bufs]) for i in range(n_out)]
        dump_buffers = {"output_buffers": n_out, "without_dump": n_bufs, "extra_bytes": sum(t.nbytes for t in ys[n_bufs:])}
        dev_calls = [(xs[i % n_bufs], ys[i % n_out], nb, xs[i % n_bufs].stride(0)) for i, (b0, nb) in enumerate(updates)]
    calls = [(a.data_ptr(), b.data_ptr(), nb, st) for a, b, nb, st in dev_calls]
    torch.cuda.synchronize()

    fe = None
    fe_pipelined = False
    if args.with_frontend:
        fe = m.Frontend(C, device=local_rank)
        adc = [(a[:, :nb * BLOCK].to(torch.int32) // 16 + 2048).clamp_(0, 4095).to(torch.int16).contiguous() for a, b, nb, st in dev_calls]
        adc_calls = [(a.data_ptr(), a.stride(0)) for a in adc]
        fe_in = [torch.empty_like(a) for a in adc]  # conditioned IF samples, the chain's input in this mode
        calls = [(f.data_ptr(), c[1], c[2], f.stride(0)) for f, c in zip(fe_in, calls)]
        # Few channels leave SMs without a chain to pin (4096 channels = 128 groups on 148 SMs).  Then the chain kernel gives those SMs
        # up ("spare_sms"), the front end packs its channel groups onto them ("sms") and conditions block batch k + 1 on its own stream
        # while the chain works on batch k.  Otherwise (or with --frontend-serial) the two kernels alternate on one stream.
        n_sms = torch.cuda.get_device_properties(dev).multi_processor_count
        spare = n_sms - (C + 31) // 32
        fe_pipelined = spare >= 8 and not args.frontend_serial
        if fe_pipelined:
            stream_fe = torch.cuda.Stream(device=dev)
            fe.set_stream(stream_fe.cuda_stream)
            fe.set_option("sms", spare)
            g.set_option("spare_sms", spare)
            ev_fe = [torch.cuda.Event() for _ in calls]
            ev_chain = [torch.cuda.Event() for _ in calls]
        else:
            fe.set_stream(stream.cuda_stream)
        torch.cuda.synchronize()

    def step():
        for i, (d_in, d_out, nb, stride) in enumerate(calls):
            if fe is not None:  # raw codes -> conditioned IF samples
                if fe_pipelined:
                    stream_fe.wait_event(ev_chain[i])  # the chain has read this batch's previous contents (no-op before the first record)
                    fe.update_device(adc_calls[i][0], d_in, nb, stride)
                    ev_fe[i].record(stream_fe)
                    stream.wait_event(ev_fe[i])
                else:
                    fe.update_device(adc_calls[i][0], d_in, nb, stride)
            g.update_device(d_in, d_out, nb, stride)
            if fe_pipelined:
                ev_chain[i].record(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local_rank)
    clocks.start()
    step()  # first touch (plan upload, allocations) before the sampler's load window
    barrier()
    clocks.t_load0 = time.time()
    for _ in range(args.warmup):
        step()
    barrier()
    l0 = g.launch_count()
    fe_l0 = fe.launch_count() if fe is not None else 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.profiler.start()  # cudaProfilerStart: `ncu --profile-from-start off` sees exactly the timed region
    clocks.t0 = time.time()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    clocks.t1 = time.time()
    torch.cuda.profiler.stop()
    # before the cool-down steps and the parity check write the output buffers again
    dump = output_sample(m, dev_calls, C, L) if args.dump_outputs and rank == 0 else None
    ms_local = e0.elapsed_time(e1)
    launches = g.launch_count() - l0 + ((fe.launch_count() - fe_l0) if fe is not None else 0)
    if clocks.t1 - clocks.t0 < 0.5:  # untimed cool-down under the same load so that the clock sampler sees it
        t_end = time.time() + 0.5
        while time.time() < t_end:
            step()
            torch.cuda.synchronize()
    clk = clocks.stop()
    ms = m.shard.max_over_ranks(ms_local, dev)  # multi-GPU timing rule: slowest rank

    samples_per_step = C * L                                   # this rank
    total_per_step = m.shard.sum_over_ranks(samples_per_step, dev)  # all ranks (equal shards for weak scaling)
    value = total_per_step * args.steps / (ms * 1e-3) / 1e6    # Msamples/s, whole job
    kernel_name = g.last_kernel()

    # ---- parity at the benchmarked launch shape, outside the timed region
    parity = None
    if not args.no_parity and fe is None:
        parity = {"device_resident": parity_check(m, w, make_chain, C, ch0, dev_calls)}

    # ---- e2e: the user-facing call with HOST (pinned) buffers; H2D and D2H inside the timed region
    e2e = None
    if args.e2e_steps > 0:
        Le = L if w.name != "c5" else bpu * BLOCK  # streaming: one update of the stream per call
        hin = m.capi.PinnedBuffer((C, Le))
        hout = m.capi.PinnedBuffer((C, Le))
        if args.layout == "rows":
            hin.array[:] = x[:, :Le].cpu().numpy()
        else:
            col = 0
            for a, b, nb, st in dev_calls:
                if col >= Le:
                    break
                hin.array[:, col:col + nb * BLOCK] = a[:, :nb * BLOCK].cpu().numpy()
                col += nb * BLOCK
        g.update(hin.array, out=hout.array)  # warm-up (allocates staging)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            g.update(hin.array, out=hout.array)
        barrier()
        dt_local = time.perf_counter() - t0
        dt = m.shard.max_over_ranks(dt_local, dev)
        total_e2e = m.shard.sum_over_ranks(C * Le, dev)
        e2e = {"value": total_e2e * args.e2e_steps / dt / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": int(total_e2e * 2), "d2h_bytes_per_step": int(total_e2e * 2), "steps": args.e2e_steps,
               "api": "msdr_chain_update (C ABI, pinned host buffers, whole batch per call)", "samples_per_call_per_gpu": int(C * Le)}
        # attribution of the host path: plain pinned copies of the same buffers, every rank at the same time, no kernel
        th, to = torch.from_numpy(hin.array), torch.from_numpy(hout.array)
        nrow = max(1, min(C, (1 << 28) // (Le * 2)))  # leading rows, contiguous, <= 256 MB
        dbuf = torch.empty((nrow, Le), dtype=torch.int16, device=dev)
        pc = {}
        for name, fn in (("h2d", lambda: dbuf.copy_(th[:nrow], non_blocking=True)), ("d2h", lambda: to[:nrow].copy_(dbuf, non_blocking=True))):
            fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            pc[name + "_gbs"] = 3 * nrow * Le * 2 / (time.perf_counter() - t0) / 1e9
            barrier()
        # both directions at once on two streams (what the end-to-end path asks of the link): the roofline of `e2e`
        dbuf2 = torch.empty((nrow, Le), dtype=torch.int16, device=dev)
        s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

        def both():
            with torch.cuda.stream(s_up):
                dbuf.copy_(th[:nrow], non_blocking=True)
            with torch.cuda.stream(s_dn):
                to[:nrow].copy_(dbuf2, non_blocking=True)
        both()
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            both()
        torch.cuda.synchronize()
        pc["both_gbs_each_way"] = 3 * nrow * Le * 2 / (time.perf_counter() - t0) / 1e9
        barrier()
        del dbuf, dbuf2
        pc["e2e_gbs_each_way"] = C * Le * 2 * args.e2e_steps / dt_local / 1e9
        pc["e2e_over_link_both_ways"] = pc["e2e_gbs_each_way"] / pc["both_gbs_each_way"]
        pc["pinned"] = bool(th.is_pinned())
        e2e["pcie_this_rank"] = pc
        if parity is not None:  # the same call on a fresh chain, sampled channels against the CPU checker over the whole call
            import oracle_lib as ol
            lib = ol.CheckerLib("ref") if ol.have_ref() else ol.CheckerLib("orc")
            chans = m.workloads.sample_channels(C)
            g3 = make_chain()
            g3.update(hin.array, out=hout.array)
            g3.close()
            modes = w.modes(C, ch0)
            o = cpu_chain(lib, w, [modes[c] for c in chans])
            want = o.run(np.ascontiguousarray(hin.array[chans]))[0]
            o.close()
            parity["e2e"] = {"channels": len(chans), "blocks": int(Le // BLOCK), "samples": int(want.size),
                             "mismatches": int((want != hout.array[chans]).sum())}
        hin.free(); hout.free()

    # ---- per-rank records (rank 0 prints them all)
    mine = {"rank": rank, "gpu": local_rank, "channels": C, "ch0": ch0, "ms_per_step": ms_local / args.steps,
            "msamples_per_s": samples_per_step * args.steps / (ms_local * 1e-3) / 1e6, "clocks": clk, "numa": numa,
            "pcie": (e2e or {}).get("pcie_this_rank"), "parity": parity}
    per_rank = [mine]
    if world > 1:
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)

    if rank == 0:
        peak, peak_src = peaks()
        per_launch_s = (ms * 1e-3) / max(1, launches)
        samples_per_launch = samples_per_step * args.steps / max(1, launches)
        achieved = ALGO_BYTES_PER_SAMPLE * samples_per_launch / per_launch_s / 1e9
        for r in per_rank:
            r["hbm_frac"] = ALGO_BYTES_PER_SAMPLE * r["msamples_per_s"] * 1e6 / 1e9 / peak
        # second ceiling (SURVEY 8d asks for the issue-side fraction next to the HBM one): the biquad is an exact-arithmetic serial
        # recurrence per channel; a channel group of 32 advances one sample per stage step of its chain warp
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        groups = (C + 31) // 32
        f_hz = float((clk or {}).get("sm_mhz") or 1965.0) * 1e6
        per_gpu = value / world
        lat_ceiling = C * f_hz / LATENCY_BOUND_CYCLES / 1e6
        iss_ceiling = min(C, (groups if groups <= sms else min(groups, 2 * sms)) * 32) * f_hz / ISSUE_BOUND_CYCLES / 1e6
        recurrence = {"applies": groups <= 2 * sms,
                      "latency_bound": {"cycles_per_sample_step": LATENCY_BOUND_CYCLES, "ceiling": lat_ceiling, "frac": per_gpu / lat_ceiling,
                                        "what": "machine bound: loop-carried latency of one stage (IMAD.HI 9 + SHF 4 + I2IP 4), every channel's chain running alone"},
                      "issue_bound_one_warp": {"cycles_per_sample_step": ISSUE_BOUND_CYCLES, "ceiling": iss_ceiling, "frac": per_gpu / iss_ceiling,
                                               "what": "a whole stage in ONE warp, 43.5 cycles per sample (tools/microbench/bqstep2.cu): round 1's reference point, not a machine bound - the time-folded kernel splits a stage over a helper warp and a chain warp and exceeds it"},
                      "unit": "Msamples/s per GPU", "source": "profiles/r01_microbench_lat.txt; DESIGN.md section 6"}
        traffic, traffic_algo, traffic_src = ncu_traffic(w.name)
        line = {
            "metric": "demodulated Msamples/s (all channels)", "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": w.scaling, "vs_baseline": None,
            "dtype": "q15/q31 fixed point (int16 data, int32 wrapping accumulate, Q2.30 biquad)", "data": "synthetic",
            "config": workload_config(args, w, C, world), "gpu_launches": int(launches), "clocks": clk,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": traffic_src, "traffic_launch_algorithmic_bytes": traffic_algo,
                         "traffic_over_algorithmic": (traffic / traffic_algo if traffic and traffic_algo else None),
                         "algorithmic_bytes_per_launch": ALGO_BYTES_PER_SAMPLE * samples_per_launch,
                         "peak_source": peak_src, "kernel": kernel_name,
                         "algorithmic_bytes_per_sample": ALGO_BYTES_PER_SAMPLE, "samples_per_launch": samples_per_launch,
                         "avg_launch_ms": per_launch_s * 1e3, "recurrence": recurrence,
                         "note": "`traffic` is the ncu DRAM byte count of ONE captured launch and `traffic_launch_algorithmic_bytes` the algorithmic bytes of that same "
                                 "launch; `algorithmic_bytes_per_launch` is this run's average launch. The biquad is an exact-arithmetic serial recurrence per channel "
                                 "(DESIGN.md section 6): few channels are latency-bound (`recurrence`), many channels issue-bound; the FIR pair runs on the tensor cores"},
            "e2e": e2e, "parity_checked": parity, "per_rank": per_rank,
        }
        if w.stream_seconds:
            sig = L / w.fs
            line["stream"] = {"signal_seconds_per_step": sig, "stream_seconds": w.stream_seconds, "steps_for_stream": w.stream_seconds / sig,
                              "projected_wall_seconds_for_stream": (ms / args.steps) * 1e-3 * w.stream_seconds / sig,
                              "realtime_factor": sig / ((ms / args.steps) * 1e-3),
                              "note": "a step is a slice of the stream: updates of blocks_per_update blocks, state carried from update to update and step to step"}
        if world == 1 and not args.no_cpu:
            cb = time_cpu(m, w)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "build", "builds", "sample")}
        if dump is not None:
            audio, chans = dump
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "audio.npy"), audio.cpu().numpy().astype(np.float32))
            line["dump_outputs"] = {"dir": args.dump_outputs, "audio": list(audio.shape), "channels": len(chans),
                                    "what": "int16 audio of the last timed step as float32; channels of workloads.sample_channels, leading samples of each",
                                    "timed_path": dump_buffers}
        print(json.dumps(line), flush=True)
    g.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
