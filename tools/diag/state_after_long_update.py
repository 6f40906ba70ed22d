"""Diagnostic: is the carried state right after a LONG update?  For several first-update lengths and kernel shapes: update nb1
blocks on a fresh chain, then 8 more; sampled channels against the CPU checker for both updates; FIR history against the input tail."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np, torch
import minimal_sdr_b200 as m
import oracle_lib as ol

K = m.load_ref_constants()
w = m.workloads.get("c3", K)
C = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
dev = torch.device("cuda:0")
lib = ol.CheckerLib("ref") if ol.have_ref() else ol.CheckerLib("orc")
chans = m.workloads.sample_channels(C, want=24)
idx = torch.tensor(chans, device=dev)
modes = w.modes(C)
for variant in (0, 2048, 256):
    for nb1 in (64, 128, 256, 384, 512, 1024):
        g = m.ReceiveChain(C, max_taps=w.max_taps)
        g.set_option("variant", variant)
        g.set_stream(torch.cuda.current_stream().cuda_stream)  # torch's default stream: ordered with the generator kernels below
        w.configure(g)
        o = lib.chain(len(chans))
        for i, c in enumerate(chans):
            o.set_mode(i, 1, modes[c]); o.fir_init(i, 1, *w.tables_for(modes[c]))
        o.biquad_set_coefficients(0, 0, len(chans), 0, w.biquad1); o.biquad_set_coefficients(1, 0, len(chans), 0, w.biquad2)
        res = []
        n0 = 0
        for nb in (nb1, 8):
            x = m.synth.torch_batch(C, nb * 128, dev, w.fs, n0=n0)
            y = torch.empty_like(x)
            g.update_device(x.data_ptr(), y.data_ptr(), nb, x.stride(0))
            g.synchronize(); torch.cuda.synchronize()
            xs, ys = x[idx].cpu().numpy(), y[idx].cpu().numpy()
            want = o.run(np.ascontiguousarray(xs))[0]
            bad = np.argwhere(want != ys)
            res.append((len(bad), (int(bad[0][0]), int(bad[0][1])) if len(bad) else None))
            if nb == nb1:
                st = g.get_state(chans[1])
                T = st.num_taps
                hist_ok = list(st.fir_history[:T - 1]) == list(xs[1, -(T - 1):])
            n0 += nb * 128
        print(f"variant {variant:5d} nb1 {nb1:5d}: update1 mismatches {res[0]}, update2 mismatches {res[1]}, hist ok {hist_ok}", flush=True)
        g.close(); o.close()
