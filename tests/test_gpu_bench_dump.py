"""bench.py --dump-outputs on the GPU: audio.npy holds the last timed step, every update of it in stream order, and not the output of
a warm-up step, of the untimed cool-down steps or of the parity re-run that follow.  The CPU oracle is fed the same update sequence
with state carried; consecutive steps and the two halves of a step differ, so only the right step in the right buffers matches."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_is_the_last_timed_step(msdr, orc, K, tmp_path):
    import torch
    import bench
    C, warmup, steps = 200, 3, 2
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "c5", "--channels", str(C), "--warmup", str(warmup),
                        "--steps", str(steps), "--no-cpu", "--e2e-steps", "0", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["steps"] == steps and d["parity_checked"]["device_resident"]["mismatches"] == 0
    got = np.load(tmp_path / "audio.npy")

    w = msdr.workloads.get("c5", K)
    L, U = w.blocks * msdr.capi.BLOCK, w.blocks_per_update * msdr.capi.BLOCK
    assert L == 4 * U  # four updates per step over two alternating input batches: the case that needs one output buffer per update
    xs = [msdr.synth.torch_batch(C, U, torch.device("cuda", 0), w.fs, n0=k * U).cpu().numpy() for k in range(2)]
    chans = msdr.workloads.sample_channels(C, want=max(1, bench.DUMP_BYTES // (4 * L)))
    assert got.dtype == np.float32 and got.shape == (len(chans), L)
    x = np.ascontiguousarray(np.concatenate([xs[0], xs[1], xs[0], xs[1]], axis=1)[chans])
    modes = w.modes(C)
    o = bench.cpu_chain(orc, w, [modes[c] for c in chans])
    outs = [o.run(x)[0] for _ in range(1 + warmup + steps + 1)]  # first-touch step, warm-up, timed steps, one cool-down step
    o.close()
    want = outs[-2]
    assert not np.array_equal(want, outs[-3]) and not np.array_equal(want, outs[-1])
    assert not np.array_equal(want[:, :2 * U], want[:, 2 * U:])
    assert np.array_equal(got, want.astype(np.float32))
