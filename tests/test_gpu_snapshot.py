"""Snapshots of channel ranges (msdr_chain_snapshot* / msdr_chain_restore*): checkpoint, resume, migration and re-sharding.

Every resume case runs the same configuration uninterrupted on the GPU and compares byte for byte, on every channel (SYNCAM and ANR
channels too: same kernels, same device).  Channels without SYNCAM and ANR are also compared with the CPU oracle."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import frontend_lib as fl
import oracle_lib as ol
from chain_helpers import assert_same, configure_pair, run_pair
from conftest import adversarial_inputs, wrap_coeffs

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _st_bytes(st):
    st.fir_set = 0  # the slot id of a table is the chain's own business; everything else must be equal
    return bytes(st)


def _states_equal(a, b, ca, cb, what=""):
    assert _st_bytes(a.get_state(ca)) == _st_bytes(b.get_state(cb)), (what, ca, cb)
    assert a.fir_taps(ca) == b.fir_taps(cb), (what, ca, cb)


def _updates(chains, x, splits):
    """Feed x in updates of `splits` blocks to every chain; returns each chain's output."""
    outs = [[] for _ in chains]
    b0 = 0
    for s in splits:
        part = np.ascontiguousarray(x[:, 128 * b0:128 * (b0 + s)])
        for o, g in zip(outs, chains):
            o.append(g.update(part))
        b0 += s
    return [np.concatenate(o, axis=1) for o in outs]


# ---- 1. resume into a bare chain -----------------------------------------------------------------------------------------------
def _rich_config(msdr, K, C_, seed=3):
    rng = np.random.default_rng(seed)
    tables = []
    for k in range(32):  # 32 distinct tables, 4..102 taps, every fourth one wrapping
        T = 4 + 2 * ((k * 49) // 31)
        if k % 4 == 3:
            tables.append((wrap_coeffs(T, rng), wrap_coeffs(T, rng)))
        else:
            tables.append((rng.integers(-3000, 3000, T).astype(np.int16), rng.integers(-3000, 3000, T).astype(np.int16)))
    modes = [(ol.MODE_SYNCAM, ol.MODE_AM, ol.MODE_LSB, ol.MODE_USB, ol.MODE_CW)[c % 5] for c in range(C_)]

    def build():
        g = msdr.ReceiveChain(C_)
        for c in range(C_):
            g.set_mode(modes[c], c, 1)
            g.fir_init(*tables[(c * 7) % 32], c, 1)
        g.biquad_set_coefficients(0, 0, K["biquad1_lowpass_coef"])
        g.biquad_set_coefficients(1, 0, K["biquad2_notch_coef"])
        for stage in (1, 2, 3):  # 4-stage cascades on some channels
            g.biquad_set_coefficients(0, stage, K["biquad1_lowpass_coef"], 40, 70)
            g.biquad_set_coefficients(1, stage, K["biquad2_notch_coef"], 200, 64)
        g.set_anr(1, 3, 20)
        g.set_anr(2, 150, 33)
        g.set_anr(2, C_ - 5, 5)
        return g
    return build


def test_resume_into_bare_chain(msdr, K):
    C_ = 300  # a partial last group
    build = _rich_config(msdr, K, C_)
    rng = np.random.default_rng(11)
    x = rng.integers(-32768, 32768, (C_, 128 * 14), dtype=np.int16)
    adv = adversarial_inputs(x.shape[1], rng)
    for i, v in enumerate(adv.values()):  # extreme inputs on some rows
        x[5 + 37 * i] = v
    u, g = build(), build()
    ya_u, = _updates([u], x[:, :128 * 6], [1, 3, 2])
    ya_g, = _updates([g], x[:, :128 * 6], [2, 1, 3])
    assert_same(ya_g, ya_u, "before the snapshot")
    blob = g.snapshot()
    assert blob.size == g.snapshot_bytes()
    info = msdr.capi.snapshot_info(blob)
    assert info["n_channels"] == C_ and info["max_taps_needed"] == 102 and info["flags"] == msdr.capi.SNAPSHOT_ANR
    r = msdr.ReceiveChain(C_)  # no setter called
    r.restore(blob)
    for c in range(C_):
        _states_equal(r, g, c, c, "restored")
        assert r.fir_taps(c) == g.fir_taps(c)
    for c in (3, 10, 22, 150, 182, C_ - 1):
        assert bytes(r.get_anr_state(c)) == bytes(g.get_anr_state(c)), c
    yb_u, yb_r, yb_g = _updates([u, r, g], x[:, 128 * 6:], [3, 1, 4])
    assert_same(yb_r, yb_u, "restored chain after the snapshot")
    assert_same(yb_g, yb_u, "source after the snapshot")
    for c in range(0, C_, 13):
        _states_equal(r, u, c, c, "after")


# ---- 2. re-sharding -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("granule", [32, 1])
def test_reshard_3_2_3(msdr, orc, K, granule):
    N = 1000
    wl = msdr.workloads.get("c3", K)
    modes = wl.modes(N)
    u, o = configure_pair(msdr, orc, K, modes)
    x = msdr.synth.batch(modes, 128 * 9)
    yu, yo = run_pair(u, o, x, [3, 3, 3])
    assert_same(yu, yo, "uninterrupted vs oracle")

    def chains(world):
        out = []
        for s in msdr.shard.plan(N, world, granule=granule):
            g = msdr.ReceiveChain(s.n)
            out.append((s, g))
        return out

    def run(shards, b0, nb):
        return np.concatenate([g.update(np.ascontiguousarray(x[s.ch0:s.ch0 + s.n, 128 * b0:128 * (b0 + nb)])) for s, g in shards], axis=0)

    def move(shards, new_world):
        blobs = [g.snapshot() for _, g in shards]
        new = chains(new_world)
        pieces = msdr.shard.reshard(N, len(shards), new_world, granule=granule)
        assert sum(p.n for p in pieces) == N
        if granule == 1:
            assert any(p.first % 32 for p in pieces) and any(p.dst_ch0 % 32 for p in pieces)
        for p in pieces:
            new[p.new_rank][1].restore(blobs[p.old_rank], ch0=p.dst_ch0, first=p.first, n=p.n)
        return new

    three = chains(3)
    for s, g in three:
        wl.configure(g, s.ch0)
    y = [run(three, 0, 3)]
    two = move(three, 2)
    y.append(run(two, 3, 3))
    three = move(two, 3)
    y.append(run(three, 6, 3))
    assert_same(np.concatenate(y, axis=1), yu, "3 -> 2 -> 3 ranks vs uninterrupted")
    assert_same(np.concatenate(y, axis=1), yo, "3 -> 2 -> 3 ranks vs oracle")


# ---- 3. different max_taps ------------------------------------------------------------------------------------------------------
def test_restore_other_max_taps(msdr, orc, K):
    C_ = 200
    modes = msdr.synth.mixed_modes(C_)
    u, o = configure_pair(msdr, orc, K, modes)
    g, _ = configure_pair(msdr, orc, K, modes)
    x = msdr.synth.batch(modes, 128 * 8)
    yu, yo = run_pair(u, o, x, [3, 5])
    _updates([g], x[:, :128 * 3], [1, 2])
    blob = g.snapshot()
    big = msdr.ReceiveChain(C_, max_taps=256)
    big.restore(blob)
    yb, = _updates([big], x[:, 128 * 3:], [2, 3])
    assert_same(yb, yu[:, 128 * 3:], "max_taps 256 after restore vs uninterrupted")
    assert_same(yb, yo[:, 128 * 3:], "max_taps 256 after restore vs oracle")
    for c in range(0, C_, 17):
        _states_equal(big, u, c, c, "256")

    # an 86-tap chain cannot take the 102-tap AM table: refused, and the chain is exactly its untouched twin
    ssb = (np.array(K["FIR_SSB_I_coeffs"], np.int16), np.array(K["FIR_SSB_Q_coeffs"], np.int16))
    small, twin = msdr.ReceiveChain(C_, max_taps=86), msdr.ReceiveChain(C_, max_taps=86)
    for t in (small, twin):
        t.set_mode(ol.MODE_USB)
        t.fir_init(*ssb)
        t.biquad_set_coefficients(0, 0, K["biquad1_lowpass_coef"])
    _updates([small, twin], x[:, :128], [1])
    with pytest.raises(msdr.MsdrError) as e:
        small.restore(blob)
    assert e.value.status == msdr.capi.ERR_ARGUMENT
    ys, yt = _updates([small, twin], x[:, 128:128 * 4], [3])
    assert_same(ys, yt, "refused restore")
    assert small.plan_build_count() == twin.plan_build_count()
    for c in range(0, C_, 9):
        _states_equal(small, twin, c, c, "refused")


# ---- 4. refusals leave the chain unchanged ---------------------------------------------------------------------------------------
def _poke(blob, off, value, dtype):
    b = blob.copy()
    b[off:off + np.dtype(dtype).itemsize] = np.array([value], dtype).view(np.uint8)
    return b


def test_refusals_leave_chain_unchanged(msdr, K):
    C_ = 64
    rng = np.random.default_rng(4)
    tabs = [(rng.integers(-2000, 2000, 20).astype(np.int16), rng.integers(-2000, 2000, 20).astype(np.int16)) for _ in range(33)]

    def target():
        t = msdr.ReceiveChain(C_)
        for c in range(C_):  # 32 live tables, two users each
            t.fir_init(*tabs[c % 32], c, 1)
        t.set_mode(ol.MODE_USB, 10, 20)
        t.biquad_set_coefficients(0, 0, K["biquad1_lowpass_coef"])
        t.enable_frontend(0.25, 40.0, True)
        return t
    t, w = target(), target()
    x = rng.integers(-20000, 20000, (C_, 128 * 6), dtype=np.int16)
    _updates([t, w], x[:, :128 * 2], [2])

    src = msdr.ReceiveChain(8)
    src.fir_init(*tabs[32])  # a 33rd table
    src.enable_frontend(0.25, 40.0, True)
    good = src.snapshot()
    q31 = msdr.ReceiveChain(8, am_q31=True)
    q31.fir_init(*tabs[0])
    agc = msdr.ReceiveChain(8)
    agc.fir_init(*tabs[0])
    agc.enable_frontend(0.5, 40.0, True)
    E = msdr.capi
    cases = {
        "33rd table": (good, 40, 0, 1, E.ERR_NOMEM),
        "am_q31": (q31.snapshot(), 0, 0, 8, E.ERR_ARGUMENT),
        "agc parameters": (agc.snapshot(), 0, 0, 8, E.ERR_ARGUMENT),
        "bad magic": (_poke(good, 0, ord("X"), np.uint8), 0, 0, 8, E.ERR_ARGUMENT),
        "version": (_poke(good, 8, 2, np.uint32), 0, 0, 8, E.ERR_UNSUPPORTED),
        "truncated": (good[:-1], 0, 0, 8, E.ERR_ARGUMENT),
        "truncated header": (good[:100], 0, 0, 1, E.ERR_ARGUMENT),
        "offset past the end": (_poke(good, 64 + 8 * 2, 1 << 40, np.uint64), 0, 0, 8, E.ERR_ARGUMENT),
        "first + n past the snapshot": (good, 0, 4, 5, E.ERR_ARGUMENT),
        "ch0 + n past the chain": (good, 60, 0, 8, E.ERR_ARGUMENT),
    }
    for name, (blob, ch0, first, n, want) in cases.items():
        with pytest.raises(msdr.MsdrError) as e:
            t.restore(blob, ch0=ch0, first=first, n=n)
        assert e.value.status == want, name
    for g in (t, w):
        g.synchronize()
    yt, yw = _updates([t, w], x[:, 128 * 2:], [1, 3])
    assert_same(yt, yw, "after refused restores")
    assert t.plan_build_count() == w.plan_build_count()
    for c in range(C_):
        _states_equal(t, w, c, c, "refused")
        assert bytes(t.get_frontend_state(c)) == bytes(w.get_frontend_state(c))


# ---- 5. front end --------------------------------------------------------------------------------------------------------------
def _v5min():
    import torch
    return min(12288, 64 * torch.cuda.get_device_properties(0).multi_processor_count + 1)


@pytest.mark.parametrize("where", ["fused", "composed"])
def test_frontend_resume(msdr, orc, K, where):
    forc = fl.Orc()
    C_ = _v5min() if where == "fused" else 300
    wl = msdr.workloads.get("c3", K)
    codes = fl.adc_stream(C_, 128 * 10, seed=31)
    xi = np.random.default_rng(32).integers(-20000, 20000, (C_, 128 * 2), dtype=np.int16)

    def build():
        g = msdr.ReceiveChain(C_, max_taps=102)
        wl.configure(g)
        g.enable_frontend()
        g.frontend_preset(2048, 7, 30)
        return g
    u, g = build(), build()
    split = lambda a, b: np.ascontiguousarray(codes[:, 128 * a:128 * b])  # noqa: E731
    yu = [u.update_adc(split(0, 4))]
    g.update_adc(split(0, 1))
    g.update_adc(split(1, 4))
    assert (("fused into the converters" in g.last_kernel()) == (where == "fused")), g.last_kernel()
    blob = g.snapshot()
    assert msdr.capi.snapshot_info(blob)["flags"] == msdr.capi.SNAPSHOT_FRONTEND
    r = msdr.ReceiveChain(C_, max_taps=102)  # no front end: the snapshot brings it
    r.restore(blob)
    yr = []
    for step in ("adc", "int16", "adc"):  # int16 and ADC updates interleave after the restore
        if step == "int16":
            yu.append(u.update(xi)); yr.append(r.update(xi))
        else:
            a = 4 if not yr else 7
            yu.append(u.update_adc(split(a, a + 3))); yr.append(r.update_adc(split(a, a + 3)))
    assert_same(np.concatenate(yr, axis=1), np.concatenate(yu[1:], axis=1), "restored vs uninterrupted")
    for c in msdr.workloads.sample_channels(C_):
        assert bytes(r.get_frontend_state(c)) == bytes(u.get_frontend_state(c)), c
    # the oracles: front end then chain, on sampled channels
    chans = msdr.workloads.sample_channels(C_)
    modes = wl.modes(C_)
    o = orc.chain(len(chans))
    for i, c in enumerate(chans):
        o.set_mode(i, 1, modes[c])
        assert o.fir_init(i, 1, *wl.tables_for(modes[c])) == 0
    o.biquad_set_coefficients(0, 0, len(chans), 0, wl.biquad1)
    o.biquad_set_coefficients(1, 0, len(chans), 0, wl.biquad2)
    fo = forc.frontend(len(chans))
    for i, c in enumerate(chans):
        if 7 <= c < 37:
            fo.preset(i, 2048)
    sub = lambda a, b: np.ascontiguousarray(codes[chans, 128 * a:128 * b])  # noqa: E731
    ref = [o.run(fo.run(sub(0, 4)))[0], o.run(fo.run(sub(4, 7)))[0], o.run(np.ascontiguousarray(xi[chans]))[0], o.run(fo.run(sub(7, 10)))[0]]
    assert_same(np.concatenate(yu, axis=1)[chans], np.concatenate(ref, axis=1), "uninterrupted vs oracles")


# ---- 6. device buffers and streams -------------------------------------------------------------------------------------------------
def test_device_snapshot_on_torch_stream(msdr, K):
    import torch
    C_, nb = 4096, 4
    wl = msdr.workloads.get("c3", K)
    x = msdr.synth.torch_batch(C_, 128 * nb * 3, "cuda")
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    chains = []
    for _ in range(3):
        g = msdr.ReceiveChain(C_)
        wl.configure(g)
        g.set_mode(ol.MODE_SYNCAM, 100, 50)  # side-lane channels in the range
        g.set_anr(2, 300, 40)
        g.set_stream(s.cuda_stream)
        chains.append(g)
    g, r, u = chains
    y = {k: torch.empty((C_, 128 * nb * 3), dtype=torch.int16, device="cuda") for k in "gru"}
    st = x.stride(0)
    buf = torch.empty(g.snapshot_bytes(), dtype=torch.uint8, device="cuda")
    part = lambda t, i: t[:, 128 * nb * i:].data_ptr()  # noqa: E731
    with torch.cuda.stream(s):
        u.update_device(part(x, 0), part(y["u"], 0), nb, st)
        g.update_device(part(x, 0), part(y["g"], 0), nb, st)
        g.snapshot_device(0, C_, buf)  # no synchronise in between: stream order
        r.restore_device(buf, 0, 0, C_)
        for i in (1, 2):
            for k, c in (("u", u), ("g", g), ("r", r)):
                c.update_device(part(x, i), part(y[k], i), nb, st)
    s.synchronize()
    tail = slice(128 * nb, None)
    assert torch.equal(y["r"][:, tail], y["u"][:, tail]), "restore_device vs uninterrupted"
    assert torch.equal(y["g"], y["u"])
    host = np.empty(g.snapshot_bytes(), np.uint8)
    g2 = msdr.ReceiveChain(C_)
    g2.restore_device(buf)
    g2.synchronize()
    assert np.array_equal(g2.snapshot(out=host), buf.cpu().numpy()), "host snapshot of the restored chain == the device snapshot"
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU: the move to device 1 is not covered")
    b1 = buf.to("cuda:1")
    x1 = x.to("cuda:1")
    y1 = torch.empty_like(x1)
    torch.cuda.synchronize(1)
    r1 = msdr.ReceiveChain(C_, device=1)
    r1.restore_device(b1)
    for i in (1, 2):
        r1.update_device(part(x1, i), part(y1, i), nb, st)
    r1.synchronize()
    assert torch.equal(y1[:, tail].cpu(), y["u"][:, tail].cpu()), "restored on device 1"


# ---- 7. plans -----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C_", [2000, 12288])
def test_restore_builds_one_plan(msdr, K, C_):
    import torch
    wl = msdr.workloads.get("c3", K)
    g, r = msdr.ReceiveChain(C_), msdr.ReceiveChain(C_)
    wl.configure(g)
    r.set_mode(ol.MODE_CW)
    r.init_FIR(ol.MODE_CW)
    x = msdr.synth.torch_batch(C_, 128 * 2, "cuda")
    y = torch.empty_like(x)
    torch.cuda.synchronize()
    for c in (g, r):
        c.update_device(x.data_ptr(), y.data_ptr(), 2, x.stride(0))
        c.synchronize()
    blob = g.snapshot()
    n0 = r.plan_build_count()
    r.restore(blob)
    assert r.plan_build_count() == n0
    r.update_device(x.data_ptr(), y.data_ptr(), 2, x.stride(0))
    r.synchronize()
    assert r.plan_build_count() - n0 <= 1
    n1 = r.plan_build_count()
    r.update_device(x.data_ptr(), y.data_ptr(), 2, x.stride(0))
    r.restore(blob, ch0=100, first=100, n=900)  # a piece: still one configuration change
    r.update_device(x.data_ptr(), y.data_ptr(), 2, x.stride(0))
    r.synchronize()
    assert r.plan_build_count() - n1 <= 1


# ---- 8. size --------------------------------------------------------------------------------------------------------------------
def test_c5_snapshot_restore(msdr, K):
    import torch
    wl = msdr.workloads.get("c5", K)
    C_, nb = wl.channels, wl.blocks_per_update
    g, u = msdr.ReceiveChain(C_, max_taps=wl.max_taps), msdr.ReceiveChain(C_, max_taps=wl.max_taps)
    for c in (g, u):
        wl.configure(c)
    x = msdr.synth.torch_batch(C_, 128 * nb, "cuda")
    x2 = msdr.synth.torch_batch(C_, 128 * nb, "cuda", n0=128 * nb)
    yu, yr = torch.empty_like(x), torch.empty_like(x)
    torch.cuda.synchronize()  # the chains run on their own streams, which are not ordered with torch's
    st = x.stride(0)
    for c in (g, u):
        c.update_device(x.data_ptr(), yu.data_ptr(), nb, st)
        c.synchronize()
    pin = msdr.capi.PinnedBuffer((g.snapshot_bytes(),), np.uint8)
    blob = g.snapshot(out=pin.array)
    del g
    r = msdr.ReceiveChain(C_, max_taps=wl.max_taps)
    r.restore(blob)
    u.update_device(x2.data_ptr(), yu.data_ptr(), nb, st)
    r.update_device(x2.data_ptr(), yr.data_ptr(), nb, st)
    u.synchronize()
    r.synchronize()
    chans = msdr.workloads.sample_channels(C_)
    assert torch.equal(yr[chans], yu[chans])
    assert torch.equal(yr, yu)
    pin.free()


# ---- 10. façade --------------------------------------------------------------------------------------------------------------------
def test_checkpoint_receiver_program(msdr, K):
    host = os.path.join(ROOT, "minimal-sdr_b200", "host")
    subprocess.run(["make", "-s", "-C", host, "checkpoint_receiver"], check=True)
    C_, NB = 40, 9
    am = np.array(K["FIR_AM_coeffs_bw2800_fs24000"], np.int16)
    x = np.random.default_rng(9).integers(-20000, 20000, (C_, 128 * NB), dtype=np.int16)
    outs = {}
    with tempfile.TemporaryDirectory() as td:
        p = {n: os.path.join(td, n) for n in ("tables.bin", "in.bin", "ck.bin")}
        np.concatenate([am, am]).tofile(p["tables.bin"])
        x.tofile(p["in.bin"])
        for stop in (0, 4):
            out = os.path.join(td, f"out{stop}.bin")
            r = subprocess.run([os.path.join(host, "checkpoint_receiver"), str(C_), str(NB), str(stop), str(am.size), p["tables.bin"], p["in.bin"],
                                p["ck.bin"], out], capture_output=True, text=True, timeout=300)
            assert r.returncode == 0, r.stdout + r.stderr
            outs[stop] = np.fromfile(out, np.int16).reshape(C_, -1)
        assert os.path.getsize(p["ck.bin"]) > 0
    assert_same(outs[4], outs[0], "checkpointed vs uninterrupted Receiver")
    # and the same configuration on the Python chain
    d = msdr.design
    g = msdr.ReceiveChain(C_)
    g.biquad_set_coefficients(0, 0, d.biquad_lowpass(3000.0, 0.7071))
    g.biquad_set_coefficients(1, 0, d.biquad_notch(5514.7, 15.0))
    g.fir_init(am, am)
    for c in range(C_):
        g.set_mode((ol.MODE_AM, ol.MODE_USB, ol.MODE_LSB, ol.MODE_CW)[c % 4], c, 1)
    for c in range(0, C_, 8):
        g.set_anr(2, c, 1)
    assert_same(g.update(x), outs[0], "Receiver vs ReceiveChain")
