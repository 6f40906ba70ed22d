"""Receive chain from raw ADC codes (msdr_chain_update_adc*): the front end fused into the converters of the row-block kernel
(csrc/msdr_chain_v5.cu, both forms), or the front-end kernel followed by the int16 path.  Every comparison is byte for byte
against the CPU oracles run one after the other: the front end (frontend_lib.Orc) feeding the chain (oracle_lib)."""
import ctypes as C

import numpy as np
import pytest

import frontend_lib as fl
import oracle_lib as ol
from chain_helpers import assert_same, configure_pair

pytestmark = pytest.mark.gpu

FUSED = "front end fused into the converters"
COMPOSED = "msdr::fe::frontend_kernel"


@pytest.fixture(scope="module")
def forc():
    return fl.Orc()


def _fe_state_equal(gs, os_, what=""):
    assert (gs.hpf_x1, gs.hpf_y1, gs.multiplier, gs.agc_idx) == (os_["hpf_x1"], os_["hpf_y1"], os_["multiplier"], os_["agc_idx"]), what
    assert np.float32(gs.agc_val).view(np.uint32) == os_["agc_val"].view(np.uint32), what
    assert np.array_equal(np.array(gs.agc_buffer[:], np.int16), os_["agc_buffer"]), what


def _chain_state_equal(orc, g, o, c, x_if, what=""):
    """FIR history = the last taps - 1 conditioned IF samples; biquad words = the oracle's AudioFilterBiquad::definition."""
    st = g.get_state(c)
    n = st.num_taps - 1
    assert list(st.fir_history[:n]) == list(x_if[c, -n:]), (what, c)
    d = np.zeros(32, np.int32)
    for obj in (0, 1):
        orc.lib.orc_chain_get_biquad_definition(C.c_void_p(o.h), c, obj, d.ctypes.data_as(C.c_void_p))
        assert list(st.biquad_definition[obj]) == list(d), (what, c, obj)


def _run(g, o, fo, codes, splits):
    """ADC codes [C, n] in updates of `splits` blocks through the GPU chain and through oracle front end + oracle chain."""
    yg, yo, xo, b0 = [], [], [], 0
    for s in splits:
        part = np.ascontiguousarray(codes[:, 128 * b0:128 * (b0 + s)])
        yg.append(g.update_adc(part))
        x = fo.run(part)
        xo.append(x)
        yo.append(o.run(x)[0])
        b0 += s
    return np.concatenate(yg, axis=1), np.concatenate(yo, axis=1), np.concatenate(xo, axis=1)


def _long_window_pair(msdr, orc, C_, tables):
    """Every channel AM on one 256-tap table pair (the window only the half-tile row-block form takes)."""
    K = msdr.load_ref_constants()
    g = msdr.ReceiveChain(C_, max_taps=256)
    o = orc.chain(C_)
    cI, cQ = tables
    g.set_mode(ol.MODE_AM)
    o.set_mode(0, C_, ol.MODE_AM)
    g.fir_init(cI, cQ)
    assert o.fir_init(0, C_, cI, cQ) == 0
    for obj, key in ((0, "biquad1_lowpass_coef"), (1, "biquad2_notch_coef")):
        g.biquad_set_coefficients(obj, 0, K[key])
        o.biquad_set_coefficients(obj, 0, C_, 0, K[key])
    return g, o


@pytest.mark.parametrize("agc_on", [True, False])
def test_fused_ragged_updates(msdr, orc, forc, K, agc_on):
    """300 channels (a partial row block), mixed modes, presets on some channels, ragged updates; output and every state."""
    modes = msdr.synth.mixed_modes(300)
    codes = fl.adc_stream(300, 128 * 63, seed=21)
    g, o = configure_pair(msdr, orc, K, modes)
    g.set_option("variant", 4096)
    g.enable_frontend(agc_on=agc_on)
    fo = forc.frontend(300, on=int(agc_on))
    for ch0, nch, first in ((5, 16, 2048), (290, 10, 1000)):
        g.frontend_preset(first, ch0, nch)
        for c in range(ch0, ch0 + nch):
            fo.preset(c, first)
    yg, yo, xo = _run(g, o, fo, codes, [1, 2, 30, 3, 27])
    assert FUSED in g.last_kernel(), g.last_kernel()
    assert_same(yg, yo, "fused, ragged")
    for c in (0, 5, 20, 31, 127, 128, 255, 256, 290, 299):
        _fe_state_equal(g.get_frontend_state(c), fo.state(c), c)
        _chain_state_equal(orc, g, o, c, xo, "fused")
    if agc_on:
        assert len({g.get_frontend_state(c).multiplier for c in range(0, 300, 7)}) > 5  # the AGC moved the gains apart


@pytest.mark.parametrize("form", ["taps256", "half_tile_short_window"])
def test_fused_window_forms(msdr, orc, forc, K, form):
    """The half-tile kernel: the 256-tap window with 1-block updates (L < H: the history moves down), and variant bit 15 with the
    sketch's short window."""
    C_ = 160
    codes = fl.adc_stream(C_, 128 * 12, seed=22)
    if form == "taps256":
        g, o = _long_window_pair(msdr, orc, C_, msdr.workloads.c4_tables()[ol.MODE_AM])
        g.set_option("variant", 4096)
        splits = [1] * 6 + [2, 1, 3]
    else:
        g, o = configure_pair(msdr, orc, K, msdr.synth.mixed_modes(C_))
        g.set_option("variant", 4096 | 32768)
        splits = [1, 3, 2, 6]
    g.enable_frontend()
    fo = forc.frontend(C_)
    yg, yo, xo = _run(g, o, fo, codes, splits)
    assert "v5l::" in g.last_kernel() and FUSED in g.last_kernel(), g.last_kernel()
    assert_same(yg, yo, form)
    for c in (0, 31, 127, 128, 159):
        _fe_state_equal(g.get_frontend_state(c), fo.state(c), c)
        _chain_state_equal(orc, g, o, c, xo, form)


def test_fused_extreme_codes(msdr, orc, forc, K):
    """Full 16-bit codes (the DC-block accumulator wraps), both rails, constant input, and a start gain next to agc_max."""
    C_, n = 136, 128 * 10
    rng = np.random.default_rng(23)
    codes = rng.integers(0, 65536, (C_, n), dtype=np.uint16)
    codes[8:16] = 65535
    codes[16:24] = 0
    codes[24:32] = 3000
    codes[32:40, ::2] = 65535
    codes[32:40, 1::2] = 0
    modes = msdr.synth.mixed_modes(C_)
    for start, mx in ((0.25, 40.0), (39.9, 40.0), (2000.0, 40000.0)):
        g, o = configure_pair(msdr, orc, K, modes)
        g.set_option("variant", 4096)
        g.enable_frontend(agc_start=start, agc_max=mx)
        fo = forc.frontend(C_, start=start, mx=mx)
        yg, yo, _ = _run(g, o, fo, codes, [3, 1, 6])
        assert FUSED in g.last_kernel()
        assert_same(yg, yo, f"extreme codes, agc_start {start}")
        for c in (0, 8, 16, 24, 32, 135):
            _fe_state_equal(g.get_frontend_state(c), fo.state(c), (start, c))


def _torch_codes(torch, C_, n, seed_ch0=0):
    """12-bit codes generated on the device: (x >> 4) + 2048 of the seeded multi-tone int16 batch."""
    import minimal_sdr_b200 as m
    x = m.synth.torch_batch(C_, n, "cuda", ch0=seed_ch0).to(torch.int32)
    return ((x >> 4) + 2048).to(torch.int16)  # 0..4095: the same bits as uint16


def test_default_dispatch_many_channels(msdr, orc, forc, K):
    """At the row-block channel count the default dispatch fuses; the result equals the two GPU objects run one after the other and
    the oracle."""
    C_, nb = 9600, 4
    modes = msdr.synth.mixed_modes(C_)
    codes = fl.adc_stream(C_, 128 * nb * 2, seed=24)
    g, o = configure_pair(msdr, orc, K, modes)
    g.enable_frontend()
    g2, _ = configure_pair(msdr, orc, K, modes)
    fe = msdr.Frontend(C_)
    fo = forc.frontend(C_)
    for u in range(2):
        part = np.ascontiguousarray(codes[:, 128 * nb * u:128 * nb * (u + 1)])
        y = g.update_adc(part)
        assert FUSED in g.last_kernel() and "v5::" in g.last_kernel(), g.last_kernel()
        y2 = g2.update(fe.update(part))
        assert_same(y, y2, "fused vs front-end object + chain")
        assert_same(y, o.run(fo.run(part))[0], "fused vs oracle")


def test_composed_paths(msdr, orc, forc, K):
    """Few channels (the group-block kernels) and a range with side-lane channels (SYNCAM PLL, LMS): the front-end kernel, then the
    int16 path.  Equal to the two GPU objects run one after the other; channels off the side lane also equal the oracle."""
    # few channels
    modes = msdr.synth.mixed_modes(40)
    codes = fl.adc_stream(40, 128 * 9, seed=25)
    g, o = configure_pair(msdr, orc, K, modes)
    g.enable_frontend()
    fo = forc.frontend(40)
    yg, yo, _ = _run(g, o, fo, codes, [2, 7])
    assert g.last_kernel().startswith(COMPOSED), g.last_kernel()
    assert_same(yg, yo, "composed, few channels")
    # side-lane channels in a range that would otherwise fuse
    C_ = 300
    modes = msdr.synth.mixed_modes(C_)
    codes = fl.adc_stream(C_, 128 * 6, seed=26)
    side = [3, 77, 200]
    outs = []
    for obj in ("chain", "objects"):
        g, o = configure_pair(msdr, orc, K, modes)
        g.set_option("variant", 4096)
        g.set_mode(ol.MODE_SYNCAM, 3, 1)
        g.set_anr(1, 77, 1)
        g.set_anr(2, 200, 1)
        if obj == "chain":
            g.enable_frontend()
            outs.append([g.update_adc(np.ascontiguousarray(codes[:, :128 * 2])), g.update_adc(np.ascontiguousarray(codes[:, 128 * 2:]))])
            assert g.last_kernel().startswith(COMPOSED) and "v5::" in g.last_kernel(), g.last_kernel()
        else:
            fe = msdr.Frontend(C_)
            outs.append([g.update(fe.update(np.ascontiguousarray(codes[:, :128 * 2]))), g.update(fe.update(np.ascontiguousarray(codes[:, 128 * 2:])))])
    for a, b in zip(*outs):
        assert_same(a, b, "composed with side-lane channels vs objects")
    fo = forc.frontend(C_)
    yo = o.run(fo.run(codes))[0]
    keep = [c for c in range(C_) if c not in side]
    assert_same(np.concatenate(outs[0], axis=1)[keep], yo[keep], "composed, off the side lane, vs oracle")


def test_interleaving_migration_and_errors(msdr, orc, forc, K):
    modes = msdr.synth.mixed_modes(300)
    codes = fl.adc_stream(300, 128 * 12, seed=27)
    x16 = msdr.synth.batch(modes, 128 * 3)
    g, o = configure_pair(msdr, orc, K, modes)
    with pytest.raises(msdr.capi.MsdrError) as ei:
        g.update_adc(np.ascontiguousarray(codes[:, :128]))
    assert ei.value.status == msdr.capi.ERR_NOT_INITIALISED
    g.set_option("variant", 4096)
    g.enable_frontend()
    fo = forc.frontend(300)
    # ADC, int16, ADC on one chain: the int16 update leaves the front end alone, the FIR history holds IF samples either way
    y1 = g.update_adc(np.ascontiguousarray(codes[:, :128 * 4]))
    fs_before = [bytes(g.get_frontend_state(c)) for c in (0, 299)]
    y2 = g.update(x16)
    assert [bytes(g.get_frontend_state(c)) for c in (0, 299)] == fs_before
    y3 = g.update_adc(np.ascontiguousarray(codes[:, 128 * 4:128 * 8]))
    o1 = o.run(fo.run(codes[:, :128 * 4]))[0]
    o2 = o.run(x16)[0]
    o3 = o.run(fo.run(np.ascontiguousarray(codes[:, 128 * 4:128 * 8])))[0]
    assert_same(np.concatenate([y1, y2, y3], axis=1), np.concatenate([o1, o2, o3], axis=1), "interleaved")
    # move every channel to a second chain (reversed order) and continue there
    g2, _ = configure_pair(msdr, orc, K, modes[::-1])
    g2.set_option("variant", 4096)
    g2.enable_frontend(agc_start=3.0)
    for c in range(300):
        g2.set_state(299 - c, g.get_state(c))
        g2.set_frontend_state(299 - c, g.get_frontend_state(c))
    y4 = g2.update_adc(np.ascontiguousarray(codes[::-1, 128 * 8:]))[::-1]
    o4 = o.run(fo.run(np.ascontiguousarray(codes[:, 128 * 8:])))[0]
    assert_same(y4, o4, "migrated")
    st = g.get_frontend_state(0)
    st.agc_idx = 26
    with pytest.raises(msdr.capi.MsdrError) as ei:
        g.set_frontend_state(0, st)
    assert ei.value.status == msdr.capi.ERR_ARGUMENT


def test_host_path_equals_device_path(msdr, orc, forc, K):
    """update_adc (pinned-ring host pipeline, several chunks) == update_adc_device."""
    import torch
    C_, nb = 300, 10
    modes = msdr.synth.mixed_modes(C_)
    codes = fl.adc_stream(C_, 128 * nb, seed=28)
    ga, _ = configure_pair(msdr, orc, K, modes)
    gb, _ = configure_pair(msdr, orc, K, modes)
    for g in (ga, gb):
        g.set_option("variant", 4096)
        g.enable_frontend()
    ga.set_option("host_chunk_channels", 128)
    ga.set_option("host_chunk_blocks", 3)
    ya = ga.update_adc(codes)
    d_in = torch.from_numpy(codes.view(np.int16)).cuda()
    d_out = torch.empty_like(d_in)
    torch.cuda.synchronize()
    gb.update_adc_device(d_in.data_ptr(), d_out.data_ptr(), nb, d_in.stride(0))
    gb.synchronize()
    assert_same(ya, d_out.cpu().numpy(), "host vs device")
    for c in (0, 127, 128, 299):
        assert bytes(ga.get_frontend_state(c)) == bytes(gb.get_frontend_state(c))


def test_at_size_fused_equals_composition(msdr, orc, forc, K):
    """131 072 channels x 32 blocks x 2 updates: fused == front-end object + chain on the GPU, and the oracle on sampled channels."""
    import torch
    wl = msdr.workloads.get("c5", K)
    C_, nb = 131072, 32
    codes = _torch_codes(torch, C_, 128 * nb * 2)
    g = msdr.ReceiveChain(C_, max_taps=wl.max_taps)
    wl.configure(g)
    g.enable_frontend()
    g2 = msdr.ReceiveChain(C_, max_taps=wl.max_taps)
    wl.configure(g2)
    fe = msdr.Frontend(C_)
    y = torch.empty(C_, 128 * nb, dtype=torch.int16, device="cuda")
    y2, x2 = torch.empty_like(y), torch.empty_like(y)
    chans = msdr.workloads.sample_channels(C_)
    modes = wl.modes(C_)
    o = orc.chain(len(chans))
    for i, c in enumerate(chans):
        o.set_mode(i, 1, modes[c])
        assert o.fir_init(i, 1, *wl.tables_for(modes[c])) == 0
    o.biquad_set_coefficients(0, 0, len(chans), 0, wl.biquad1)
    o.biquad_set_coefficients(1, 0, len(chans), 0, wl.biquad2)
    fo = forc.frontend(len(chans))
    for u in range(2):
        part = codes[:, 128 * nb * u:128 * nb * (u + 1)].contiguous()  # in and out rows share one stride
        torch.cuda.synchronize()
        g.update_adc_device(part.data_ptr(), y.data_ptr(), nb, part.stride(0))
        g.synchronize()
        assert FUSED in g.last_kernel()
        fe.update_device(part.data_ptr(), x2.data_ptr(), nb, part.stride(0))
        fe.synchronize()
        g2.update_device(x2.data_ptr(), y2.data_ptr(), nb, x2.stride(0))
        g2.synchronize()
        assert torch.equal(y, y2), f"update {u}: {(y != y2).sum().item()} samples differ"
        sub = np.ascontiguousarray(part[chans].cpu().numpy().view(np.uint16))
        assert_same(y[chans].cpu().numpy(), o.run(fo.run(sub))[0], f"update {u}, sampled channels vs oracle")


def test_facade_receiver_from_adc_codes(msdr, orc, forc, K):
    """minimal-sdr_b200/host/adc_receiver: Receiver::begin_frontend / update_adc / AGC_val on the C++ façade == the oracles."""
    import os
    import subprocess
    import tempfile
    host = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "minimal-sdr_b200", "host")
    subprocess.run(["make", "-s", "-C", host, "adc_receiver"], check=True)
    C_, NB = 6, 10
    am = np.array(K["FIR_AM_coeffs_bw2800_fs24000"], np.int16)
    codes = fl.adc_stream(C_, 128 * NB, seed=29)
    with tempfile.TemporaryDirectory() as td:
        p = {n: os.path.join(td, n) for n in ("tables.bin", "codes.bin", "out.bin", "agc.bin")}
        np.concatenate([am, am]).tofile(p["tables.bin"])
        codes.tofile(p["codes.bin"])
        r = subprocess.run([os.path.join(host, "adc_receiver"), str(C_), str(NB), str(am.size), p["tables.bin"], p["codes.bin"], p["out.bin"],
                            p["agc.bin"]], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout + r.stderr
        y = np.fromfile(p["out.bin"], np.int16).reshape(C_, NB * 128)
        agc = np.fromfile(p["agc.bin"], np.float32)
    d = msdr.design
    o = orc.chain(C_)
    o.set_mode(0, C_, ol.MODE_AM)
    assert o.fir_init(0, C_, am, am) == 0
    o.biquad_set_coefficients(0, 0, C_, 0, d.biquad_lowpass(3000.0, 0.7071))
    o.biquad_set_coefficients(1, 0, C_, 0, d.biquad_notch(5514.7, 15.0))
    fo = forc.frontend(C_)
    assert_same(y, o.run(fo.run(codes))[0], "adc_receiver")
    assert [a.view(np.uint32) for a in agc] == [fo.state(c)["agc_val"].view(np.uint32) for c in range(C_)]
