"""Chain-level parity: the fused CUDA chain (through the C ABI, host buffers) against the CPU oracle, the compiled
reference where it travelled, and the golden vectors.  Everything is fixed point => bit-exact, no tolerance."""
import os

import numpy as np
import pytest

import oracle_lib as ol
from chain_helpers import assert_same, configure_pair, run_pair, tables_for
from conftest import adversarial_inputs, wrap_coeffs

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
AM, USB, LSB, CW, SYNCAM = ol.MODE_AM, ol.MODE_USB, ol.MODE_LSB, ol.MODE_CW, ol.MODE_SYNCAM


def test_c1_single_channel_am(msdr, orc, K):
    """BASELINE config 1: one AM channel, 1 s at 44.1 kHz (345 blocks), IF = fs/4, live biquads."""
    x = msdr.synth.batch([AM], 345 * 128)
    g, o = configure_pair(msdr, orc, K, [AM])
    yg, yo = run_pair(g, o, x)
    assert_same(yg, yo, "C1")
    assert np.abs(yg.astype(np.int32)).max() > 500


@pytest.mark.parametrize("mode", [USB, LSB, CW])
def test_c2_single_channel_ssb(msdr, orc, K, mode):
    """BASELINE config 2: one SSB channel with the +-45 degree Hilbert pair, bit-exact vs the q15 path."""
    x = msdr.synth.batch([mode], 345 * 128)
    g, o = configure_pair(msdr, orc, K, [mode])
    yg, yo = run_pair(g, o, x)
    assert_same(yg, yo, f"C2 mode {mode}")
    assert np.abs(yg.astype(np.int32)).max() > 500


def test_chain_golden(msdr, K):
    z = np.load(os.path.join(G, "chain_kat.npz"))
    modes = [int(v) for v in z["modes"]]
    for q31 in (0, 1):
        g = msdr.ReceiveChain(len(modes), am_q31=bool(q31))
        for c, md in enumerate(modes):
            g.set_mode(md, c, 1)
            g.fir_init(*tables_for(K, md), c, 1)
        g.biquad_set_coefficients(0, 0, K["biquad1_lowpass_coef"])
        g.biquad_set_coefficients(1, 0, K["biquad2_notch_coef"])
        assert_same(g.update(z["x"]), z[f"y_q31_{q31}"], f"golden q31={q31}")
        g.close()


def test_against_compiled_reference(msdr, ref, K):
    """Where oracle/_ref travelled: the CUDA chain against the reference's own compiled sources directly."""
    modes = [AM, USB, LSB, CW] * 9 + [AM]  # 37 channels: partial last group
    x = msdr.synth.batch(modes, 128 * 24)
    g, o = configure_pair(msdr, ref, K, modes)
    yg, yo = run_pair(g, o, x, splits=[5, 1, 18])
    assert_same(yg, yo, "vs compiled reference")


@pytest.mark.parametrize("am_q31", [False, True])
def test_mixed_modes_state_carry(msdr, orc, K, am_q31):
    """Mixed AM/SSB/CW batch, state carried across many updates of ragged length (1, 2, 3, 4, 5, 7, 64 blocks ...)."""
    modes = msdr.synth.mixed_modes(70)
    if am_q31:
        modes[5] = SYNCAM  # Teensy 3.2: SYNCAM shares the q31 envelope (.ino:618-620)
    x = msdr.synth.batch(modes, 128 * 90)
    g, o = configure_pair(msdr, orc, K, modes, am_q31=am_q31)
    yg, yo = run_pair(g, o, x, splits=[1, 2, 3, 4, 5, 7, 1, 64, 3])
    assert_same(yg, yo, "mixed modes")


def test_partition_invariance(msdr, K):
    """Same stream in one update vs block-by-block vs uneven chunks gives identical output (GPU vs GPU)."""
    modes = msdr.synth.mixed_modes(33)
    x = msdr.synth.batch(modes, 128 * 20)
    outs = []
    for splits in ([20], [1] * 20, [3, 9, 8], [4, 4, 4, 4, 4]):
        g = msdr.ReceiveChain(len(modes))
        for c, md in enumerate(modes):
            g.setup_like_sketch(md, c, 1)
        b0, ys = 0, []
        for s in splits:
            ys.append(g.update(np.ascontiguousarray(x[:, b0 * 128:(b0 + s) * 128])))
            b0 += s
        outs.append(np.concatenate(ys, axis=1))
        g.close()
    for y in outs[1:]:
        assert_same(y, outs[0], "partition")


def test_adversarial_wrap_and_saturation(msdr, orc, K):
    """Full-scale inputs x taps with sum|c| >> 65536 (accumulator wraps, outputs saturate) x biquads with gain > 1."""
    rng = np.random.default_rng(42)
    ins = adversarial_inputs(128 * 12, rng)
    names = sorted(ins)
    modes = ([AM, USB, LSB, CW] * 8)[:len(names) * 4]
    x = np.stack([ins[names[i // 4]] for i in range(len(modes))])
    tabs = {}
    for c in range(len(modes)):
        T = (86, 102, 38, 4)[c % 4]
        tabs[c] = (wrap_coeffs(T, rng), wrap_coeffs(T, rng))
    hot = [int(1.9 * 2 ** 30), int(-1.7 * 2 ** 30), int(1.9 * 2 ** 30), int(-1.2 * 2 ** 30), int(0.5 * 2 ** 30)]
    bq = [(0, 0, hot, 0, None), (1, 0, K["biquad2_notch_coef"], 0, None)]
    for am_q31 in (False, True):
        g, o = configure_pair(msdr, orc, K, modes, am_q31=am_q31, biquads=bq, tables=tabs)
        yg, yo = run_pair(g, o, x, splits=[5, 7])
        assert_same(yg, yo, f"adversarial q31={am_q31}")
    assert (np.abs(yo.astype(np.int32)) == 32768).any() or (yo == 32767).any()


def test_reference_tables_full_scale(msdr, orc, K):
    """The shipped tables on full-scale inputs (alternating +-32767 at fs/4, all -32768: the -(-32768) corner)."""
    rng = np.random.default_rng(43)
    ins = adversarial_inputs(128 * 8, rng)
    names = sorted(ins)
    modes = [AM, USB, LSB, CW] * len(names)
    x = np.stack([ins[names[i // 4]] for i in range(len(modes))])
    g, o = configure_pair(msdr, orc, K, modes)
    yg, yo = run_pair(g, o, x)
    assert_same(yg, yo, "full scale")


def test_default_biquad_is_silent(msdr, orc, K):
    """A default-constructed AudioFilterBiquad passes nothing (filter_biquad.h:36-39)."""
    x = msdr.synth.batch([AM, USB], 128 * 4)
    g, o = configure_pair(msdr, orc, K, [AM, USB], biquads=None)
    yg, yo = run_pair(g, o, x)
    assert_same(yg, yo, "silent")
    assert not yg.any()


def test_multi_stage_cascades_generic_path(msdr, orc, K):
    """Up to 4 stages per object, different per channel range, a gap (stage 2 without stage 1), stage >= 4 ignored."""
    modes = msdr.synth.mixed_modes(40)
    x = msdr.synth.batch(modes, 128 * 12)
    lp, notch = K["biquad1_lowpass_coef"], K["biquad2_notch_coef"]
    hp = [int(v) for v in msdr.design.biquad_highpass(300.0, 0.7071)]
    bq = [(0, 0, lp, 0, None), (1, 0, notch, 0, None),
          (0, 1, hp, 0, 16), (0, 2, notch, 8, 8), (1, 1, lp, 4, 20), (1, 2, hp, 4, 4), (1, 3, lp, 4, 2),
          (0, 2, hp, 30, 5), (1, 5, lp, 0, None)]
    g, o = configure_pair(msdr, orc, K, modes, biquads=bq)
    yg, yo = run_pair(g, o, x, splits=[3, 9])
    assert_same(yg, yo, "multi-stage")


def test_inplace_coefficient_rewrite_and_mode_change(msdr, orc, K):
    """calc_demod_filter() rewrites the AM table in place mid-stream (state kept, UI.cpp:337-345); tune() re-inits
    (state zeroed, .ino:355); setCoefficients mid-stream keeps x/y history (filter_biquad.cpp:95-98)."""
    modes = [AM] * 40 + [USB] * 8
    x = msdr.synth.batch(modes, 128 * 12)
    g, o = configure_pair(msdr, orc, K, modes)
    y1g, y1o = run_pair(g, o, x[:, :128 * 4])
    am2 = msdr.design.calc_FIR_coeffs(102, 1200, 70, 0, 0.0, 24000)
    g.fir_set_coefficients(am2, am2, 0, 40)            # every user of the table: rewritten in place
    assert o.fir_set_coefficients(0, 40, am2, am2) == 0
    am3 = msdr.design.calc_FIR_coeffs(102, 4000, 70, 0, 0.0, 24000)
    g.fir_set_coefficients(am3, am3, 10, 5)            # a sub-range: copy-on-write, history still kept
    assert o.fir_set_coefficients(10, 5, am3, am3) == 0
    g.biquad_set_coefficients(1, 0, K["biquad1_lowpass_coef"], 0, 20)
    o.biquad_set_coefficients(1, 0, 20, 0, K["biquad1_lowpass_coef"])
    y2g, y2o = run_pair(g, o, x[:, 128 * 4:128 * 8])
    g.set_mode(LSB, 40, 8)                              # mode only: tables and history stay (the sketch needs tune() for more)
    o.set_mode(40, 8, LSB)
    g.set_mode(CW, 0, 3); g.fir_init(*tables_for(K, CW), 0, 3)  # tune(): re-init zeroes the delay lines
    o.set_mode(0, 3, CW); o.fir_init(0, 3, *tables_for(K, CW))
    y3g, y3o = run_pair(g, o, x[:, 128 * 8:])
    for a, b, w in ((y1g, y1o, "before"), (y2g, y2o, "after rewrite"), (y3g, y3o, "after retune")):
        assert_same(a, b, w)


@pytest.mark.parametrize("variant", [0, 4096, 4097])
def test_long_taps_256(msdr, orc, K, variant):
    """BASELINE config 4 shape: 255 taps + one zero (arm_fir_init_q15.c:55-64), 256-tap delay line.  variant 0: the chain kernel (few
    channels); 4096 / 4097: the row-block kernel in its half-tile form for the long window (msdr_chain_v5l.cu), both stage forms."""
    rng = np.random.default_rng(44)
    modes = [AM, USB, LSB, CW] * 5
    c255 = rng.integers(-600, 600, 255).astype(np.int16)
    cI = np.concatenate([c255, [0]]).astype(np.int16)
    cQ = cI[::-1].copy()
    tabs = {c: (cI, cQ) if c % 2 else (wrap_coeffs(256, rng), wrap_coeffs(256, rng)) for c in range(len(modes))}
    x = np.stack([rng.integers(-32768, 32768, 128 * 16, dtype=np.int16) for _ in modes])
    g, o = configure_pair(msdr, orc, K, modes, max_taps=256, tables=tabs)
    g.set_option("variant", variant)
    yg, yo = run_pair(g, o, x, splits=[1, 1, 2, 12])
    assert_same(yg, yo, "256 taps")
    assert ("v5l" in g.last_kernel()) == bool(variant & 4096)


@pytest.mark.parametrize("taps", [30, 150, 200, 250])
def test_window_sizes_on_the_time_folded_kernel(msdr, orc, K, taps):
    """The time-folded kernel (msdr_chain_v6.cu) sizes its operand buffers, its Toeplitz operands and the number of sub-tile slots from
    the window: 30 taps (the shortest window), 150 and 200 (128 words), 250 (160 words, the longest it takes; 256 taps go to the chain
    kernel).  Six tables over 35 channels: half blocks are mostly padding and pair up across tables; mixed modes, wrapping
    taps on some channels, one-block and odd-length updates (a span is 256 samples: the last one is half empty)."""
    rng = np.random.default_rng(taps)
    modes = [AM, USB, LSB, CW, USB] * 7
    six = []
    for k in range(6):
        if k % 3 == 0:
            six.append((wrap_coeffs(taps, rng), wrap_coeffs(taps, rng)))
        else:
            cI = rng.integers(-700, 700, taps).astype(np.int16)
            six.append((cI, cI[::-1].copy()))
    tabs = {c: six[(c * 5) % 6] for c in range(len(modes))}
    x = np.stack([rng.integers(-32768, 32768, 128 * 23, dtype=np.int16) for _ in modes])
    g, o = configure_pair(msdr, orc, K, modes, max_taps=taps, tables=tabs)
    yg, yo = run_pair(g, o, x, splits=[1, 3, 1, 2, 16])
    assert_same(yg, yo, f"{taps} taps")
    if not os.environ.get("MSDR_VARIANT"):  # (the whole-file re-runs force another kernel through the environment)
        assert "v6::" in g.last_kernel(), g.last_kernel()


def test_errors_match_reference_conventions(msdr, K):
    g = msdr.ReceiveChain(8)
    am = np.array(K["FIR_AM_coeffs_bw2800_fs24000"], np.int16)
    x = np.zeros((8, 128), np.int16)
    with pytest.raises(msdr.MsdrError) as e:
        g.update(x)                                     # FIR never bound
    assert e.value.status == msdr.capi.ERR_NOT_INITIALISED
    assert g.fir_init(am[:85], am[:85], check=False) == -1   # ARM_MATH_ARGUMENT_ERROR for odd numTaps
    with pytest.raises(msdr.MsdrError):
        g.fir_init(np.zeros(104, np.int16), np.zeros(104, np.int16))  # longer than this chain's max_taps (102)
    with pytest.raises(msdr.MsdrError):
        g.set_mode(7)
    g.fir_init(am, am)
    g.biquad_set_coefficients(0, 7, K["biquad1_lowpass_coef"])  # stage >= 4: silently ignored
    assert not g.update(x).any()
    with pytest.raises(msdr.MsdrError):
        g.set_mode(AM, 4, 5)                            # range past the end
    g.close()


def test_state_checkpoint_resume_and_migration(msdr, orc, K):
    """get_state/set_state: stop a stream, move every channel into a fresh chain in permuted order, continue — the
    output equals the uninterrupted run; the exported state equals what the reference objects hold."""
    modes = msdr.synth.mixed_modes(12)
    x = msdr.synth.batch(modes, 128 * 10)
    g, o = configure_pair(msdr, orc, K, modes)
    yg, yo = run_pair(g, o, x)
    g1 = msdr.ReceiveChain(len(modes))
    for c, md in enumerate(modes):
        g1.setup_like_sketch(md, c, 1)
    ya = g1.update(np.ascontiguousarray(x[:, :128 * 6]))
    perm = np.random.default_rng(3).permutation(len(modes))
    g2 = msdr.ReceiveChain(len(modes))
    for dst, src in enumerate(perm):
        st = g1.get_state(int(src))
        assert st.mode == modes[src] and st.num_taps in (86, 102)
        # FIR history = the last num_taps-1 raw input samples
        assert list(st.fir_history[:st.num_taps - 1]) == list(x[src, 128 * 6 - (st.num_taps - 1):128 * 6])
        g2.fir_init(*tables_for(K, modes[src]), dst, 1)
        g2.set_state(dst, st)
    yb = g2.update(np.ascontiguousarray(x[perm][:, 128 * 6:]))
    assert_same(np.concatenate([ya, yb[np.argsort(perm)]], axis=1), yo, "resume")
    # biquad words match the oracle's AudioFilterBiquad::definition after the same stream
    import ctypes as C
    d = np.zeros(32, np.int32)
    for c in (0, 5, 11):
        st = g.get_state(c)
        for obj in (0, 1):
            orc.lib.orc_chain_get_biquad_definition(C.c_void_p(o.h), c, obj, d.ctypes.data_as(C.c_void_p))
            assert list(st.biquad_definition[obj]) == list(d), (c, obj)


def test_strided_host_buffers(msdr, orc, K):
    """Row stride larger than the payload, on both host buffers."""
    modes = msdr.synth.mixed_modes(9)
    x = msdr.synth.batch(modes, 128 * 5)
    big = np.full((9, 128 * 5 + 24), 7, np.int16)
    big[:, :128 * 5] = x
    outbig = np.full_like(big, -3)
    g, o = configure_pair(msdr, orc, K, modes)
    g.update(big[:, :128 * 5], out=outbig[:, :128 * 5])
    assert_same(outbig[:, :128 * 5], o.run(x)[0], "strided")
    assert (outbig[:, 128 * 5:] == -3).all()


def test_device_buffers_and_stream(msdr, orc, K):
    """msdr_chain_update_device on torch tensors, on torch's current stream."""
    import torch
    modes = msdr.synth.mixed_modes(64)
    x = msdr.synth.batch(modes, 128 * 16)
    g, o = configure_pair(msdr, orc, K, modes)
    d_in = torch.from_numpy(x).cuda()
    d_out = torch.zeros_like(d_in)
    g.set_stream(torch.cuda.current_stream().cuda_stream)
    g.update_device(d_in.data_ptr(), d_out.data_ptr(), 16, d_in.stride(0))
    torch.cuda.synchronize()
    assert_same(d_out.cpu().numpy(), o.run(x)[0], "device")
    with pytest.raises(msdr.MsdrError):
        g.update_device(d_in.data_ptr() + 2, d_out.data_ptr(), 16, d_in.stride(0))  # misaligned


def test_host_update_pipeline_chunks(msdr, orc, K):
    """msdr_chain_update streams channel chunks through a 3-slot device ring; force tiny chunks (incl. a ragged last one,
    more chunks than slots) and check against the oracle and against the unchunked call."""
    modes = msdr.synth.mixed_modes(203)
    x = msdr.synth.batch(modes, 128 * 9)
    g, o = configure_pair(msdr, orc, K, modes)
    g.set_option("host_chunk_channels", 32)
    g.set_option("host_chunk_blocks", 2)
    yg, yo = run_pair(g, o, x, splits=[2, 7])
    assert_same(yg, yo, "chunked host update")
    pin, pout = msdr.capi.PinnedBuffer(x.shape), msdr.capi.PinnedBuffer(x.shape)
    pin.array[:] = x
    g2, _ = configure_pair(msdr, orc, K, modes)
    g2.set_option("host_chunk_channels", 64)
    g2.update(pin.array, out=pout.array)
    assert_same(pout.array, yo, "pinned buffers")
    pin.free(); pout.free()


def test_update_range_device(msdr, orc, K):
    """Channel sub-ranges updated independently (any order) equal the whole-chain update."""
    import torch
    modes = msdr.synth.mixed_modes(100)
    x = msdr.synth.batch(modes, 128 * 6)
    g, o = configure_pair(msdr, orc, K, modes)
    yo = o.run(x)[0]
    d_in = torch.from_numpy(x).cuda()
    d_out = torch.zeros_like(d_in)
    s = torch.cuda.Stream()
    g.set_stream(s.cuda_stream)
    for c0, n in ((64, 36), (0, 32), (32, 32)):
        g.update_range_device(c0, n, d_in[c0:].data_ptr(), d_out[c0:].data_ptr(), 6, d_in.stride(0))
    g.synchronize()
    assert_same(d_out.cpu().numpy(), yo, "range update")


@pytest.mark.parametrize("variant,name", [(0, "default (time-folded kernel, msdr_chain_v6.cu)"), (16384, "chain kernel (msdr_chain_v4.cu), feed-forward helper warps"),
                                            (2048, "tensor-core FIR + post warps"),
                                            (256, "tensor-core FIR, inline epilogue"), (128, "helper warps, forced"),
                                            (2, "time-folded kernel, DFMA feed-forward"), (4096, "row-block kernel (msdr_chain_v5.cu), forced"),
                                            (4097, "row-block kernel, IMAD.WIDE stages"), (4098, "row-block kernel, DFMA feed-forward"),
                                            (4100, "row-block kernel, chained DFMA feed-forward"), (4104, "row-block kernel, all five products one DFMA chain"),
                                            (4108, "row-block kernel, split 16 x 16-bit products")])
def test_every_kernel_shape_is_bit_exact(msdr, orc, K, variant, name):
    """All shapes of the fused kernel (option "variant") produce the oracle's bits: mixed modes, ragged updates, 4-stage cascades on
    some channels, full-range (wrapping) taps on others, extreme inputs, a partial last group."""
    rng = np.random.default_rng(variant)
    modes = msdr.synth.mixed_modes(200) + [USB, AM, CW]
    x = msdr.synth.batch(modes, 128 * 41)
    x[7] = rng.integers(-32768, 32768, x.shape[1], dtype=np.int16)
    x[8] = -32768
    lp, notch = K["biquad1_lowpass_coef"], K["biquad2_notch_coef"]
    bq = [(0, 0, lp, 0, None), (1, 0, notch, 0, None)]
    bq += [(0, st, lp, 40, 10) for st in range(1, 4)] + [(1, st, lp, 100, 32) for st in range(1, 4)]
    # b2 != b0 (band-pass / shelf shapes): a whole channel group of object 1, and single lanes of otherwise symmetric groups
    asym = [int(0.31 * 2 ** 30), int(0.05 * 2 ** 30), int(-0.29 * 2 ** 30), int(1.1 * 2 ** 30), int(-0.6 * 2 ** 30)]
    bq += [(0, 0, asym, 64, 32), (1, 0, asym, 130, 1), (0, 0, asym, 199, 1)]
    g, o = configure_pair(msdr, orc, K, modes, biquads=bq)
    g.set_option("variant", variant)
    cI, cQ = wrap_coeffs(86, rng), wrap_coeffs(86, rng)  # the accumulator wraps, outputs saturate
    g.fir_init(cI, cQ, 7, 2)
    assert o.fir_init(7, 2, cI, cQ) == 0
    yg, yo = run_pair(g, o, x, splits=[3, 1, 17, 2, 18])
    assert_same(yg, yo, name)
    want = "v6::" if variant in (0, 2) else "v5::" if variant & 4096 else "v4::"
    assert want in g.last_kernel(), (variant, g.last_kernel())


def test_syncam_channels_in_a_chain(msdr, orc, K):
    """Mode SYNCAM on the f32 build = the PLL demodulator (Minimal-SDR.ino:631-688), run beside the fused kernel for those channels.
    Every other channel stays bit-exact; SYNCAM channels meet the float tolerance (libm-dependent path) after both biquads, with
    FIR history, PLL state and biquad state carried over ragged updates and across a migration to another chain."""
    modes = msdr.synth.mixed_modes(70)
    pll = [3, 4, 5, 40, 64, 69]
    for c in pll:
        modes[c] = SYNCAM
    x = msdr.synth.batch(modes, 128 * 60)
    g, o = configure_pair(msdr, orc, K, modes)
    yo = o.run(x)[0]
    outs, b0 = [], 0
    for n in (1, 7, 22):
        outs.append(g.update(np.ascontiguousarray(x[:, b0 * 128:(b0 + n) * 128])))
        b0 += n
    g2, _ = configure_pair(msdr, orc, K, modes)  # migrate every channel to a fresh chain mid-stream
    for c in range(len(modes)):
        g2.set_state(c, g.get_state(c))
    outs.append(g2.update(np.ascontiguousarray(x[:, b0 * 128:])))
    yg = np.concatenate(outs, axis=1)
    others = [c for c in range(len(modes)) if c not in pll]
    assert_same(yg[others], yo[others], "non-SYNCAM channels next to SYNCAM ones")
    a, b = yg[pll].astype(np.float64), yo[pll].astype(np.float64)
    assert np.abs(b).max() > 300
    assert np.abs(a - b).max() <= 2                                                  # a 1-LSB difference through two biquads
    assert np.sqrt(np.mean((a - b) ** 2)) <= 1e-5 * np.sqrt(np.mean(b ** 2)) + 0.02   # 1e-5 relative RMS (+ the LSB flips of quiet channels)
    assert (yg[pll] != yo[pll]).mean() < 0.01


def test_anr_channels_in_a_chain(msdr, orc, K):
    """ANR_on per channel (LMS notch = 1 / noise reduction = 2, Minimal-SDR.ino:702-770) sits between demodulation and the biquads.
    The float LMS is bit-exact, so channels with ANR on are bit-exact too; ANR is switched on and off mid-stream (its state is
    kept), channels migrate with their LMS state; a SYNCAM + ANR channel meets the float tolerance."""
    modes = msdr.synth.mixed_modes(40)
    modes[9] = SYNCAM
    x = msdr.synth.batch(modes, 128 * 48)
    g, _ = configure_pair(msdr, orc, K, modes)
    notch_ch, nr_ch = [1, 2, 3, 9, 33], [16, 17, 39]

    def set_anr(gg, chans, v):
        for c in chans:
            gg.set_anr(v, c, 1)
    outs = [g.update(np.ascontiguousarray(x[:, :128 * 4]))]           # ANR off everywhere
    set_anr(g, notch_ch, 1)
    set_anr(g, nr_ch, 2)
    outs.append(g.update(np.ascontiguousarray(x[:, 128 * 4:128 * 20])))
    set_anr(g, [2], 0)                                              # off again for one channel ...
    outs.append(g.update(np.ascontiguousarray(x[:, 128 * 20:128 * 30])))
    set_anr(g, [2], 2)                                              # ... and back on in the other mode: the LMS state was kept
    g2, _ = configure_pair(msdr, orc, K, modes)                        # migrate to a fresh chain
    set_anr(g2, notch_ch, 1)
    set_anr(g2, nr_ch, 2)
    set_anr(g2, [2], 2)
    for c in range(len(modes)):
        g2.set_state(c, g.get_state(c))
    for c in notch_ch + nr_ch:
        g2.set_anr_state(c, g.get_anr_state(c))
    outs.append(g2.update(np.ascontiguousarray(x[:, 128 * 30:])))
    yg = np.concatenate(outs, axis=1)
    # the oracle sees the same schedule
    o2_parts = []
    g_, oo = configure_pair(msdr, orc, K, modes)  # a second oracle chain driven through the same schedule at the same block boundaries
    g_.close()
    o2_parts.append(oo.run(np.ascontiguousarray(x[:, :128 * 4]))[0])
    for c in notch_ch:
        assert oo.set_anr(c, 1, 1) == 0
    for c in nr_ch:
        assert oo.set_anr(c, 1, 2) == 0
    o2_parts.append(oo.run(np.ascontiguousarray(x[:, 128 * 4:128 * 20]))[0])
    assert oo.set_anr(2, 1, 0) == 0
    o2_parts.append(oo.run(np.ascontiguousarray(x[:, 128 * 20:128 * 30]))[0])
    assert oo.set_anr(2, 1, 2) == 0
    o2_parts.append(oo.run(np.ascontiguousarray(x[:, 128 * 30:]))[0])
    yo = np.concatenate(o2_parts, axis=1)
    exact = [c for c in range(len(modes)) if c != 9]
    assert_same(yg[exact], yo[exact], "chain with ANR channels")
    a, b = yg[9].astype(np.float64), yo[9].astype(np.float64)        # SYNCAM + notch: float tolerance
    assert np.abs(a - b).max() <= 3 and np.sqrt(np.mean((a - b) ** 2)) <= 1e-4 * np.sqrt(np.mean(b ** 2)) + 0.05


def test_side_lane_is_cached_and_asynchronous(msdr, orc, K):
    """Channels with the LMS notch on are finished beside the fused kernel; the lane's index vectors are cached per range and
    configuration and nothing waits for the stream.  Device-resident updates queued back to back on one stream without a host sync in
    between: the same range repeated (cache hits), two ranges alternating (misses that overwrite the cached vectors while earlier lane
    kernels are still queued), the ANR switch of a channel changed between updates (invalidation).  Bit-exact against the oracle."""
    import torch
    modes = msdr.synth.mixed_modes(96)
    nb = [3, 2, 4, 3]
    x = msdr.synth.batch(modes, 128 * sum(nb))
    g, o = configure_pair(msdr, orc, K, modes)
    anr = {1: 1, 2: 2, 40: 1, 63: 2, 64: 1, 95: 2}
    for c, v in anr.items():
        g.set_anr(v, c, 1)
        assert o.set_anr(c, 1, v) == 0
    d_in = torch.from_numpy(x).cuda()
    d_out = torch.zeros_like(d_in)
    st = torch.cuda.Stream()
    g.set_stream(st.cuda_stream)
    parts, b0 = [], 0
    for i, n in enumerate(nb):
        if i == 2:  # between updates: one channel's notch off, another one on
            g.synchronize()
            g.set_anr(0, 40, 1); g.set_anr(1, 41, 1)
            assert o.set_anr(40, 1, 0) == 0 and o.set_anr(41, 1, 1) == 0
        col = b0 * 128
        if i == 1:  # the whole chain in one call, twice the same range afterwards
            g.update_range_device(0, 96, d_in[:, col:].data_ptr(), d_out[:, col:].data_ptr(), n, d_in.stride(0))
        else:       # two ranges alternating
            for c0, cn in ((64, 32), (0, 64)):
                g.update_range_device(c0, cn, d_in[c0:, col:].data_ptr(), d_out[c0:, col:].data_ptr(), n, d_in.stride(0))
        parts.append(o.run(np.ascontiguousarray(x[:, col:col + n * 128]))[0])
        b0 += n
    g.synchronize()
    assert_same(d_out.cpu().numpy(), np.concatenate(parts, axis=1), "side lane, cached index vectors")


def test_whole_file_on_the_chain_kernel():
    """The time-folded kernel (msdr_chain_v6.cu) is the default for few channels, so this file runs on it; MSDR_VARIANT=16384 forbids it
    and the chain tests run again on the chain kernel (msdr_chain_v4.cu), which still serves the channel counts between the two
    other kernels and the 256-tap window at few channels."""
    import subprocess
    import sys
    env = dict(os.environ, MSDR_VARIANT="16384")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-m", "gpu", "-k",
                        "not every_kernel_shape and not whole_file and not errors_match"], env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]


def test_whole_file_on_the_row_block_kernel():
    """The row-block kernel (msdr_chain_v5.cu) is chosen for many channels; MSDR_VARIANT=4096 forces it for ANY channel count, and
    this file's chain tests run again on it in a child process: single channels, ragged updates, partial row blocks, wrap / saturation
    taps, multi-stage cascades, coefficient rewrites, state migration, host chunking, range updates, SYNCAM / ANR side lanes.
    (256 taps do not fit that kernel: those cases fall back to the chain kernel, as in production.)"""
    import subprocess
    import sys
    env = dict(os.environ, MSDR_VARIANT="4096")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-m", "gpu", "-k",
                        "not every_kernel_shape and not whole_file and not errors_match"], env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
