"""Full-size checks at BASELINE config 3 scale (4096 channels) through properties that do not need the CPU oracle
on every sample: sampled-channel parity, shard equivalence, partition invariance, determinism."""
import numpy as np
import pytest

import oracle_lib as ol
from chain_helpers import assert_same, tables_for

pytestmark = pytest.mark.gpu


def _setup(msdr, K, C, ch0=0):
    g = msdr.ReceiveChain(C)
    modes = msdr.synth.mixed_modes(C, ch0)
    # channels of the four modes are interleaved: configure everything as AM, then re-tune the others one by one
    g.setup_like_sketch(ol.MODE_AM)
    for c, md in enumerate(modes):
        if md != ol.MODE_AM:
            g.tune(md, c, 1)
    return g, modes


def test_c3_sampled_parity_and_sharding(msdr, orc, K):
    import torch
    C, nb = 4096, 64
    dev = torch.device("cuda:0")
    x = msdr.synth.torch_batch(C, nb * 128, dev)
    g, modes = _setup(msdr, K, C)
    y = torch.empty_like(x)
    g.set_stream(torch.cuda.current_stream().cuda_stream)
    # two updates of 32 blocks: state carried at full size
    for h in range(2):
        xs, ys = x[:, h * 32 * 128:(h + 1) * 32 * 128], y[:, h * 32 * 128:(h + 1) * 32 * 128]
        g.update_device(xs.data_ptr(), ys.data_ptr(), 32, x.stride(0))
    torch.cuda.synchronize()
    yh, xh = y.cpu().numpy(), x.cpu().numpy()
    # (1) oracle on a spread of channels incl. group edges
    pick = sorted(set([0, 1, 2, 3, 31, 32, 33, 1000, 2047, 2048, 4064, 4095] + list(np.random.default_rng(0).integers(0, C, 20))))
    o = orc.chain(len(pick))
    for i, c in enumerate(pick):
        o.set_mode(i, 1, modes[c])
        o.fir_init(i, 1, *tables_for(K, modes[c]))
    o.biquad_set_coefficients(0, 0, len(pick), 0, K["biquad1_lowpass_coef"])
    o.biquad_set_coefficients(1, 0, len(pick), 0, K["biquad2_notch_coef"])
    assert_same(yh[pick], o.run(np.ascontiguousarray(xh[pick]))[0], "C3 sampled channels")
    # (2) determinism + single-update equivalence: a fresh chain fed everything at once gives the same bytes
    g2, _ = _setup(msdr, K, C)
    y2 = torch.empty_like(x)
    g2.set_stream(torch.cuda.current_stream().cuda_stream)
    g2.update_device(x.data_ptr(), y2.data_ptr(), nb, x.stride(0))
    torch.cuda.synchronize()
    assert torch.equal(y, y2)
    # (3) shard equivalence: channels [1024, 2048) processed as their own chain (what another GPU would own)
    g3, _ = _setup(msdr, K, 1024, ch0=1024)
    xs = x[1024:2048].contiguous()
    y3 = torch.empty_like(xs)
    g3.set_stream(torch.cuda.current_stream().cuda_stream)
    g3.update_device(xs.data_ptr(), y3.data_ptr(), nb, xs.stride(0))
    torch.cuda.synchronize()
    assert torch.equal(y3, y[1024:2048])
    assert int(y.abs().max()) > 1000


def test_two_waves_long_update_all_shapes_agree(msdr, orc, K):
    """6000 channels = 188 groups = two waves of chains on 148 SMs, one update of 48 blocks = 12 spans (longer than the
    producers' flow-control window): every kernel shape gives the same bytes, and sampled channels (both waves) match the oracle."""
    import torch
    C, nb = 6000, 48
    dev = torch.device("cuda:0")
    x = msdr.synth.torch_batch(C, nb * 128, dev)
    outs = {}
    # 0 = the chain kernel with two chain sets per SM (188 groups > 148 SMs), 65536 = the time-folded kernel forced (188 group blocks on
    # 148 SMs: 40 CTAs walk two blocks), 512 = one set, helper warps
    for variant in (0, 65536, 512, 2048, 256, 128):
        g, modes = _setup(msdr, K, C)
        g.set_option("variant", variant)
        y = torch.empty_like(x)
        g.set_stream(torch.cuda.current_stream().cuda_stream)
        g.update_device(x.data_ptr(), y.data_ptr(), nb, x.stride(0))
        torch.cuda.synchronize()
        outs[variant] = y
        g.close()
    for variant in (65536, 512, 2048, 256, 128):
        assert torch.equal(outs[0], outs[variant]), f"variant {variant} differs from the default shape"
    pick = [0, 31, 4735, 4736, 4737, 5000, 5999]
    o = orc.chain(len(pick))
    for i, c in enumerate(pick):
        o.set_mode(i, 1, modes[c])
        o.fir_init(i, 1, *tables_for(K, modes[c]))
    o.biquad_set_coefficients(0, 0, len(pick), 0, K["biquad1_lowpass_coef"])
    o.biquad_set_coefficients(1, 0, len(pick), 0, K["biquad2_notch_coef"])
    assert_same(outs[0].cpu().numpy()[pick], o.run(np.ascontiguousarray(x.cpu().numpy()[pick]))[0], "two waves, sampled channels")


def test_c5_channel_count(msdr, orc, K):
    """BASELINE config 5's channel count on one GPU: 2^20 channels (32768 groups, 111 waves of two chain sets per SM), two
    updates of 4 blocks with state carried; sampled channels incl. mode-range, group and wave edges match the oracle, and a
    shard cut out of the middle (what another GPU would own) gives the same bytes."""
    import torch
    C, nb = 1 << 20, 8
    dev = torch.device("cuda:0")
    x = msdr.synth.torch_batch(C, nb * 128, dev)
    q = C // 4
    ranges = [(ol.MODE_AM, 0), (ol.MODE_USB, q), (ol.MODE_LSB, 2 * q), (ol.MODE_CW, 3 * q)]

    def make(c0, n):
        g = msdr.ReceiveChain(n)
        g.setup_like_sketch(ol.MODE_AM)
        for md, start in ranges:
            lo, hi = max(start, c0), min(start + q, c0 + n)
            if md != ol.MODE_AM and lo < hi:
                g.tune(md, lo - c0, hi - lo)
        g.set_stream(torch.cuda.current_stream().cuda_stream)
        return g

    g = make(0, C)
    y = torch.empty_like(x)
    for h in range(2):
        xs, ys = x[:, h * 512:(h + 1) * 512], y[:, h * 512:(h + 1) * 512]
        g.update_device(xs.data_ptr(), ys.data_ptr(), nb // 2, x.stride(0))
    torch.cuda.synchronize()
    rng = np.random.default_rng(5)
    pick = sorted(set([0, 31, 32, 9471, 9472, q - 1, q, q + 1, 2 * q - 1, 2 * q, 3 * q - 1, 3 * q, C - 33, C - 32, C - 1] + list(rng.integers(0, C, 25))))
    idx = torch.tensor(pick, device=dev)
    xh, yh = x[idx].cpu().numpy(), y[idx].cpu().numpy()
    o = orc.chain(len(pick))
    for i, c in enumerate(pick):
        md = ranges[min(c // q, 3)][0]
        o.set_mode(i, 1, md)
        o.fir_init(i, 1, *tables_for(K, md))
    o.biquad_set_coefficients(0, 0, len(pick), 0, K["biquad1_lowpass_coef"])
    o.biquad_set_coefficients(1, 0, len(pick), 0, K["biquad2_notch_coef"])
    assert_same(yh, o.run(np.ascontiguousarray(xh))[0], "C5 channel count, sampled channels")
    assert int(y[idx].abs().max()) > 1000
    # a shard across the USB/LSB boundary, fed everything in one update
    c0, n = 2 * q - 3000, 6000
    g3 = make(c0, n)
    xs = x[c0:c0 + n].contiguous()
    y3 = torch.empty_like(xs)
    g3.update_device(xs.data_ptr(), y3.data_ptr(), nb, xs.stride(0))
    torch.cuda.synchronize()
    assert torch.equal(y3, y[c0:c0 + n])


def _checker_for(msdr, lib, w, chans, ch0=0):
    modes = w.modes(max(chans) + 1, ch0)
    o = lib.chain(len(chans))
    for i, c in enumerate(chans):
        o.set_mode(i, 1, modes[c])
        assert o.fir_init(i, 1, *w.tables_for(modes[c])) == 0
    o.biquad_set_coefficients(0, 0, len(chans), 0, w.biquad1)
    o.biquad_set_coefficients(1, 0, len(chans), 0, w.biquad2)
    return o


def _best_checker(orc):
    return ol.CheckerLib("ref") if ol.have_ref() else orc


def test_c3_benchmarked_launch_shape(msdr, orc, K):
    """The shape bench.py times: 4096 channels, ONE update of 1024 blocks (131 072 samples per channel, 256 spans — far beyond the
    producers' flow-control window), then a second update of 64 blocks carrying the state; 48 sampled channels incl. group and tile
    edges against the compiled reference (oracle/_ref), bit for bit."""
    import torch
    w = msdr.workloads.get("c3", K)
    C = w.channels
    dev = torch.device("cuda:0")
    g = msdr.ReceiveChain(C, max_taps=w.max_taps)
    w.configure(g)
    g.set_stream(torch.cuda.current_stream().cuda_stream)
    chans = msdr.workloads.sample_channels(C)
    o = _checker_for(msdr, _best_checker(orc), w, chans)
    idx = torch.tensor(chans, device=dev)
    n0 = 0
    for nb in (1024, 64):
        x = msdr.synth.torch_batch(C, nb * 128, dev, w.fs, n0=n0)
        y = torch.empty_like(x)
        g.update_device(x.data_ptr(), y.data_ptr(), nb, x.stride(0))
        torch.cuda.synchronize()
        assert_same(y[idx].cpu().numpy(), o.run(np.ascontiguousarray(x[idx].cpu().numpy()))[0], f"C3, update of {nb} blocks")
        assert int(y[idx].abs().max()) > 1000
        n0 += nb * 128
    assert g.plan_build_count() == 1


def test_c4_at_size_fused_chain(msdr, orc, K):
    """BASELINE config 4 at size through the FUSED chain: 16 384 channels (512 groups: more than two per SM), 256 taps (255 + the zero
    arm_fir_init_q15 asks for, arm_fir_init_q15.c:55-64), 192 kHz, updates of 64 + 32 blocks with state carried; sampled channels
    against the compiled reference.  Also: an unchanged configuration builds its row plan once (the 256-tap window used to rebuild it
    twice per update)."""
    import torch
    w = msdr.workloads.get("c4", K)
    C = w.channels
    dev = torch.device("cuda:0")
    g = msdr.ReceiveChain(C, max_taps=w.max_taps)
    w.configure(g)
    assert g.fir_taps(0) == 256 and g.fir_taps(1) == 256
    g.set_stream(torch.cuda.current_stream().cuda_stream)
    chans = msdr.workloads.sample_channels(C)
    o = _checker_for(msdr, _best_checker(orc), w, chans)
    idx = torch.tensor(chans, device=dev)
    n0 = 0
    for nb in (64, 32, 32):
        x = msdr.synth.torch_batch(C, nb * 128, dev, w.fs, n0=n0)
        x[3] = -32768                       # two sampled rows made adversarial: the fs/4 negation corner ...
        x[33, ::2] = 32767                  # ... and full-scale alternation into the long taps
        y = torch.empty_like(x)
        g.update_device(x.data_ptr(), y.data_ptr(), nb, x.stride(0))
        torch.cuda.synchronize()
        assert_same(y[idx].cpu().numpy(), o.run(np.ascontiguousarray(x[idx].cpu().numpy()))[0], f"C4, update of {nb} blocks")
        n0 += nb * 128
    assert int(y[idx].abs().max()) > 300
    assert g.plan_build_count() == 1, "an unchanged configuration must not rebuild the row plan"


def test_c5_interleaved_modes_list_setters(msdr, orc, K):
    """BASELINE config 5's layout as the benchmark runs it: 2^20 channels with mode = {AM,USB,LSB,CW}[c mod 4] (configured with the
    list setters, one call per mode), streamed in three updates of 8 blocks with state carried; sampled channels against the compiled
    reference; a shard from the middle (what another GPU of the job owns: shard.plan) gives the same bytes."""
    import torch
    w = msdr.workloads.get("c5", K)
    C = w.channels
    dev = torch.device("cuda:0")
    g = msdr.ReceiveChain(C, max_taps=w.max_taps)
    w.configure(g)
    g.set_stream(torch.cuda.current_stream().cuda_stream)
    chans = msdr.workloads.sample_channels(C, want=64)
    o = _checker_for(msdr, _best_checker(orc), w, chans)
    idx = torch.tensor(chans, device=dev)
    sh = msdr.shard.plan(C, 8, rank=3)
    g3 = msdr.ReceiveChain(sh.n, max_taps=w.max_taps)
    w.configure(g3, sh.ch0)
    g3.set_stream(torch.cuda.current_stream().cuda_stream)
    for k in range(3):
        x = msdr.synth.torch_batch(C, 8 * 128, dev, w.fs, n0=k * 1024)
        y = torch.empty_like(x)
        g.update_device(x.data_ptr(), y.data_ptr(), 8, x.stride(0))
        xs = x[sh.ch0:sh.ch0 + sh.n].contiguous()
        y3 = torch.empty_like(xs)
        g3.update_device(xs.data_ptr(), y3.data_ptr(), 8, xs.stride(0))
        torch.cuda.synchronize()
        assert_same(y[idx].cpu().numpy(), o.run(np.ascontiguousarray(x[idx].cpu().numpy()))[0], f"C5 layout, update {k}")
        assert torch.equal(y3, y[sh.ch0:sh.ch0 + sh.n]), f"shard of rank 3 of 8 differs in update {k}"
    assert g.plan_build_count() == 1


def test_list_setters_match_ranged_setters(msdr, K):
    """msdr_chain_set_mode_list / msdr_fir_init_q15_list == the ranged calls channel by channel (same output bytes, same state)."""
    import torch
    C, nb = 300, 6
    dev = torch.device("cuda:0")
    w = msdr.workloads.get("c3", K)
    x = msdr.synth.torch_batch(C, nb * 128, dev)
    ga, _ = _setup(msdr, K, C)          # ranged / per-channel calls
    gb = msdr.ReceiveChain(C)
    w.configure(gb)                     # list calls
    outs = []
    for g in (ga, gb):
        y = torch.empty_like(x)
        g.set_stream(torch.cuda.current_stream().cuda_stream)
        g.update_device(x.data_ptr(), y.data_ptr(), nb, x.stride(0))
        torch.cuda.synchronize()
        outs.append(y)
    assert torch.equal(outs[0], outs[1])
    for c in (0, 1, 2, 3, 299):
        sa, sb = ga.get_state(c), gb.get_state(c)
        assert sa.mode == sb.mode and sa.num_taps == sb.num_taps and list(sa.fir_history) == list(sb.fir_history)
        assert [list(r) for r in sa.biquad_definition] == [list(r) for r in sb.biquad_definition]
    # re-binding by list zeroes exactly the listed channels' delay lines (init_FIR, Minimal-SDR.ino:902-903)
    gb.fir_init_list(*w.tables_for(ol.MODE_USB), [1, 5])
    assert not any(gb.get_state(1).fir_history) and not any(gb.get_state(5).fir_history) and any(gb.get_state(2).fir_history)
    with pytest.raises(msdr.MsdrError):
        gb.fir_set_coefficients(np.zeros(10, np.int16), np.zeros(10, np.int16), 0, 1)  # wrong tap count: refused before the C ABI reads past the arrays


def test_row_block_kernel_equals_chain_kernel_at_size(msdr, orc, K):
    """65 536 channels (512 row blocks on 148 SMs: several per CTA, table changes in between), three updates with state carried:
    the row-block kernel (msdr_chain_v5.cu, the default at this size) and the chain kernel (msdr_chain_v4.cu, variant 8192 forbids
    the former) produce the same bytes for EVERY channel, and sampled channels match the compiled reference."""
    import torch
    w = msdr.workloads.get("c5", K)
    C = 65536
    dev = torch.device("cuda:0")
    chains = []
    for variant in (0, 8192):
        g = msdr.ReceiveChain(C, max_taps=w.max_taps)
        g.set_option("variant", variant)
        w.configure(g)
        g.set_stream(torch.cuda.current_stream().cuda_stream)
        chains.append(g)
    chans = msdr.workloads.sample_channels(C)
    o = _checker_for(msdr, _best_checker(orc), w, chans)
    idx = torch.tensor(chans, device=dev)
    n0 = 0
    for nb in (16, 1, 7):
        x = msdr.synth.torch_batch(C, nb * 128, dev, w.fs, n0=n0)
        x[3] = -32768
        ys = []
        for g in chains:
            y = torch.empty_like(x)
            g.update_device(x.data_ptr(), y.data_ptr(), nb, x.stride(0))
            ys.append(y)
        torch.cuda.synchronize()
        assert "v5" in chains[0].last_kernel() and "v4" in chains[1].last_kernel()
        assert torch.equal(ys[0], ys[1]), f"row-block kernel != chain kernel, update of {nb} blocks"
        assert_same(ys[0][idx].cpu().numpy(), o.run(np.ascontiguousarray(x[idx].cpu().numpy()))[0], f"65536 channels, update of {nb} blocks")
        n0 += nb * 128
    for c in (0, 1, 2, 3, 65535):  # carried state words are the same too
        sa, sb = chains[0].get_state(c), chains[1].get_state(c)
        assert list(sa.fir_history) == list(sb.fir_history) and [list(r) for r in sa.biquad_definition] == [list(r) for r in sb.biquad_definition]
