"""The host code between a chain update and its kernel (csrc/msdr_capi.cu), at its edges: which kernel update_range picks on both
sides of every channel-count threshold, the row plans of build_tc_plan over MSDR_MAX_FIR_SETS tables with ragged row counts and mixed
windows, table slots given back and reused by both FIR setters, channel ranges that start anywhere, and the per-range plan cache and
its eviction.  A padding row, a wrong table id in a row block or a stale cached plan gives wrong bits, so every comparison is byte for
byte against the CPU oracle, on every channel; every case also asserts the kernel family it expects in last_kernel()."""
import os
import re
from collections import Counter

import numpy as np
import pytest

import frontend_lib as fl
import oracle_lib as ol
from chain_helpers import assert_same, configure_pair
from conftest import wrap_coeffs

pytestmark = pytest.mark.gpu
AM, USB, LSB, CW = ol.MODE_AM, ol.MODE_USB, ol.MODE_LSB, ol.MODE_CW
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _max_fir_sets():
    with open(os.path.join(ROOT, "include", "msdr.h")) as f:
        return int(re.search(r"#define\s+MSDR_MAX_FIR_SETS\s+(\d+)", f.read()).group(1))


MAX_SETS = _max_fir_sets()
RAGGED_ROWS = (1, 15, 16, 17, 31, 33, 127, 128, 129)  # around the 16-row half block (v6) and the 128-row block (v4 / v5)
SHORT_TAPS = (4, 6, 30, 38, 86, 100, 102)


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def forc():
    return fl.Orc()


# ---- what update_range should pick ------------------------------------------------------------------------------------------

def family(kernel):
    """Kernel family named by msdr_chain_last_kernel."""
    if "v6::" in kernel:
        return "v6"
    if "v5l::" in kernel:
        return "v5l"
    if "v5::" in kernel:
        return "v5"
    if "v4::" in kernel:
        return "v4 two sets" if "two chain sets per SM" in kernel else "v4 one set"
    raise AssertionError(f"unknown kernel: {kernel}")


def v6_group_blocks(table_of):
    """Group blocks of the time-folded kernel's plan: each table's rows cut into 16-row halves (the last one padded), two halves a block."""
    halves = sum(-(-n // 16) for n in Counter(table_of).values())
    return -(-halves // 2)


def predict(nch, n_gb, sms, spare=0):
    """update_range's choice with variant 0 for windows every kernel takes (up to 102 taps): the row-block kernel from
    min(12288, 64 SMs + 1) channels on, the time-folded kernel while its group blocks fit the SMs not kept spare (and at most 8192
    channels), else the chain kernel, with two chain sets per SM when there are more channel groups than SMs."""
    if nch >= min(12288, 64 * sms + 1):
        return "v5"
    if nch <= 8192 and n_gb <= max(1, sms - spare):
        return "v6"
    return "v4 two sets" if -(-nch // 32) > sms else "v4 one set"


# ---- chains ----------------------------------------------------------------------------------------------------------------

def _table(T, rng, wrap=False):
    if wrap:  # sum |c| >> 65536: the accumulator wraps and the outputs saturate
        return wrap_coeffs(T, rng), wrap_coeffs(T, rng)
    cI = rng.integers(-700, 700, T).astype(np.int16)
    return cI, cI[::-1].copy()


def _interleave(counts, rng):
    """table id per channel: table k on counts[k] channels, shuffled so that no table with more than one row is contiguous."""
    table_of = rng.permutation(np.repeat(np.arange(len(counts)), counts))
    for k, n in enumerate(counts):
        where = np.flatnonzero(table_of == k)
        assert n < 2 or where[-1] - where[0] + 1 > n, f"table {k} came out contiguous"
    return table_of


def _pair(msdr, orc, K, modes, table_of, tables, max_taps=0):
    """GPU chain and oracle chain with tables[table_of[c]] on channel c (one ranged call per channel), the sketch's live biquads."""
    return configure_pair(msdr, orc, K, modes, max_taps=max_taps, tables={c: tables[t] for c, t in enumerate(table_of)})


def _run(g, o, x, splits, want):
    """x through both chains in updates of `splits` blocks; the kernel family is checked after every update."""
    yg, yo, b0 = [], [], 0
    for s in splits:
        part = np.ascontiguousarray(x[:, 128 * b0:128 * (b0 + s)])
        yg.append(g.update(part))
        assert family(g.last_kernel()) == want, (want, g.last_kernel())
        yo.append(o.run(part)[0])
        b0 += s
    return np.concatenate(yg, axis=1), np.concatenate(yo, axis=1)


def _adversarial_rows(x, rng, low, full):
    """all -32768 (the fs/4 negation corner) on `low`, full-scale noise on `full`."""
    for c in low:
        x[c] = -32768
    for c in full:
        x[c] = rng.integers(-32768, 32768, x.shape[1], dtype=np.int16)


# ---- 1. the selection thresholds, both sides --------------------------------------------------------------------------------

THRESHOLD_CASES = {  # name: (channels, spare_sms, family) from the SM count
    "32sms": lambda s: (32 * s, 0, "v6"),
    "32sms+1": lambda s: (32 * s + 1, 0, "v4 two sets"),
    "v5min-1": lambda s: (min(12288, 64 * s + 1) - 1, 0, "v4 two sets"),
    "v5min": lambda s: (min(12288, 64 * s + 1), 0, "v5"),
    "ragged_tables": lambda s: (32 * (s - 4), 0, "v4 one set"),
    "spare8": lambda s: (32 * (s - 8), 8, "v6"),
    "spare8+1": lambda s: (32 * (s - 8) + 1, 8, "v4 one set"),
}


@pytest.mark.parametrize("case", list(THRESHOLD_CASES))
def test_selection_threshold_every_channel(msdr, orc, K, sms, case):
    """Channel counts on both sides of each threshold of the kernel choice, derived from the SM count: 32 SMs (time-folded kernel)
    against 32 SMs + 1 (chain kernel, two chain sets per SM), the last count below the row-block kernel and the first one on it,
    spare_sms = 8 moving the time-folded kernel's edge, and fewer channel groups than SMs whose ragged tables still need more group
    blocks than there are SMs.  Mixed modes; the bulk of the channels share one table pair, a wrapping table sits on 16 channels
    including 31 / 32, 127 / 128 and the last one (16 rows: the group-block count stays ceil(channels / 32)), with adversarial inputs
    on those; updates of 3, 1 and 2 blocks; every channel against the oracle."""
    nch, spare, want = THRESHOLD_CASES[case](sms)
    rng = np.random.default_rng(nch)
    modes = msdr.synth.mixed_modes(nch)
    am = np.array(K["FIR_AM_coeffs_bw2800_fs24000"], np.int16)
    tables = [(am, am), _table(86, rng, wrap=True)]
    table_of = np.zeros(nch, np.int64)
    edge = [31, 32, 127, 128, nch - 1]
    table_of[edge + [1, 2, 33, 95, 96, 160, 255, 256, 257, 1000, 1001]] = 1
    if case == "ragged_tables":  # 24 more tables of 33 rows, interleaved: 15 padding rows in every last half block
        for k in range(24):
            tables.append(_table(SHORT_TAPS[k % len(SHORT_TAPS)], rng, wrap=k % 5 == 0))
        free = np.flatnonzero(table_of == 0)
        pick = rng.choice(free, 24 * 33, replace=False)
        table_of[pick] = 2 + np.arange(24 * 33) // 33
    n_gb = v6_group_blocks(table_of)
    if case != "ragged_tables":
        assert n_gb == -(-nch // 32)
    else:
        assert -(-nch // 32) <= sms < n_gb
    assert predict(nch, n_gb, sms, spare) == want, (case, nch, n_gb, sms)
    x = msdr.synth.batch(modes, 128 * 6)
    _adversarial_rows(x, rng, low=[31, 128, nch - 1], full=[32, 127])
    g, o = _pair(msdr, orc, K, modes, table_of, tables)
    g.set_option("variant", 0)
    g.set_option("spare_sms", spare)
    yg, yo = _run(g, o, x, [3, 1, 2], want)
    assert_same(yg, yo, f"{case}: {nch} channels, {n_gb} group blocks, {sms} SMs, spare {spare}")


def test_forced_time_folded_kernel_after_a_cached_plan(msdr, orc, K, sms):
    """A variant that asks for the time-folded kernel takes effect on a range whose plan is already cached.  9000 channels run the
    chain kernel with two chain sets per SM at variant 0, and that plan has no group blocks (more than 8192 channels); after
    set_option("variant", 65536) the next update of the same range runs the time-folded kernel.  Every channel against the oracle."""
    nch = 9000
    rng = np.random.default_rng(nch)
    modes = msdr.synth.mixed_modes(nch)
    am = np.array(K["FIR_AM_coeffs_bw2800_fs24000"], np.int16)
    tables = [(am, am), _table(86, rng, wrap=True)]
    table_of = np.zeros(nch, np.int64)
    table_of[[1, 31, 32, 127, 128, 4000, nch - 1]] = 1
    assert predict(nch, v6_group_blocks(table_of), sms) == "v4 two sets"
    x = msdr.synth.batch(modes, 128 * 4)
    _adversarial_rows(x, rng, low=[31, nch - 1], full=[32, 128])
    g, o = _pair(msdr, orc, K, modes, table_of, tables)
    g.set_option("variant", 0)
    y0 = _run(g, o, x[:, :128 * 2], [2], "v4 two sets")
    g.set_option("variant", 65536)
    y1 = _run(g, o, x[:, 128 * 2:], [2], "v6")
    assert_same(np.concatenate([y0[0], y1[0]], axis=1), np.concatenate([y0[1], y1[1]], axis=1), f"{nch} channels, variant 0 then 65536")


# ---- 2. MSDR_MAX_FIR_SETS tables on every kernel ----------------------------------------------------------------------------

def _full_layout(msdr, K, sms, layout):
    """MSDR_MAX_FIR_SETS distinct tables with ragged row counts, interleaved over the channels.
    base: the short taps, some wrapping.  wide: the same with one table grown (128 k + 1 rows) past 32 SMs channels, so that there
    are more channel groups than SMs.  taps256: 256-tap tables among the short ones (a max_taps=256 chain: one window for all)."""
    rng = np.random.default_rng(len(layout))
    counts = [RAGGED_ROWS[k % len(RAGGED_ROWS)] for k in range(MAX_SETS)]
    if layout == "wide":
        k = counts.index(129)
        counts[k] += 128 * max(0, -(-(32 * sms + 1 - sum(counts)) // 128))
    taps = list(SHORT_TAPS) + ([256] if layout == "taps256" else [])
    tables = [_table(taps[k % len(taps)], rng, wrap=k % 3 == 1) for k in range(MAX_SETS)]
    table_of = _interleave(counts, rng)
    modes = [(AM, USB, LSB, CW, USB)[(c * 7) % 5] for c in range(len(table_of))]
    return modes, table_of, tables, rng


FULL_CASES = [("base", 0, "v6"), ("base", 16384, "v4 one set"), ("base", 512, "v4 one set"), ("base", 4096, "v5"),
              ("base", 4096 | 32768, "v5l"), ("wide", 0, "v4 two sets"), ("wide", 512, "v4 one set"),
              ("taps256", 0, "v4 one set"), ("taps256", 4096, "v5l")]


@pytest.mark.parametrize("layout,variant,want", FULL_CASES)
def test_full_table_count_every_kernel(msdr, orc, K, sms, layout, variant, want):
    """MSDR_MAX_FIR_SETS tables of 4 ... 102 taps (256 in the long-window chain), some wrapping, on 1, 15, 16, 17, 31, 33, 127, 128 and
    129 channels each, no table contiguous: every row block and half block of the plans mixes padding and table changes.  Each kernel
    in turn (wide: more channel groups than SMs, two chain sets per SM, and one set in two waves).  Then a table beyond the limit is
    refused with ERR_NOMEM by both setters, and the chain carries on unchanged."""
    modes, table_of, tables, rng = _full_layout(msdr, K, sms, layout)
    nch = len(table_of)
    if variant == 0 and layout != "taps256":
        assert predict(nch, v6_group_blocks(table_of), sms) == want
    x = msdr.synth.batch(modes, 128 * 7)
    rows = Counter(table_of.tolist())
    ones = [c for c in range(nch) if rows[table_of[c]] > 1]
    _adversarial_rows(x, rng, low=ones[:3] + [nch - 1], full=ones[3:6])
    g, o = _pair(msdr, orc, K, modes, table_of, tables, max_taps=256 if layout == "taps256" else 0)
    g.set_option("variant", variant)
    yg, yo = _run(g, o, x[:, :128 * 6], [1, 3, 2], want)
    assert_same(yg, yo, f"{layout}, variant {variant}: {nch} channels, {MAX_SETS} tables")
    # one more distinct table, on a channel whose table keeps other users: no slot to give it
    c = ones[7]
    slot = g.get_state(c).fir_set
    extra = _table(30, rng)
    assert g.fir_init(*extra, c, 1, check=False) == msdr.capi.ERR_NOMEM
    with pytest.raises(msdr.MsdrError) as e:  # listed as often as its table has users: still one user of it
        g.fir_init_list(*extra, [c] * rows[table_of[c]])
    assert e.value.status == msdr.capi.ERR_NOMEM
    assert g.get_state(c).fir_set == slot
    yg, yo = _run(g, o, x[:, 128 * 6:], [1], want)
    assert_same(yg, yo, f"{layout}, variant {variant}: after the refused table")


# ---- 3. slots given back and reused, by the ranged and the list setter -------------------------------------------------------

def _list_chain(msdr, K, modes, table_of, tables):
    """The chain of _pair, configured with the list setters: one call per mode and per table, tables in order of first use (the slot
    numbers of the per-channel ranged calls)."""
    g = msdr.ReceiveChain(len(modes))
    for md in sorted(set(modes)):
        g.set_mode_list(md, [c for c, m in enumerate(modes) if m == md])
    _, first = np.unique(table_of, return_index=True)
    for t in table_of[np.sort(first)]:
        g.fir_init_list(*tables[t], np.flatnonzero(table_of == t))
    for obj, key in ((0, "biquad1_lowpass_coef"), (1, "biquad2_notch_coef")):
        g.biquad_set_coefficients(obj, 0, K[key])
    return g


@pytest.mark.parametrize("variant,want", [(0, "v6"), (16384, "v4 one set"), (4096, "v5")])
def test_full_chain_retune_ranged_and_list(msdr, orc, K, variant, want):
    """A chain with MSDR_MAX_FIR_SETS live tables re-tunes every user of one table to a new table, through the ranged call on one chain
    and through the list call on another: both give the old table's slot to the new one.  Then back to the old table and to the new
    one again: the same slot holds other taps each time, so a cached plan or Toeplitz operand that outlived the change would show.
    After each change the next update builds exactly one plan, both chains equal the oracle, and they equal each other in output and
    in every channel's state.  Last, the list call re-tunes a table whose users are spread over the chain."""
    rng = np.random.default_rng(variant + 7)
    counts = [(1, 15, 16, 17, 31, 33)[k % 6] for k in range(MAX_SETS)]
    tables = [_table(SHORT_TAPS[k % len(SHORT_TAPS)], rng, wrap=k % 4 == 2) for k in range(MAX_SETS)]
    a = 3  # 17 rows, made contiguous at channels [a0, a0 + 17) for the ranged call
    assert counts[a] == 17
    rest = _interleave([0 if k == a else n for k, n in enumerate(counts)], rng)
    a0 = 100
    table_of = np.concatenate([rest[:a0], np.full(17, a), rest[a0:]])
    nch = len(table_of)
    modes = [(AM, USB, LSB, CW)[(c * 3) % 4] for c in range(nch)]
    x = msdr.synth.batch(modes, 128 * 7)
    _adversarial_rows(x, rng, low=[a0, nch - 1], full=[a0 + 16, 31])
    gr, o = _pair(msdr, orc, K, modes, table_of, tables)
    gl = _list_chain(msdr, K, modes, table_of, tables)
    chains = {"ranged": gr, "list": gl}
    for g in chains.values():
        g.set_option("variant", variant)
    slot_a = gr.get_state(a0).fir_set
    assert gl.get_state(a0).fir_set == slot_a

    def step(b0, nb, what):
        builds = {k: g.plan_build_count() for k, g in chains.items()}
        part = np.ascontiguousarray(x[:, 128 * b0:128 * (b0 + nb)])
        yo = o.run(part)[0]
        ys = {}
        for k, g in chains.items():
            ys[k] = g.update(part)
            assert family(g.last_kernel()) == want, (k, g.last_kernel())
            assert_same(ys[k], yo, f"{k} setter, {what}")
            assert g.plan_build_count() == builds[k] + 1, (k, what, "one plan per configuration")

    step(0, 2, "32 tables")
    new = _table(38, rng, wrap=True)
    for b0, tab, what in ((2, new, "new table in the freed slot"), (3, tables[a], "the old table back"), (4, new, "the new one again")):
        gr.fir_init(*tab, a0, 17)
        gl.fir_init_list(*tab, np.arange(a0, a0 + 17)[::-1])
        assert o.fir_init(a0, 17, *tab) == 0
        for g in chains.values():
            assert g.get_state(a0).fir_set == slot_a and g.fir_taps(a0 + 16) == len(tab[0])
        step(b0, 1, what)
    for c in range(nch):
        assert bytes(gr.get_state(c)) == bytes(gl.get_state(c)), f"channel {c}: ranged and list chains differ in state"
    # spread users, listed twice in places: only the list call can move them all in one call
    b = int(table_of[np.flatnonzero(table_of != a)[0]])
    users = np.flatnonzero(table_of == b)
    assert len(users) > 1 and users[-1] - users[0] + 1 > len(users)
    slot_b = gl.get_state(int(users[0])).fir_set
    tab_b = _table(100, rng)
    builds = gl.plan_build_count()
    gl.fir_init_list(*tab_b, np.concatenate([users, users[:2]]))
    for c in users:
        assert o.fir_init(int(c), 1, *tab_b) == 0
    assert gl.get_state(int(users[-1])).fir_set == slot_b
    part = np.ascontiguousarray(x[:, 128 * 5:])
    assert_same(gl.update(part), o.run(part)[0], "list setter, spread users")
    assert family(gl.last_kernel()) == want and gl.plan_build_count() == builds + 1


# ---- 4. channel ranges that start anywhere, and the plan cache ---------------------------------------------------------------

RANGE_CUTS = [  # (blocks, ranges in the order they are updated): every cut covers the chain once
    (3, [(0, 1), (1, 31), (32, 97), (129, 300), (429, 271)]),
    (1, [(429, 271), (248, 181), (245, 3), (45, 200), (0, 45)]),
    (2, [(0, 699), (699, 1)]),
]
RANGE_CHANNELS = 700


def _range_layout(msdr, seed):
    """700 channels over 10 interleaved tables of 4 ... 102 taps (two wrapping), mixed modes."""
    rng = np.random.default_rng(seed)
    counts = [1, 15, 16, 17, 31, 33, 127, 128, 129, 203]
    assert sum(counts) == RANGE_CHANNELS
    tables = [_table((4, 6, 30, 38, 86, 100, 102, 102, 86, 30)[k], rng, wrap=k in (2, 7)) for k in range(len(counts))]
    table_of = _interleave(counts, rng)
    return msdr.synth.mixed_modes(RANGE_CHANNELS), table_of, tables, rng


def _update_ranges(g, upd, d_in, d_out, col, nb, ranges, want, fused=None):
    """One update of `nb` blocks from column `col`, range by range; fused: ADC codes, with the front end fused or composed."""
    for c0, n in ranges:
        upd(c0, n, d_in[c0:, col:].data_ptr(), d_out[c0:, col:].data_ptr(), nb, d_in.stride(0))
        kernel = g.last_kernel()
        assert family(kernel) == want, (c0, n, kernel)
        if fused is not None:
            assert ("front end fused into the converters" in kernel) == fused, (c0, n, kernel)
            assert kernel.startswith("msdr::fe::frontend_kernel") != fused, (c0, n, kernel)


RANGE_CASES = [(0, "v6"), (16384, "v4 one set"), (4096, "v5"), (4096 | 32768, "v5l")]


@pytest.mark.parametrize("variant,want", RANGE_CASES)
def test_unaligned_ranges_and_plan_eviction(msdr, orc, K, variant, want):
    """update_range_device over ranges that start and end anywhere (1 channel, 31, 97 from channel 32, 300 from 129 ...), cut
    differently in every update and taken in any order, each with its own row plan; then the chain cut into more ranges than the plan
    cache holds, twice round, so that plans are evicted and rebuilt.  The whole chain against the oracle fed the same blocks."""
    import torch
    modes, table_of, tables, rng = _range_layout(msdr, 41)
    nb_all = sum(nb for nb, _ in RANGE_CUTS) + 3
    x = msdr.synth.batch(modes, 128 * nb_all)
    _adversarial_rows(x, rng, low=[0, 31, 429], full=[32, 128, 699])
    g, o = _pair(msdr, orc, K, modes, table_of, tables)
    g.set_option("variant", variant)
    d_in = torch.from_numpy(x).cuda()
    d_out = torch.zeros_like(d_in)
    s = torch.cuda.Stream()
    g.set_stream(s.cuda_stream)
    torch.cuda.synchronize()  # the copies above ran on torch's stream
    col = 0
    for nb, ranges in RANGE_CUTS:
        assert sum(n for _, n in ranges) == RANGE_CHANNELS
        _update_ranges(g, g.update_range_device, d_in, d_out, col, nb, ranges, want)
        col += 128 * nb
    g.synchronize()
    yo = o.run(np.ascontiguousarray(x[:, :col]))[0]
    assert_same(d_out[:, :col].cpu().numpy(), yo, f"variant {variant}, unaligned ranges")
    # more ranges than the cache holds (64 plans), in the same order twice
    cuts = np.sort(rng.choice(np.arange(1, RANGE_CHANNELS), 71, replace=False))
    ranges = [(int(a), int(b - a)) for a, b in zip(np.r_[0, cuts], np.r_[cuts, RANGE_CHANNELS])]
    built = []
    for nb in (1, 2):
        b0 = g.plan_build_count()
        _update_ranges(g, g.update_range_device, d_in, d_out, col, nb, ranges, want)
        built.append(g.plan_build_count() - b0)
        col += 128 * nb
    g.synchronize()
    assert built[0] >= len(ranges) - 64 and built[1] > 0, f"plans built per round {built}: nothing was evicted"
    yo = o.run(np.ascontiguousarray(x[:, 128 * (nb_all - 3):]))[0]
    assert_same(d_out[:, 128 * (nb_all - 3):].cpu().numpy(), yo, f"variant {variant}, {len(ranges)} ranges, evicted plans")


@pytest.mark.parametrize("path", ["fused", "composed"])
def test_unaligned_ranges_adc(msdr, orc, forc, K, path):
    """update_adc_range_device over the same unaligned cuts on a front-end chain: the front end fused into the row-block kernel's
    converters (variant 4096), or the front-end kernel over the range and then the time-folded kernel.  Against the front-end oracle
    followed by the chain oracle."""
    import torch
    modes, table_of, tables, rng = _range_layout(msdr, 42)
    nb_all = sum(nb for nb, _ in RANGE_CUTS)
    codes = fl.adc_stream(RANGE_CHANNELS, 128 * nb_all, seed=43)
    codes[31] = 0
    codes[128, ::2] = 65535
    codes[128, 1::2] = 0
    g, o = _pair(msdr, orc, K, modes, table_of, tables)
    g.set_option("variant", 4096 if path == "fused" else 0)
    g.enable_frontend()
    fo = forc.frontend(RANGE_CHANNELS)
    for ch0, nch, first in ((5, 40, 2048), (650, 50, 1000)):
        g.frontend_preset(first, ch0, nch)
        for c in range(ch0, ch0 + nch):
            fo.preset(c, first)
    d_in = torch.from_numpy(codes.view(np.int16)).cuda()
    d_out = torch.zeros_like(d_in)
    torch.cuda.synchronize()  # the copies above ran on torch's stream
    col = 0
    for nb, ranges in RANGE_CUTS:
        _update_ranges(g, g.update_adc_range_device, d_in, d_out, col, nb, ranges, "v5" if path == "fused" else "v6",
                       fused=path == "fused")
        col += 128 * nb
    g.synchronize()
    yo = o.run(fo.run(codes))[0]
    assert_same(d_out.cpu().numpy(), yo, f"{path}, unaligned ranges of ADC codes")
