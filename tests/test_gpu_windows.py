"""Every fused kernel at every FIR window it can run.  A kernel sizes its shared memory, sub-tiles and halo from the window of
roundup32(32 + KP - 1) words (KP = roundup4(T / 2 + 1) for the longest table T of the update) and from the history of
roundup8(2 KP - 2) samples for the chain's max_taps; which kernels fit depends on the window.  Each (kernel, shape, window) pairing
that update_range can pick runs here: tables of every padding class KP - T / 2 in {1, 2, 3, 4}, both edges of each window, shorter
tables of lower windows interleaved with them, a wrapping table, adversarial inputs, updates shorter than, equal to and longer than
the history, and the same windows through the ADC-code and channel-list entry points.  Every channel is compared byte for byte with
the CPU oracle, and every update asserts the kernel and v4 shape that the window-aware copy of the selection rule (predict) names."""
import ctypes as C
from collections import Counter

import numpy as np
import pytest

import frontend_lib as fl
import oracle_lib as ol
from chain_helpers import assert_same
from conftest import wrap_coeffs

pytestmark = pytest.mark.gpu
AM, USB, LSB, CW = ol.MODE_AM, ol.MODE_USB, ol.MODE_LSB, ol.MODE_CW
FORCE_V5, NO_V5, NO_V6, V5L_ANY, FORCE_V6 = 4096, 8192, 16384, 32768, 65536
V4_HELPER, V4_CLASSIC, V4_ONE_SET, V4_POST = 128, 256, 512, 2048  # v4 only, one chain set per SM, this shape where it fits
V4_STUDY = V4_HELPER | V4_CLASSIC | V4_ONE_SET | V4_POST
# v4 shapes by their names in msdr_chain_last_kernel (kV4ShapeNames, csrc/msdr_capi.cu)
POST, CLASSIC, HELPER, DUAL = "post-warp shape", "classic shape", "feed-forward helper-warp shape", "two chain sets per SM"
FUSED = "front end fused into the converters"


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def forc():
    return fl.Orc()


def kp_of_taps(T):
    return (T // 2 + 1 + 3) & ~3


def window_words(T):
    return (32 + kp_of_taps(T) - 1 + 31) & ~31


def history(max_taps):
    return (2 * kp_of_taps(max_taps) - 2 + 7) & ~7


# ---- the windows and what fits them -----------------------------------------------------------------------------------------
# Which kernels fit each window (in words): what chain_v6_config, chain_v4_config (its rings: post-warp, classic, helper-warp, two
# sets) and chain_v5_config in both forms (csrc/msdr_chain_v*.cu) return for that window with the B200's opt-in shared memory of
# 232 448 bytes per block, evaluated on the host from the same sources.  The cases below check on the device that update_range picks
# accordingly: a change of a shared-memory budget that moves a fit fails them, and this table changes with it.
# taps: the tables of a chain in that window, the upper edge (the longest) first: both edges of the window, every padding class
# T mod 8 in {0, 2, 4, 6} (KP - T / 2 = 4, 3, 2, 1), tables of lower windows.  wrap: the table whose taps wrap the accumulator.
WINDOWS = {
    64: dict(taps=(62, 4, 8, 34, 44), wrap=44, v6=True, v4=(POST, CLASSIC, HELPER, DUAL), v5=True, v5l=True),
    96: dict(taps=(126, 64, 66, 100, 88, 30, 62), wrap=88, v6=True, v4=(POST, CLASSIC, HELPER, DUAL), v5=True, v5l=True),
    128: dict(taps=(190, 128, 130, 172, 150, 38, 100, 126), wrap=150, v6=True, v4=(POST, CLASSIC), v5=True, v5l=True),
    160: dict(taps=(254, 192, 194, 220, 250, 200, 6, 86, 150, 190), wrap=250, v6=True, v4=(CLASSIC, DUAL), v5=False, v5l=True),
    192: dict(taps=(256, 4, 102, 190, 254), wrap=256, v6=False, v4=(CLASSIC,), v5=False, v5l=True),
}
EDGES = {64: (4, 62), 96: (64, 126), 128: (128, 190), 160: (192, 254), 192: (256, 256)}


def test_window_table_is_consistent():
    """Each window's tables land in it or below, its longest table is its upper edge, both edges are present and are the edges
    (two taps fewer is the window below), and every padding class appears in each window short of 256 taps.  (Host only, but kept
    with the GPU cases it describes.)"""
    for W, w in WINDOWS.items():
        lo, hi = EDGES[W]
        assert window_words(w["taps"][0]) == W and w["taps"][0] == max(w["taps"]) == hi
        assert max(window_words(T) for T in w["taps"]) == W and lo in w["taps"]
        assert window_words(lo) == W and (W == 64 or window_words(lo - 2) == W - 32) and (W == 192 or window_words(hi + 2) == W + 32)
        if W < 192:
            assert {kp_of_taps(T) - T // 2 for T in w["taps"] if window_words(T) == W} == {1, 2, 3, 4}, W
    assert history(62) == 64 and history(126) == 128 and history(190) == 192 and history(254) == 256 and history(256) == 264


def predict(nch, n_gb, sms, W, variant=0, spare=0):
    """update_range's choice for a range of nch channels whose longest table has the window W (choose_kernel, csrc/msdr_capi.cu):
    from min(12288, 64 SMs + 1) channels (or with variant 4096) the row-block kernel, its half-tile form v5l where v5 does not fit
    (160 and 192 words) or variant 32768 asks for it; else the time-folded kernel v6 while the window fits it (not 192 words), the
    range has at most 8192 channels and its group blocks fit the SMs not kept spare; else the chain kernel v4: two chain sets per SM
    when there are more channel groups than SMs and the window leaves room for the second set (64, 96 and 160 words), otherwise one
    set, in waves of one group per SM, in the helper-warp shape where it fits, else the post-warp shape, else the classic shape.
    The v4 study bits (128, 256, 512, 2048) run v4 with one chain set per SM, in the shape they name where the window fits it.
    Returns (family, v4 shape or None)."""
    w = WINDOWS[W]
    study = variant & V4_STUDY
    if (variant & FORCE_V5 or nch >= min(12288, 64 * sms + 1)) and not variant & NO_V5 and not study and (w["v5"] or w["v5l"]):
        return ("v5l" if not w["v5"] or variant & V5L_ANY else "v5"), None
    want_v6 = not variant & NO_V6 and not study and (nch <= 8192 or variant & FORCE_V6)
    if want_v6 and w["v6"] and (variant & FORCE_V6 or n_gb <= max(1, sms - spare)):
        return "v6", None
    if -(-nch // 32) > sms and not study and DUAL in w["v4"]:
        return "v4", DUAL
    shape = next(s for s in (HELPER, POST, CLASSIC) if s in w["v4"])
    for bit, s in ((V4_POST, POST), (V4_CLASSIC, CLASSIC), (V4_HELPER, HELPER)):
        if variant & bit and s in w["v4"]:
            shape = s
    return "v4", shape


def predict_list(n, n_gb, sms, W, variant=0):
    """The list rule of choose_kernel: the time-folded kernel when the window fits it and the list's channel groups and group
    blocks fit the SMs, else the row-block kernel, v5l where v5 does not fit or with variant 32768."""
    w = WINDOWS[W]
    want_v6 = not variant & (NO_V6 | FORCE_V5) and (variant & FORCE_V6 or -(-n // 32) <= sms)
    if want_v6 and w["v6"] and (variant & FORCE_V6 or n_gb <= sms):
        return "v6", None
    return ("v5l" if not w["v5"] or variant & V5L_ANY else "v5"), None


def kernel_of(last):
    """(family, v4 shape or None) named by msdr_chain_last_kernel."""
    for f in ("v6", "v5l", "v5", "v4"):
        if f"msdr::{f}::chain_kernel" in last:
            if f != "v4":
                return f, None
            shape = [s for s in (POST, CLASSIC, HELPER, DUAL) if f"; {s})" in last]
            assert len(shape) == 1, last
            return f, shape[0]
    raise AssertionError(f"unknown kernel: {last}")


def v6_group_blocks(table_of):
    """Group blocks of the time-folded kernel's plan: each table's rows in 16-row halves (the last one padded), two halves a block."""
    return -(-sum(-(-n // 16) for n in Counter(np.asarray(table_of).tolist()).values()) // 2)


# ---- chains ----------------------------------------------------------------------------------------------------------------

class Layout:
    """The tables of window W on n channels: every table twice within the first 2 x (number of tables) channels, so that every
    prefix a case takes holds all of them, in the same slots; the rest random, no table contiguous, so that row blocks and half
    blocks mix tables.  Mixed modes (AM, USB, LSB, CW by channel mod 4), the sketch's live biquads, and object 0 as a 4-stage
    cascade on the second 32-channel group."""
    CASCADE = (32, 32)

    def __init__(self, W, n):
        rng = np.random.default_rng(W * 100003 + n)
        w = WINDOWS[W]
        self.W, self.n, self.taps = W, n, list(w["taps"])
        self.tables = []
        for T in self.taps:
            if T == w["wrap"]:
                self.tables.append((wrap_coeffs(T, rng), wrap_coeffs(T, rng)))
            else:
                cI = rng.integers(-700, 700, T).astype(np.int16)
                self.tables.append((cI, cI[::-1].copy()))
        nt = len(self.taps)
        self.table_of = rng.integers(0, nt, n)
        self.table_of[:2 * nt] = rng.permutation(np.repeat(np.arange(nt), 2))
        for k in range(nt):
            where = np.flatnonzero(self.table_of == k)
            assert where[-1] - where[0] + 1 > len(where), f"table {k} came out contiguous"
        self.modes = np.array([(AM, USB, LSB, CW)[c % 4] for c in range(n)], np.int32)

    def window(self, chans):
        return max(window_words(self.taps[t]) for t in self.table_of[chans])

    def gpu(self, msdr, K, n, max_taps, variant):
        """GPU chain of the first n channels."""
        g = msdr.ReceiveChain(n, max_taps=max_taps)
        for m in (AM, USB, LSB, CW):
            g.set_mode_list(m, np.flatnonzero(self.modes[:n] == m))
        for t, tab in enumerate(self.tables):
            g.fir_init_list(*tab, np.flatnonzero(self.table_of[:n] == t))
        for obj, key in ((0, "biquad1_lowpass_coef"), (1, "biquad2_notch_coef")):
            g.biquad_set_coefficients(obj, 0, K[key])
        c0, nc = self.CASCADE
        for stage in (1, 2, 3):
            g.biquad_set_coefficients(0, stage, K["biquad1_lowpass_coef"], c0, nc)
        g.set_option("variant", variant)
        return g

    def oracle(self, orc, K):
        o = orc.chain(self.n)
        for c in range(self.n):
            o.set_mode(c, 1, int(self.modes[c]))
            assert o.fir_init(c, 1, *self.tables[self.table_of[c]]) == 0
        for obj, key in ((0, "biquad1_lowpass_coef"), (1, "biquad2_notch_coef")):
            o.biquad_set_coefficients(obj, 0, self.n, 0, K[key])
        c0, nc = self.CASCADE
        for stage in (1, 2, 3):
            o.biquad_set_coefficients(0, c0, nc, stage, K["biquad1_lowpass_coef"])
        return o


def _biquads_equal(orc, g, o, chans, what):
    """The GPU chain's biquad words equal the oracle's AudioFilterBiquad::definition."""
    d = np.zeros(32, np.int32)
    for c in chans:
        st = g.get_state(int(c))
        for obj in (0, 1):
            orc.lib.orc_chain_get_biquad_definition(C.c_void_p(o.h), int(c), obj, d.ctypes.data_as(C.c_void_p))
            assert list(st.biquad_definition[obj]) == list(d), (what, c, obj)


# ---- 1. every kernel and shape at every window, through update() --------------------------------------------------------------
# Two input groups.  The small cases take prefixes of 300 channels in updates of 1, 2, 1, 3 and 16 blocks: L < H, L == H (2 blocks
# at 250 ... 254 taps when max_taps is 254, 1 block at 126 taps), L > H and a long update.  The large cases take prefixes of
# min(12288, 64 SMs + 1) channels in 1, 2 and 5 blocks.  The cases of a group share channels, tables and input, so their final
# channel states must agree.
GROUPS = {"small": [1, 2, 1, 3, 16], "large": [1, 2, 5]}
CASES = {  # name: (group, channels from the SM count, variant)
    "few": ("small", lambda s: 70, 0),
    "v4_one_set": ("small", lambda s: 200, NO_V6),
    "v4_post": ("small", lambda s: 200, V4_POST),
    "v4_classic": ("small", lambda s: 200, V4_CLASSIC),
    "wide": ("large", lambda s: 32 * s + 1, 0),
    "many": ("large", lambda s: min(12288, 64 * s + 1), 0),
    "v5_forced": ("small", lambda s: 300, FORCE_V5),
    "v5l_forced": ("small", lambda s: 300, FORCE_V5 | V5L_ANY),
}
EXPECTED = {  # case: kernel at 64, 96, 128, 160, 192 words (the coverage this file promises; predict must agree)
    "few": [("v6", None)] * 4 + [("v4", CLASSIC)],
    "v4_one_set": [("v4", HELPER), ("v4", HELPER), ("v4", POST), ("v4", CLASSIC), ("v4", CLASSIC)],
    "v4_post": [("v4", POST)] * 3 + [("v4", CLASSIC)] * 2,
    "v4_classic": [("v4", CLASSIC)] * 5,
    "wide": [("v4", DUAL), ("v4", DUAL), ("v4", POST), ("v4", DUAL), ("v4", CLASSIC)],  # W128, W192: one set, two waves
    "many": [("v5", None)] * 3 + [("v5l", None)] * 2,
    "v5_forced": [("v5", None)] * 3 + [("v5l", None)] * 2,
    "v5l_forced": [("v5l", None)] * 5,
}
WINDOW_MAX_TAPS = [(W, mt) for W, w in WINDOWS.items() for mt in sorted({max(w["taps"]), 256})]
WMT_IDS = [f"W{W}-max{mt}" for W, mt in WINDOW_MAX_TAPS]

_CACHE = {}  # one module run: inputs, oracle runs and first final states, shared by the cases of a window and group


def _cached(key, make):
    if key not in _CACHE:
        _CACHE[key] = make()
    return _CACHE[key]


def _group_size(group, sms):
    return 300 if group == "small" else min(12288, 64 * sms + 1)


def _group_input(msdr, group, sms):
    """IF samples of a group: the synthetic streams; all -32768 (the fs/4 negation corner) or full-scale noise on rows at the edges
    of 32-channel groups and 128-row blocks and on the cases' last channels."""
    def make():
        n = _group_size(group, sms)
        rng = np.random.default_rng(n)
        x = msdr.synth.batch([(AM, USB, LSB, CW)[c % 4] for c in range(n)], 128 * sum(GROUPS[group]))
        ends = sorted({f(sms) - 1 for g, f, _ in CASES.values() if g == group})
        for c in [1, 31, 128] + ends[::2]:
            x[c] = -32768
        for c in [32, 127, 255] + ends[1::2]:
            x[c] = rng.integers(-32768, 32768, x.shape[1], dtype=np.int16)
        return x
    return _cached(("input", group), make)


def _group_oracle(msdr, orc, K, W, group, sms):
    """(layout, oracle chain after the whole input, its output) for a window and group.  Channels are independent, so each case
    compares its prefix of channels with this one run."""
    def make():
        lay = Layout(W, _group_size(group, sms))
        o = lay.oracle(orc, K)
        return lay, o, o.run(_group_input(msdr, group, sms))[0]
    return _cached(("oracle", W, group), make)


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("W,max_taps", WINDOW_MAX_TAPS, ids=WMT_IDS)
def test_every_kernel_at_every_window(msdr, orc, K, sms, W, max_taps, case):
    """One case of the table above at one window and history: its kernel and v4 shape asserted after every update, every channel
    against the oracle, the final state of every channel equal to that of the other cases of the window fed the same input, the
    FIR history the last taps - 1 input samples, and the biquad words of a few channels (the 4-stage cascade among them) the
    oracle's."""
    group, size, variant = CASES[case]
    nch = size(sms)
    lay, o, yo = _group_oracle(msdr, orc, K, W, group, sms)
    x = _group_input(msdr, group, sms)[:nch]
    assert lay.window(np.arange(nch)) == W
    want = predict(nch, v6_group_blocks(lay.table_of[:nch]), sms, W, variant)
    assert want == EXPECTED[case][list(WINDOWS).index(W)], (case, W, want)
    g = lay.gpu(msdr, K, nch, max_taps, variant)
    H = history(max_taps)
    yg, b0 = [], 0
    for nb in GROUPS[group]:
        yg.append(g.update(np.ascontiguousarray(x[:, 128 * b0:128 * (b0 + nb)])))
        assert kernel_of(g.last_kernel()) == want, (case, W, max_taps, 128 * nb, H, g.last_kernel())
        b0 += nb
    what = f"{case} at {W} words, max_taps {max_taps} (H {H}): {nch} channels, {want}"
    assert_same(np.concatenate(yg, axis=1), yo[:nch], what)
    seen = _cached(("states", W, group), dict)  # channel: (state, the case that left it)
    for c in range(nch):
        st = bytes(g.get_state(c))
        if c in seen:
            assert st == seen[c][0], f"{what}: channel {c} ends in another state than after {seen[c][1]}"
        else:
            seen[c] = (st, f"{case}, max_taps {max_taps}")
    for c in sorted({0, 31, 32, 63, 128, nch - 1} & set(range(nch))):
        st = g.get_state(c)
        T = lay.taps[lay.table_of[c]]
        assert st.num_taps == T and list(st.fir_history[:T - 1]) == list(x[c, -(T - 1):]), (what, c)
    _biquads_equal(orc, g, o, (0, 32, 45, 63, 64, nch - 1), what)
    g.close()


# ---- 2. ADC codes: the front end fused into the row-block converters, at every window ------------------------------------------

def _adc_codes():
    def make():
        codes = fl.adc_stream(300, 128 * sum(GROUPS["small"]), seed=61)
        codes[31] = 0
        codes[128, ::2] = 65535
        codes[128, 1::2] = 0
        codes[255] = 65535
        return codes
    return _cached(("adc",), make)


PRESETS = ((5, 40, 2048), (250, 30, 1000))  # (first channel, channels, first reading)


def _adc_oracle(orc, forc, K, W):
    def make():
        lay = Layout(W, 300)
        fo = forc.frontend(300)
        for ch0, n, first in PRESETS:
            for c in range(ch0, ch0 + n):
                fo.preset(c, first)
        xo = fo.run(_adc_codes())
        return lay, lay.oracle(orc, K).run(xo)[0], xo, fo
    return _cached(("adc oracle", W), make)


@pytest.mark.parametrize("variant", [FORCE_V5, FORCE_V5 | V5L_ANY])
@pytest.mark.parametrize("W,max_taps", WINDOW_MAX_TAPS, ids=WMT_IDS)
def test_adc_codes_fused_front_end_every_window(msdr, orc, forc, K, sms, W, max_taps, variant):
    """update_adc_range_device on 300 channels with the front end fused into the converters of v5 or v5l (which start conditioning
    codes at tile unit window / 32 - 1), AGC on, some channels preset, codes at both rails; updates of 1, 2, 1, 3 and 16 blocks.
    Against the front-end oracle followed by the chain oracle, with the front-end state and FIR history of a few channels."""
    import torch
    lay, yo, xo, fo = _adc_oracle(orc, forc, K, W)
    codes = _adc_codes()
    want = predict(300, 0, sms, W, variant)
    g = lay.gpu(msdr, K, 300, max_taps, variant)
    g.enable_frontend()
    for ch0, n, first in PRESETS:
        g.frontend_preset(first, ch0, n)
    d_in = torch.from_numpy(codes.view(np.int16)).cuda()
    d_out = torch.zeros_like(d_in)
    torch.cuda.synchronize()  # the copies above ran on torch's stream, the chain has its own
    col = 0
    for nb in GROUPS["small"]:
        g.update_adc_range_device(0, 300, d_in[:, col:].data_ptr(), d_out[:, col:].data_ptr(), nb, d_in.stride(0))
        last = g.last_kernel()
        assert kernel_of(last) == want and FUSED in last and not last.startswith("msdr::fe::"), (W, max_taps, nb, last)
        col += 128 * nb
    g.synchronize()
    what = f"ADC codes at {W} words, max_taps {max_taps}, variant {variant}: {want}"
    assert_same(d_out.cpu().numpy(), yo, what)
    for c in (0, 5, 44, 127, 128, 255, 299):
        gs, os_ = g.get_frontend_state(c), fo.state(c)
        assert (gs.hpf_x1, gs.hpf_y1, gs.multiplier, gs.agc_idx) == (os_["hpf_x1"], os_["hpf_y1"], os_["multiplier"], os_["agc_idx"]), (what, c)
        assert np.float32(gs.agc_val).view(np.uint32) == os_["agc_val"].view(np.uint32), (what, c)
        T = lay.taps[lay.table_of[c]]
        assert list(g.get_state(c).fir_history[:T - 1]) == list(xo[c, -(T - 1):]), (what, c)
    g.close()


# ---- 3. channel lists at every window ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("variant", [0, FORCE_V5, FORCE_V5 | V5L_ANY])
@pytest.mark.parametrize("W,max_taps", WINDOW_MAX_TAPS, ids=WMT_IDS)
def test_channel_lists_every_window(msdr, orc, K, sms, W, max_taps, variant):
    """update_list_device on random permuted subsets of a 300-channel chain (and once all of it, permuted) in updates of 1, 2, 1, 3
    and 5 blocks, on the kernel the list rule picks for the subset's own window; each channel against the oracle fed exactly the
    samples it received."""
    import torch
    lay = Layout(W, 300)
    rng = np.random.default_rng(W + max_taps + variant)
    steps = [1, 2, 1, 3, 5]
    x = _group_input(msdr, "small", sms)[:, :128 * sum(steps)]
    g = lay.gpu(msdr, K, 300, max_taps, variant)
    pos = np.zeros(300, np.int64)
    got = [[] for _ in range(300)]
    for i, nb in enumerate(steps):
        L = 128 * nb
        chans = rng.permutation(300)[:300 if i == 3 else int(rng.integers(60, 300))]
        rows = np.stack([x[c, pos[c]:pos[c] + L] for c in chans])
        d_in = torch.from_numpy(rows).cuda()
        d_out = torch.zeros_like(d_in)
        torch.cuda.synchronize()
        g.update_list_device(chans, d_in.data_ptr(), d_out.data_ptr(), nb, d_in.stride(0))
        g.synchronize()
        want = predict_list(len(chans), v6_group_blocks(lay.table_of[chans]), sms, lay.window(chans), variant)
        assert kernel_of(g.last_kernel()) == want and g.last_kernel().endswith("; channel list"), (W, variant, g.last_kernel())
        y = d_out.cpu().numpy()
        for r, c in enumerate(chans):
            got[c].append(y[r])
            pos[c] += L
    xo = np.zeros_like(x)
    for c in range(300):
        xo[c, :pos[c]] = x[c, :pos[c]]
    yo = lay.oracle(orc, K).run(xo)[0]
    for c in range(300):
        if pos[c]:
            assert_same(np.concatenate(got[c])[None], yo[c:c + 1, :pos[c]], f"list at {W} words, max_taps {max_taps}, variant "
                        f"{variant}: channel {c} after {pos[c] // 128} blocks")
    g.close()
