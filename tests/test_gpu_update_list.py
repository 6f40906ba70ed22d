"""Channel-list updates (msdr_chain_update_list_device / msdr_chain_update_list): any set of a chain's channels, in any order, through
the fused kernels in one call.  Every comparison is byte for byte on every channel unless a case says otherwise: against the CPU
oracle fed exactly the samples each channel received, and against twin chains that took the same channels as range updates."""
from collections import Counter

import numpy as np
import pytest

import oracle_lib as ol
from chain_helpers import assert_same, tables_for

pytestmark = pytest.mark.gpu
AM, USB, LSB, CW, SYNCAM = ol.MODE_AM, ol.MODE_USB, ol.MODE_LSB, ol.MODE_CW, ol.MODE_SYNCAM
FORCE_V5, NO_V6, V5L_ANY, FORCE_V6 = 4096, 16384, 32768, 65536


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def family(kernel):
    assert kernel.endswith("; channel list"), kernel
    for f in ("v6", "v5l", "v5"):
        if f"::{f}::" in kernel or kernel.startswith(f"msdr::{f}::"):
            return f
    raise AssertionError(f"a list ran on {kernel}")


def predict(lay, chans, sms, variant=0, spare=0):
    """The list selection rule of choose_kernel: the time-folded kernel while its group blocks (each table's rows in 16-row halves,
    two halves a block) fit the SMs not kept spare and the window fits it (up to 102 taps here), else the row-block kernel, its
    half-tile form for the 256-tap window.  Variant bits 4096, 16384, 32768 and 65536 apply."""
    n, v6_sms = len(chans), max(1, sms - spare)
    long_window = lay.taps[chans].max() > 200
    want_v6 = not variant & (NO_V6 | FORCE_V5) and (variant & FORCE_V6 or -(-n // 32) <= v6_sms)
    n_gb = -(-sum(-(-k // 16) for k in Counter(lay.table_of[chans].tolist()).values()) // 2)
    if want_v6 and not long_window and (variant & FORCE_V6 or n_gb <= v6_sms):
        return "v6"
    return "v5l" if long_window or variant & V5L_ANY else "v5"


# ---- chains ----------------------------------------------------------------------------------------------------------------

def _tables(rng, long_window):
    """four tables, one with wrapping taps (sum |c| >> 65536), and a 256-tap one for the long window"""
    from conftest import wrap_coeffs
    tabs = [tables_for_taps(38, rng), (wrap_coeffs(86, rng), wrap_coeffs(86, rng)), tables_for_taps(102, rng), tables_for_taps(30, rng)]
    if long_window:
        tabs[2] = tables_for_taps(256, rng)
    return tabs


def tables_for_taps(T, rng):
    cI = rng.integers(-700, 700, T).astype(np.int16)
    return cI, cI[::-1].copy()


class Layout:
    """Modes, tables, ANR switches and biquad cascades of a chain, applied alike to GPU chains and an oracle chain."""

    def __init__(self, K, C, seed, long_window=False, modes=None, anr=()):
        rng = np.random.default_rng(seed)
        self.K, self.C, self.rng = K, C, rng
        self.modes = np.array(modes if modes is not None else rng.choice([AM, USB, LSB, CW], C), np.int32)
        self.tables = _tables(rng, long_window)
        self.table_of = rng.integers(0, len(self.tables), C)
        self.taps = np.array([len(self.tables[t][0]) for t in self.table_of])
        self.anr = dict(anr)  # channel -> 1 (notch) / 2 (noise reduction)
        c0 = int(rng.integers(0, C - 40))
        self.cascade = (c0, 40)  # object 1 as a 4-stage cascade on these channels

    def gpu(self, msdr, variant=0):
        g = msdr.ReceiveChain(self.C, max_taps=256)
        self._apply(g, True)
        g.set_option("variant", variant)
        return g

    def oracle(self, orc, channels=None):
        chans = np.arange(self.C) if channels is None else np.asarray(channels)
        sub = Layout.__new__(Layout)
        sub.__dict__.update(self.__dict__)
        sub.C = len(chans)
        sub.modes, sub.table_of = self.modes[chans], self.table_of[chans]
        sub.anr = {i: self.anr[c] for i, c in enumerate(chans) if c in self.anr}
        c0, n = self.cascade
        hit = np.flatnonzero((chans >= c0) & (chans < c0 + n))
        sub.cascade = (hit, None)
        o = orc.chain(sub.C)
        sub._apply(o, False)
        return o

    def _apply(self, ch, is_gpu):
        K, C = self.K, self.C
        for m in np.unique(self.modes):
            idx = np.flatnonzero(self.modes == m)
            if is_gpu:
                ch.set_mode_list(int(m), idx)
            else:
                for c in idx:
                    ch.set_mode(int(c), 1, int(m))
        for t, tab in enumerate(self.tables):
            idx = np.flatnonzero(self.table_of == t)
            if is_gpu:
                ch.fir_init_list(*tab, idx)
            else:
                for c in idx:
                    assert ch.fir_init(int(c), 1, *tab) == 0
        for obj, key in ((0, "biquad1_lowpass_coef"), (1, "biquad2_notch_coef")):
            if is_gpu:
                ch.biquad_set_coefficients(obj, 0, K[key])
            else:
                ch.biquad_set_coefficients(obj, 0, C, 0, K[key])
        c0, n = self.cascade
        for stage in (1, 2, 3):
            coef = K["biquad1_lowpass_coef"]
            if is_gpu:
                ch.biquad_set_coefficients(0, stage, coef, c0, n)
            else:
                for c in (c0 if n is None else range(c0, c0 + n)):
                    ch.biquad_set_coefficients(0, int(c), 1, stage, coef)
        for c, v in self.anr.items():
            if is_gpu:
                ch.set_anr(v, int(c), 1)
            else:
                assert ch.set_anr(int(c), 1, v) == 0


def _to_dev(a):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    torch.cuda.synchronize()  # the copy ran on torch's stream, the chain has its own
    return t


def _list_update(g, chans, rows):
    """rows [len(chans), L] through update_list_device -> outputs (host)"""
    import torch
    d_in = _to_dev(rows)
    d_out = torch.zeros_like(d_in)
    g.update_list_device(chans, d_in.data_ptr(), d_out.data_ptr(), rows.shape[1] // 128, d_in.stride(0))
    g.synchronize()
    return d_out.cpu().numpy()


def _range_update(g, ch0, rows):
    import torch
    d_in = _to_dev(rows)
    d_out = torch.zeros_like(d_in)
    g.update_range_device(ch0, rows.shape[0], d_in.data_ptr(), d_out.data_ptr(), rows.shape[1] // 128, d_in.stride(0))
    g.synchronize()
    return d_out.cpu().numpy()


def _states(g, chans):
    return [bytes(g.get_state(int(c))) for c in chans]


# ---- 1. every kernel against the oracle ------------------------------------------------------------------------------------

KERNEL_CHAINS = {  # name: (channels, variant, long window)
    "v6": (700, 0, False),
    "v5": (700, FORCE_V5, False),
    "v5l": (600, 0, True),
}


@pytest.mark.parametrize("name", list(KERNEL_CHAINS))
def test_list_updates_every_kernel_against_oracle(msdr, orc, K, sms, name):
    """Random subsets in random order with 1, 3 and 32 blocks, mixed with range updates.  Every chain here is created with max_taps
    256, so its history is 264 samples and the 1-block updates take the short-update path (L < H) on v6, v5 and v5l alike.  Each channel's outputs against the oracle fed exactly the samples that channel received, and its final
    state against a twin chain that took each channel's samples in one range update of its own."""
    C, variant, long_window = KERNEL_CHAINS[name]
    lay = Layout(K, C, seed={"v6": 101, "v5": 102, "v5l": 103}[name], long_window=long_window)
    rng = lay.rng
    g = lay.gpu(msdr, variant)
    steps = [("list", 1), ("range", 3), ("list", 3), ("list", 32), ("list", 1), ("range", 1), ("list", 3)]
    total = sum(nb for _, nb in steps)
    x = msdr.synth.batch(list(lay.modes), 128 * total)
    x[rng.integers(0, C)] = -32768  # the fs/4 negation corner
    pos = np.zeros(C, np.int64)
    got = [[] for _ in range(C)]
    seen = set()
    for kind, nb in steps:
        L = 128 * nb
        if kind == "list":
            chans = rng.permutation(C)[:int(rng.integers(C // 4, C))]
            rows = np.stack([x[c, pos[c]:pos[c] + L] for c in chans])
            y = _list_update(g, chans, rows)
            fam = family(g.last_kernel())
            assert fam == predict(lay, chans, sms, variant), (fam, g.last_kernel())
            seen.add(fam)
        else:
            c0 = int(rng.integers(0, C // 2))
            chans = np.arange(c0, C)
            rows = np.stack([x[c, pos[c]:pos[c] + L] for c in chans])
            y = _range_update(g, c0, rows)
        for i, c in enumerate(chans):
            got[c].append(y[i])
            pos[c] += L
    assert seen == {name}
    xo = np.zeros_like(x)
    for c in range(C):
        xo[c, :pos[c]] = x[c, :pos[c]]
    yo = lay.oracle(orc).run(xo)[0]
    for c in range(C):
        if pos[c]:
            assert_same(np.concatenate(got[c])[None], yo[c:c + 1, :pos[c]], f"{name}: channel {c} after {pos[c] // 128} blocks")
    twin = lay.gpu(msdr)
    for c in range(C):
        if pos[c]:
            _range_update(twin, c, x[c:c + 1, :pos[c]])
    assert _states(g, range(C)) == _states(twin, range(C)), f"{name}: final channel states differ from range updates"


# ---- 2. channels outside the list are left alone ---------------------------------------------------------------------------

def test_unlisted_channels_untouched(msdr, K):
    lay = Layout(K, 300, seed=5)
    g = lay.gpu(msdr)
    x = msdr.synth.batch(list(lay.modes), 128 * 4)
    g.update(np.ascontiguousarray(x[:, :256]))  # every channel has history and biquad state
    chans = lay.rng.permutation(300)[:170]
    rest = np.setdiff1d(np.arange(300), chans)
    before = [bytes(g.snapshot(int(c), 1)) for c in rest]
    _list_update(g, chans, x[chans, 256:])
    assert [bytes(g.snapshot(int(c), 1)) for c in rest] == before


# ---- 3. a permutation of every channel as one list equals one range update ---------------------------------------------------

def _lane_layout(K, C, seed, long_window=False):
    rng = np.random.default_rng(seed + 1)
    modes = rng.choice([AM, USB, LSB, CW], C)
    pll = rng.choice(C, 7, replace=False)
    modes[pll] = SYNCAM
    anr_ch = rng.choice(np.setdiff1d(np.arange(C), pll), 9, replace=False)
    anr = {int(c): 1 + i % 2 for i, c in enumerate(anr_ch)}
    anr[int(pll[0])] = 1  # one SYNCAM channel with the notch as well
    lay = Layout(K, C, seed, long_window, modes=modes, anr=anr)
    lay.tables.append(tables_for(K, AM))  # the PLL channels on the sketch's AM table, where the float tolerance is stated
    lay.table_of[pll] = len(lay.tables) - 1
    lay.taps = np.array([len(lay.tables[t][0]) for t in lay.table_of])
    return lay, np.sort(pll)


@pytest.mark.parametrize("size", ["v6", "v5", "v5l"])
def test_permuted_list_equals_range(msdr, orc, K, sms, size):
    """Twin chains with SYNCAM (PLL side lane) and ANR channels: one takes a permutation of all channels as one list per update, the
    other one range update.  Outputs after un-permuting and full snapshots are byte-identical, so the side lane over a list is the
    side lane over the range bit for bit.  Non-SYNCAM channels (ANR ones too) also equal the oracle; SYNCAM ones meet its float
    tolerance."""
    C = {"v6": 32 * sms - 100, "v5": 32 * sms + 200, "v5l": 900}[size]
    lay, pll = _lane_layout(K, C, seed={"v6": 1, "v5": 2, "v5l": 3}[size], long_window=size == "v5l")
    a, b = lay.gpu(msdr), lay.gpu(msdr)
    x = msdr.synth.batch(list(lay.modes), 128 * 9)
    ya, yb = [], []
    b0 = 0
    for nb in (3, 1, 5):
        perm = lay.rng.permutation(C)
        part = x[:, 128 * b0:128 * (b0 + nb)]
        y = _list_update(a, perm, part[perm])
        assert family(a.last_kernel()) == predict(lay, perm, sms) == size
        un = np.empty_like(y)
        un[perm] = y
        ya.append(un)
        yb.append(_range_update(b, 0, part))
        b0 += nb
    ya, yb = np.concatenate(ya, axis=1), np.concatenate(yb, axis=1)
    assert_same(ya, yb, f"{size}: permuted list against range")
    assert np.array_equal(a.snapshot(), b.snapshot()), f"{size}: snapshots differ"
    yo = lay.oracle(orc).run(x)[0]
    exact = np.setdiff1d(np.arange(C), pll)
    assert_same(ya[exact], yo[exact], f"{size}: list update against the oracle")
    p, q = ya[pll].astype(np.float64), yo[pll].astype(np.float64)
    assert np.abs(p - q).max() <= 3 and np.sqrt(np.mean((p - q) ** 2)) <= 1e-4 * np.sqrt(np.mean(q ** 2)) + 0.05


# ---- 4. the plan cache -----------------------------------------------------------------------------------------------------

def test_list_plan_cache(msdr, orc, K):
    """The same list again builds no plan; the same channels in another order build one; a table change rebuilds; more distinct
    lists than the cache holds (64 plans) evict plans and the results stay right."""
    C = 400
    lay = Layout(K, C, seed=9)
    g = lay.gpu(msdr)
    o = lay.oracle(orc)
    x = msdr.synth.batch(list(lay.modes), 128 * (4 + 2 * 70))
    pos = np.zeros(C, np.int64)
    got = [[] for _ in range(C)]

    def step(ch):
        rows = np.stack([x[c, pos[c]:pos[c] + 128] for c in ch])
        y = _list_update(g, ch, rows)
        for i, c in enumerate(ch):
            got[c].append(y[i])
            pos[c] += 128

    every = lay.rng.permutation(C)
    b0 = g.plan_build_count()
    step(every)
    assert g.plan_build_count() == b0 + 1
    step(every)
    assert g.plan_build_count() == b0 + 1, "the same list rebuilt its plan"
    step(every[::-1].copy())
    assert g.plan_build_count() == b0 + 2, "another order of the same channels needs its own plan"
    # every channel has 3 blocks: the oracle follows, then both rewrite one table in place (same tap count, new contents)
    o.run(np.ascontiguousarray(x[:, :128 * 3]))
    t = int(lay.table_of[every[0]])
    cI, cQ = lay.tables[t]
    users = np.flatnonzero(lay.table_of == t)
    g.fir_set_coefficients(cQ, cI, int(users[0]), 1)  # one user of a shared table: it moves to a table of its own
    assert o.fir_set_coefficients(int(users[0]), 1, cQ, cI) == 0
    step(every)
    assert g.plan_build_count() == b0 + 3, "a table change must rebuild"
    lists = [lay.rng.permutation(C)[:int(lay.rng.integers(20, 200))] for _ in range(70)]
    built = []
    for _ in range(2):
        n0 = g.plan_build_count()
        for ch in lists:
            step(ch)
        built.append(g.plan_build_count() - n0)
    assert built[0] == 70 and built[1] > 0, f"plans built per round {built}: nothing was evicted"
    xo = np.zeros((C, int(pos.max()) - 128 * 3), np.int16)
    for c in range(C):
        xo[c, :pos[c] - 128 * 3] = x[c, 128 * 3:pos[c]]
    yo = o.run(xo)[0]
    for c in range(C):
        yg = np.concatenate(got[c])
        assert_same(yg[None, 128 * 3:], yo[c:c + 1, :pos[c] - 128 * 3], f"channel {c} after the rewrite and the evictions")


# ---- 5. refused calls change nothing ---------------------------------------------------------------------------------------

def test_refused_list_calls(msdr, K):
    import ctypes as C_
    import torch
    lay = Layout(K, 200, seed=11)
    g = lay.gpu(msdr)
    x = msdr.synth.batch(list(lay.modes), 128 * 2)
    g.update(np.ascontiguousarray(x[:, :128]))
    d_in = _to_dev(x[:, 128:])
    d_out = torch.zeros_like(d_in)
    L = g._L
    pin, pout, st = d_in.data_ptr(), d_out.data_ptr(), d_in.stride(0)
    snap = g.snapshot()
    launches = g.launch_count()

    def call(ch, n, a=pin, b=pout, nb=1, stride=st):
        arr = None if ch is None else np.ascontiguousarray(ch, np.uint32)
        return L.msdr_chain_update_list_device(g.h, msdr.capi.ptr(arr), n, C_.c_void_p(a), C_.c_void_p(b), nb, stride)

    E = msdr.capi.ERR_ARGUMENT
    cases = {
        "duplicate": ([3, 7, 3], 3, {}),
        "channel >= C": ([0, 200], 2, {}),
        "NULL list": (None, 4, {}),
        "unaligned in": ([1, 2], 2, {"a": pin + 2}),
        "unaligned out": ([1, 2], 2, {"b": pout + 2}),
        "stride below the update": ([1, 2], 2, {"nb": 2, "stride": 128}),
    }
    for what, (ch, n, kw) in cases.items():
        assert call(ch, n, **kw) == E, what
        g.synchronize()
        assert np.array_equal(g.snapshot(), snap), f"{what}: a refused call changed the chain"
    assert g.launch_count() == launches
    assert call(None, 0) == 0 and call([5], 0) == 0
    assert g.launch_count() == launches, "n == 0 launched something"
    assert L.msdr_chain_update_list(g.h, None, 3, None, None, 1, 128) == E
    # a channel without a FIR table: the range rule
    g2 = msdr.ReceiveChain(64)
    g2.set_mode(USB, 0, 64)
    g2.fir_init(*tables_for(K, USB), 0, 63)
    s2 = g2.snapshot(0, 63)
    two = np.array([1, 2], np.uint32)
    assert L.msdr_chain_update_list_device(g2.h, msdr.capi.ptr(two), 2, C_.c_void_p(pin), C_.c_void_p(pout), 1, st) == msdr.capi.ERR_NOT_INITIALISED
    g2.synchronize()
    assert np.array_equal(g2.snapshot(0, 63), s2)


# ---- 6. the host call ------------------------------------------------------------------------------------------------------

def test_host_list_call_in_chunks(msdr, K):
    """msdr_chain_update_list with host_chunk_channels forcing 4 chunks of the list equals the device call on a twin chain."""
    C = 500
    lay = Layout(K, C, seed=13)
    a, b = lay.gpu(msdr), lay.gpu(msdr)
    a.set_option("host_chunk_channels", 96)
    x = msdr.synth.batch(list(lay.modes), 128 * 6)
    for b0, nb in ((0, 2), (2, 4)):
        chans = lay.rng.permutation(C)[:350]
        rows = np.ascontiguousarray(x[chans, 128 * b0:128 * (b0 + nb)])
        ya = a.update_list(chans, rows)
        yb = _list_update(b, chans, rows)
        assert_same(ya, yb, "host list call against the device call")
    assert np.array_equal(a.snapshot(), b.snapshot())


# ---- 7. the front end ------------------------------------------------------------------------------------------------------

def test_int16_list_updates_leave_the_front_end_alone(msdr, orc, K):
    """ADC range updates interleaved with int16 list updates: the front-end state equals the front-end oracle, which advances on the
    ADC updates only."""
    import frontend_lib as fl
    import torch
    C = 300
    lay = Layout(K, C, seed=17)
    g = lay.gpu(msdr)
    g.enable_frontend()
    fo = fl.Orc().frontend(C)
    codes = fl.adc_stream(C, 128 * 6, seed=19)
    x = msdr.synth.batch(list(lay.modes), 128 * 4)
    col = 0
    for kind, nb in (("adc", 2), ("list", 2), ("adc", 1), ("list", 2), ("adc", 3)):
        if kind == "adc":
            d_in = _to_dev(codes[:, col:col + 128 * nb].view(np.int16))
            d_out = torch.zeros_like(d_in)
            g.update_adc_range_device(0, C, d_in.data_ptr(), d_out.data_ptr(), nb, d_in.stride(0))
            g.synchronize()
            fo.run(np.ascontiguousarray(codes[:, col:col + 128 * nb]))
            col += 128 * nb
        else:
            chans = lay.rng.permutation(C)[:200]
            _list_update(g, chans, x[chans, :128 * nb])
        for c in range(0, C, 7):
            gs, os_ = g.get_frontend_state(c), fo.state(c)
            what = f"front end of channel {c} after {kind}"
            assert (gs.hpf_x1, gs.hpf_y1, gs.multiplier, gs.agc_idx) == (os_["hpf_x1"], os_["hpf_y1"], os_["multiplier"], os_["agc_idx"]), what
            assert np.float32(gs.agc_val).view(np.uint32) == os_["agc_val"].view(np.uint32), what
            assert np.array_equal(np.array(gs.agc_buffer[:], np.int16), os_["agc_buffer"]), what


# ---- 8. at size --------------------------------------------------------------------------------------------------------------

def test_scattered_list_at_size(msdr, orc, K):
    """131 072 scattered channels of a 262 144-channel chain over 3 updates equal the twin chain's range updates of those channels'
    rows; 48 sampled channels against the oracle."""
    import torch
    C, n = 262144, 131072
    rng = np.random.default_rng(23)
    modes = np.array(msdr.synth.mixed_modes(C), np.int32)
    lay = Layout(K, C, seed=23, modes=modes)
    a, b = lay.gpu(msdr), lay.gpu(msdr)
    chans = np.sort(rng.choice(C, n, replace=False))
    chans = chans[rng.permutation(n)]
    nb = 32
    gen = torch.Generator(device="cuda").manual_seed(29)
    full_in = torch.randint(-32768, 32768, (C, 128 * nb), dtype=torch.int16, device="cuda", generator=gen)
    torch.cuda.synchronize()
    idx = torch.from_numpy(chans.astype(np.int64)).cuda()
    sample = rng.choice(n, 48, replace=False)
    got, xin = [], []
    for u in range(3):
        full_in.copy_(torch.randint(-32768, 32768, (C, 128 * nb), dtype=torch.int16, device="cuda", generator=gen))
        d_in = full_in[idx].contiguous()
        d_out = torch.zeros_like(d_in)
        torch.cuda.synchronize()
        a.update_list_device(chans, d_in.data_ptr(), d_out.data_ptr(), nb, d_in.stride(0))
        assert family(a.last_kernel()) == "v5"
        d_full = torch.zeros_like(full_in)
        b.update_range_device(0, C, full_in.data_ptr(), d_full.data_ptr(), nb, full_in.stride(0))  # every channel, then compare the listed
        a.synchronize(); b.synchronize()
        ya = d_out.cpu().numpy()
        yb = d_full[idx].cpu().numpy()
        assert_same(ya, yb, f"update {u}: list against range at size")
        got.append(ya[sample])
        xin.append(d_in[torch.from_numpy(sample).cuda()].cpu().numpy())
    for c in chans[sample[:8]]:
        assert bytes(a.get_state(int(c))) == bytes(b.get_state(int(c)))
    o = lay.oracle(orc, chans[sample])
    yo = o.run(np.concatenate(xin, axis=1))[0]
    assert_same(np.concatenate(got, axis=1), yo, "48 sampled channels against the oracle")
