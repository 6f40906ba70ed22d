"""Channel-list updates from raw ADC codes (msdr_chain_update_adc_list_device / msdr_chain_update_adc_list) and the list form of the
front-end preset.  The front-end kernel conditions the listed rows with the listed channels' front-end states, then the int16
list path runs on them, on whichever kernel the list rule picks.  Every comparison is byte for byte
unless a case says otherwise: against the front-end oracle of each channel feeding the chain oracle, and against twin chains that
took the same channels as ADC range updates."""
import ctypes as C

import numpy as np
import pytest

import frontend_lib as fl
from chain_helpers import assert_same, tables_for
from test_gpu_chain_adc import _chain_state_equal, _fe_state_equal
from test_gpu_update_list import FORCE_V5, USB, Layout, _lane_layout, _range_update, _to_dev, family, predict

pytestmark = pytest.mark.gpu
COMPOSED = "msdr::fe::frontend_kernel (front end), then "


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def forc():
    return fl.Orc()


def expect_path(g, lay, chans, sms, variant=0):
    """The kernel family by the list rule, behind the front-end kernel."""
    k = g.last_kernel()
    fam = family(k)
    assert fam == predict(lay, chans, sms, variant), (fam, k)
    assert k.startswith(COMPOSED) and "fused into the converters" not in k, k
    return fam


def _adc_list(g, chans, codes):
    """codes [len(chans), L] uint16 through update_adc_list_device -> outputs (host)"""
    import torch
    d_in = _to_dev(codes.view(np.int16))
    d_out = torch.zeros_like(d_in)
    g.update_adc_list_device(chans, d_in.data_ptr(), d_out.data_ptr(), codes.shape[1] // 128, d_in.stride(0))
    g.synchronize()
    return d_out.cpu().numpy()


def _adc_range(g, ch0, codes):
    import torch
    d_in = _to_dev(codes.view(np.int16))
    d_out = torch.zeros_like(d_in)
    g.update_adc_range_device(ch0, codes.shape[0], d_in.data_ptr(), d_out.data_ptr(), codes.shape[1] // 128, d_in.stride(0))
    g.synchronize()
    return d_out.cpu().numpy()


def _list16(g, chans, rows):
    import torch
    d_in = _to_dev(rows)
    d_out = torch.zeros_like(d_in)
    g.update_list_device(chans, d_in.data_ptr(), d_out.data_ptr(), rows.shape[1] // 128, d_in.stride(0))
    g.synchronize()
    return d_out.cpu().numpy()


def _codes(C_, n, seed, extreme=True):
    codes = fl.adc_stream(C_, n, seed=seed)
    if extreme:  # both rails, full 16-bit codes (the DC-block accumulator wraps), alternating rails
        rng = np.random.default_rng(seed + 1)
        codes[0::37] = 65535
        codes[1::37] = 0
        codes[2::37] = rng.integers(0, 65536, codes[2::37].shape, dtype=np.uint16)
        codes[3::37, ::2] = 65535
        codes[3::37, 1::2] = 0
    return codes


# ---- 1. against the oracles, interleaved with ADC range and int16 list / range updates ----------------------------------------

KERNEL_CHAINS = {  # name: (channels, variant, long window)
    "v6": (700, 0, False),
    "v5": (700, FORCE_V5, False),
    "v5l": (600, 0, True),
    "v5l_short_window": (600, FORCE_V5 | 32768, False),
}


@pytest.mark.parametrize("agc_on", [True, False])
@pytest.mark.parametrize("name", list(KERNEL_CHAINS))
def test_adc_list_updates_against_oracles(msdr, orc, forc, K, sms, name, agc_on):
    """Random subsets in random order with 1, 3 and 32 blocks (the chains' history is 264 samples, so 1 block is the short-update
    path), interleaved with ADC range, int16 list and int16 range updates, presets on some channels and extreme codes.  Each channel
    has a front-end oracle of its own that advances on that channel's ADC updates only; its conditioned samples (or the int16 rows)
    feed the chain oracle.  Output, FIR history, biquad words and front-end state of every channel."""
    C_, variant, long_window = KERNEL_CHAINS[name]
    lay = Layout(K, C_, seed={"v6": 201, "v5": 202, "v5l": 203, "v5l_short_window": 204}[name], long_window=long_window)
    rng = lay.rng
    g = lay.gpu(msdr, variant)
    g.enable_frontend(agc_on=agc_on)
    fos = [forc.frontend(1, on=int(agc_on)) for _ in range(C_)]
    preset = rng.choice(C_, 60, replace=False)
    g.frontend_preset_list(1900, preset)
    for c in preset:
        fos[c].preset(0, 1900)
    steps = [("adc_list", 1), ("adc_range", 3), ("adc_list", 3), ("list", 1), ("adc_list", 32), ("range", 1), ("adc_list", 1),
             ("adc_list", 3)]
    n_max = 2 * 128 * sum(nb for _, nb in steps)
    codes = _codes(C_, n_max, seed=31)
    x16 = msdr.synth.batch(list(lay.modes), n_max)
    pos = np.zeros(C_, np.int64)
    got, xin = [[] for _ in range(C_)], [[] for _ in range(C_)]
    fams = set()

    def take(kind, chans, L):
        if kind in ("adc_list", "adc_range"):
            rows = np.stack([codes[c, pos[c]:pos[c] + L] for c in chans])
            y = _adc_list(g, chans, rows) if kind == "adc_list" else _adc_range(g, int(chans[0]), rows)
            for i, c in enumerate(chans):
                xin[c].append(fos[c].run(rows[i:i + 1])[0])
        else:
            rows = np.stack([x16[c, pos[c]:pos[c] + L] for c in chans])
            y = _list16(g, chans, rows) if kind == "list" else _range_update(g, int(chans[0]), rows)
            for i, c in enumerate(chans):
                xin[c].append(rows[i])
        if kind == "adc_list":
            fams.add(expect_path(g, lay, chans, sms, variant))
        for i, c in enumerate(chans):
            got[c].append(y[i])
            pos[c] += L

    for kind, nb in steps:
        if kind.endswith("list"):
            chans = rng.permutation(C_)[:int(rng.integers(C_ // 4, C_))]
        else:
            chans = np.arange(int(rng.integers(0, C_ // 2)), C_)
        take(kind, chans, 128 * nb)
    # every channel to the same length with one ADC list per deficit, so that one oracle run covers the whole chain
    m = pos.max()
    for d in np.unique(m - pos):
        if d:
            take("adc_list", rng.permutation(np.flatnonzero(pos == m - d)), int(d))
    assert name.split("_")[0] in fams, fams  # small catch-up lists may pick another kernel: predict() checked each
    xo = np.stack([np.concatenate(xin[c]) for c in range(C_)])
    o = lay.oracle(orc)
    yo = o.run(xo)[0]
    assert_same(np.stack([np.concatenate(got[c]) for c in range(C_)]), yo, f"{name}: ADC list updates against the oracles")
    for c in range(C_):
        _fe_state_equal(g.get_frontend_state(c), fos[c].state(0), (name, c))
        _chain_state_equal(orc, g, o, c, xo, name)


# ---- 2. channels outside the list are left alone ---------------------------------------------------------------------------

@pytest.mark.parametrize("variant", [0, FORCE_V5])
def test_unlisted_channels_untouched(msdr, K, variant):
    lay = Layout(K, 300, seed=5)
    g = lay.gpu(msdr, variant)
    g.enable_frontend()
    codes = _codes(300, 128 * 4, seed=7)
    _adc_range(g, 0, np.ascontiguousarray(codes[:, :256]))  # every channel has history, biquad and front-end state
    chans = lay.rng.permutation(300)[:170]
    rest = np.setdiff1d(np.arange(300), chans)
    before = [(bytes(g.get_state(int(c))), bytes(g.get_frontend_state(int(c)))) for c in rest]
    _adc_list(g, chans, np.ascontiguousarray(codes[chans, 256:]))
    assert [(bytes(g.get_state(int(c))), bytes(g.get_frontend_state(int(c)))) for c in rest] == before


# ---- 3. a permuted list equals ADC range updates on a twin chain, side-lane channels included ---------------------------------

@pytest.mark.parametrize("size", ["v6", "v5", "v5l"])
def test_permuted_adc_list_equals_range(msdr, orc, forc, K, sms, size):
    """Twin chains with SYNCAM (PLL side lane) and ANR channels: one takes a permutation of all channels as one ADC list per update,
    the other ADC range updates.  Then a list without the side-lane channels on one, range updates of its contiguous runs on the
    other.  Outputs, snapshots and front-end states are byte-identical; non-SYNCAM channels equal the oracles, SYNCAM ones meet the
    float tolerance."""
    C_ = {"v6": 32 * sms - 100, "v5": 32 * sms + 200, "v5l": 900}[size]
    lay, pll = _lane_layout(K, C_, seed={"v6": 1, "v5": 2, "v5l": 3}[size], long_window=size == "v5l")
    lane = np.array(sorted(set(pll.tolist()) | set(lay.anr)))
    a, b = lay.gpu(msdr), lay.gpu(msdr)
    a.enable_frontend(); b.enable_frontend()
    codes = _codes(C_, 128 * 13, seed=41, extreme=False)
    ya, yb, b0 = [], [], 0
    for nb in (3, 1, 5):
        perm = lay.rng.permutation(C_)
        part = np.ascontiguousarray(codes[:, 128 * b0:128 * (b0 + nb)])
        y = _adc_list(a, perm, np.ascontiguousarray(part[perm]))
        assert expect_path(a, lay, perm, sms) == size
        un = np.empty_like(y)
        un[perm] = y
        ya.append(un)
        yb.append(_adc_range(b, 0, part))
        b0 += nb
    ya, yb = np.concatenate(ya, axis=1), np.concatenate(yb, axis=1)
    assert_same(ya, yb, f"{size}: permuted ADC list against ADC range")
    assert np.array_equal(a.snapshot(), b.snapshot()), f"{size}: snapshots differ"
    fo = forc.frontend(C_)
    yo = lay.oracle(orc).run(fo.run(np.ascontiguousarray(codes[:, :128 * b0])))[0]
    exact = np.setdiff1d(np.arange(C_), pll)
    assert_same(ya[exact], yo[exact], f"{size}: ADC list update against the oracles")
    p, q = ya[pll].astype(np.float64), yo[pll].astype(np.float64)
    assert np.abs(p - q).max() <= 3 and np.sqrt(np.mean((p - q) ** 2)) <= 1e-4 * np.sqrt(np.mean(q ** 2)) + 0.05
    # the channels off the side lane, permuted, as one list; on b the same rows as range updates of each channel
    off = lay.rng.permutation(np.setdiff1d(np.arange(C_), lane))
    part = np.ascontiguousarray(codes[off, 128 * b0:128 * (b0 + 4)])
    y = _adc_list(a, off, part)
    expect_path(a, lay, off, sms)
    order = np.argsort(off)
    yr = _adc_range_each(b, off[order], part[order])
    assert_same(y[order], yr, f"{size}: off-lane list against range updates")
    for c in range(0, C_, 13):
        assert bytes(a.get_state(c)) == bytes(b.get_state(c)) and bytes(a.get_frontend_state(c)) == bytes(b.get_frontend_state(c)), c


def _adc_range_each(g, chans, rows):
    """ascending channels: one ADC range update per contiguous run"""
    out, i = [], 0
    while i < len(chans):
        j = i + 1
        while j < len(chans) and chans[j] == chans[j - 1] + 1:
            j += 1
        out.append(_adc_range(g, int(chans[i]), np.ascontiguousarray(rows[i:j])))
        i = j
    return np.concatenate(out)


# ---- 4. refused calls change nothing ---------------------------------------------------------------------------------------

def test_refused_adc_list_calls(msdr, K):
    import torch
    lay = Layout(K, 200, seed=11)
    g = lay.gpu(msdr)
    codes = _codes(200, 128 * 2, seed=13, extreme=False)
    d_in = _to_dev(codes.view(np.int16))
    d_out = torch.zeros_like(d_in)
    L = g._L
    pin, pout, st = d_in.data_ptr(), d_out.data_ptr(), d_in.stride(0)

    def call(ch, n, a=pin, b=pout, nb=1, stride=st):
        arr = None if ch is None else np.ascontiguousarray(ch, np.uint32)
        return L.msdr_chain_update_adc_list_device(g.h, msdr.capi.ptr(arr), n, C.c_void_p(a), C.c_void_p(b), nb, stride)

    def preset(ch, n):
        arr = None if ch is None else np.ascontiguousarray(ch, np.uint32)
        return L.msdr_chain_frontend_preset_list(g.h, msdr.capi.ptr(arr), n, 1234)

    NI, E = msdr.capi.ERR_NOT_INITIALISED, msdr.capi.ERR_ARGUMENT
    launches = g.launch_count()
    assert call([1, 2], 2) == NI and preset([1, 2], 2) == NI
    assert L.msdr_chain_update_adc_list(g.h, msdr.capi.ptr(np.array([1, 2], np.uint32)), 2, None, None, 1, 128) == NI
    assert g.launch_count() == launches
    g.enable_frontend()
    _adc_range(g, 0, np.ascontiguousarray(codes[:, :128]))
    g.frontend_preset_list(2000, [4, 9, 150])
    snap, fe = g.snapshot(), [bytes(g.get_frontend_state(c)) for c in range(200)]
    launches = g.launch_count()
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
    assert preset([0, 200], 2) == E and preset(None, 3) == E
    assert L.msdr_chain_update_adc_list(g.h, None, 3, None, None, 1, 128) == E
    assert L.msdr_chain_update_adc_list(g.h, msdr.capi.ptr(np.array([5, 5], np.uint32)), 2, None, None, 1, 128) == E
    assert call(None, 0) == 0 and call([5], 0) == 0 and preset(None, 0) == 0
    g.synchronize()
    assert g.launch_count() == launches, "a refused call or n == 0 launched something"
    assert np.array_equal(g.snapshot(), snap), "a refused call changed the chain"
    assert [bytes(g.get_frontend_state(c)) for c in range(200)] == fe, "a refused call changed a front end"
    # an empty ADC list call after a launched one leaves last_kernel as that update named it (an idle bank polls with n == 0)
    _adc_list(g, [7, 3], np.ascontiguousarray(codes[[7, 3], 128:]))
    k = g.last_kernel()
    assert k.count("frontend_kernel") == 1 and k.startswith(COMPOSED), k
    n_in = np.zeros((1, 128), np.uint16)
    for _ in range(3):
        assert call(None, 0) == 0 and call([5], 1, nb=0) == 0
        assert L.msdr_chain_update_adc_list(g.h, None, 0, None, None, 1, 128) == 0
        assert L.msdr_chain_update_adc_list(g.h, msdr.capi.ptr(np.array([5], np.uint32)), 1, msdr.capi.ptr(n_in), msdr.capi.ptr(n_in), 0, 128) == 0
        assert L.msdr_chain_update_adc_range_device(g.h, 0, 0, C.c_void_p(pin), C.c_void_p(pout), 1, st) == 0
    assert g.last_kernel() == k, g.last_kernel()
    # a channel without a FIR table: the range rule
    g2 = msdr.ReceiveChain(64)
    g2.set_mode(USB, 0, 64)
    g2.fir_init(*tables_for(K, USB), 0, 63)
    g2.enable_frontend()
    s2, f2 = g2.snapshot(0, 63), bytes(g2.get_frontend_state(1))
    two = np.array([1, 2], np.uint32)
    assert L.msdr_chain_update_adc_list_device(g2.h, msdr.capi.ptr(two), 2, C.c_void_p(pin), C.c_void_p(pout), 1, st) == NI
    g2.synchronize()
    assert np.array_equal(g2.snapshot(0, 63), s2) and bytes(g2.get_frontend_state(1)) == f2


# ---- 5. the host call ------------------------------------------------------------------------------------------------------

def test_host_adc_list_call_in_chunks(msdr, K):
    """msdr_chain_update_adc_list with host_chunk_channels forcing 4 chunks of a 350-channel list equals the device call on a twin
    chain, with an int16 host list call in between."""
    C_ = 500
    lay = Layout(K, C_, seed=13)
    a, b = lay.gpu(msdr), lay.gpu(msdr)
    a.enable_frontend(); b.enable_frontend()
    a.set_option("host_chunk_channels", 96)
    codes = _codes(C_, 128 * 6, seed=17)
    x16 = msdr.synth.batch(list(lay.modes), 128 * 2)
    for b0, nb in ((0, 2), (2, 4)):
        chans = lay.rng.permutation(C_)[:350]
        rows = np.ascontiguousarray(codes[chans, 128 * b0:128 * (b0 + nb)])
        assert_same(a.update_adc_list(chans, rows), _adc_list(b, chans, rows), "host ADC list call against the device call")
        chans = lay.rng.permutation(C_)[:350]
        rows = np.ascontiguousarray(x16[chans, :128])
        assert_same(a.update_list(chans, rows), _list16(b, chans, rows), "host int16 list call against the device call")
    assert np.array_equal(a.snapshot(), b.snapshot())
    assert all(bytes(a.get_frontend_state(c)) == bytes(b.get_frontend_state(c)) for c in range(C_))


# ---- 6. the plan cache -----------------------------------------------------------------------------------------------------

def test_adc_and_int16_list_share_a_plan(msdr, K):
    lay = Layout(K, 400, seed=9)
    g = lay.gpu(msdr, FORCE_V5)
    g.enable_frontend()
    codes = _codes(400, 128 * 3, seed=19, extreme=False)
    x16 = msdr.synth.batch(list(lay.modes), 128)
    chans = lay.rng.permutation(400)[:333]
    n0 = g.plan_build_count()
    _adc_list(g, chans, np.ascontiguousarray(codes[chans, :128]))
    assert g.plan_build_count() == n0 + 1
    _adc_list(g, chans, np.ascontiguousarray(codes[chans, 128:256]))
    assert g.plan_build_count() == n0 + 1, "the same list rebuilt its plan"
    _list16(g, chans, np.ascontiguousarray(x16[chans]))
    assert g.plan_build_count() == n0 + 1, "an int16 update of the same list built another plan"
    _adc_list(g, chans, np.ascontiguousarray(codes[chans, 256:]))
    assert g.plan_build_count() == n0 + 1


# ---- 7. frontend_preset_list -----------------------------------------------------------------------------------------------

def test_frontend_preset_list_equals_range_presets(msdr, K):
    lay = Layout(K, 300, seed=21)
    a, b = lay.gpu(msdr), lay.gpu(msdr)
    a.enable_frontend(); b.enable_frontend()
    codes = _codes(300, 128 * 2, seed=23, extreme=False)
    _adc_range(a, 0, np.ascontiguousarray(codes[:, :128])); _adc_range(b, 0, np.ascontiguousarray(codes[:, :128]))
    chans = np.concatenate([[299, 0], lay.rng.permutation(np.arange(1, 299))[:75]])  # both ends: the states between stay as they were
    a.frontend_preset_list(3100, chans)
    for c in chans:
        b.frontend_preset(3100, int(c), 1)
    assert all(bytes(a.get_frontend_state(c)) == bytes(b.get_frontend_state(c)) for c in range(300))
    assert_same(_adc_range(a, 0, np.ascontiguousarray(codes[:, 128:])), _adc_range(b, 0, np.ascontiguousarray(codes[:, 128:])), "after presets")


# ---- 8. at size --------------------------------------------------------------------------------------------------------------

def test_scattered_adc_list_at_size(msdr, K):
    """131 072 scattered channels of a 262 144-channel chain over 3 ADC list updates of 32 blocks equal the twin chain's ADC range
    updates of every channel, compared on every listed channel; states of sampled channels."""
    import torch
    C_, n, nb = 262144, 131072, 32
    rng = np.random.default_rng(27)
    lay = Layout(K, C_, seed=27, modes=np.array(msdr.synth.mixed_modes(C_), np.int32))
    a, b = lay.gpu(msdr), lay.gpu(msdr)
    a.enable_frontend(); b.enable_frontend()
    chans = rng.choice(C_, n, replace=False)
    idx = torch.from_numpy(chans.astype(np.int64)).cuda()
    gen = torch.Generator(device="cuda").manual_seed(31)
    for u in range(3):
        full = torch.randint(0, 4096, (C_, 128 * nb), dtype=torch.int16, device="cuda", generator=gen)
        full[::997] = -1  # code 65535
        d_in = full[idx].contiguous()
        d_out, d_full = torch.zeros_like(d_in), torch.zeros_like(full)
        torch.cuda.synchronize()
        a.update_adc_list_device(chans, d_in.data_ptr(), d_out.data_ptr(), nb, d_in.stride(0))
        assert a.last_kernel().startswith(COMPOSED + "msdr::v5::") and a.last_kernel().endswith("; channel list"), a.last_kernel()
        b.update_adc_range_device(0, C_, full.data_ptr(), d_full.data_ptr(), nb, full.stride(0))
        a.synchronize(); b.synchronize()
        assert torch.equal(d_out, d_full[idx]), f"update {u}: ADC list against ADC range at size"
        del full, d_in, d_out, d_full
    for c in chans[rng.choice(n, 64, replace=False)]:
        assert bytes(a.get_state(int(c))) == bytes(b.get_state(int(c))), c
        assert bytes(a.get_frontend_state(int(c))) == bytes(b.get_frontend_state(int(c))), c
