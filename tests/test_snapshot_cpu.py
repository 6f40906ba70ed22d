"""Snapshot format and re-sharding plans without a GPU: msdr_snapshot_info reads a header built here from the layout DESIGN.md 7
documents; shard.reshard covers every channel once; the device entry points fail loudly (there is no CPU fallback)."""
import numpy as np
import pytest

HEADER = 256
TABLES = 32 * (4 + 2 * 256 + 2 * 256)


def _align(x):
    return (x + 255) // 256 * 256


def layout(nch, hist_len, frontend, anr):
    """Section offsets (tables, meta, hist, bq, pll, fe, anr d, w, lidx, ngamma, in_idx; 0 = absent) and the total size."""
    sizes = [TABLES, 4 * nch, 2 * nch * hist_len, 4 * 64 * nch, 4 * 3 * nch, 72 * nch if frontend else None]
    sizes += [4 * 512 * nch, 4 * 64 * nch, 4 * nch, 4 * nch, 4 * nch] if anr else [None] * 5
    off, p = [], HEADER
    for s in sizes:
        if s is None:
            off.append(0)
        else:
            off.append(p)
            p = _align(p + s)
    return off, p


def header(nch=100, hist_len=104, frontend=True, anr=False, flags=0, version=1, magic=b"MSDRSNAP", max_taps=102):
    off, total = layout(nch, hist_len, frontend, anr)
    h = np.zeros(HEADER, np.uint8)
    h[:8] = np.frombuffer(magic, np.uint8)
    fields = np.array([version, HEADER], np.uint32).tobytes() + np.array([total], np.uint64).tobytes()
    fields += np.array([nch, flags, hist_len, (1 if frontend else 0) | (2 if anr else 0)], np.uint32).tobytes()
    fields += np.array([0.25, 40.0], np.float32).tobytes() + np.array([1], np.int32).tobytes()
    fields += np.array([3, max_taps, 0], np.uint32).tobytes() + np.array(off, np.uint64).tobytes()
    h[8:8 + len(fields)] = np.frombuffer(fields, np.uint8)
    return h, total


def test_layout_sizes():
    """About 480 bytes a channel for the C5 shape (H = 104): history 208, biquads 256, PLL 12, meta 4."""
    _, total = layout(1 << 20, 104, False, False)
    per = (total - HEADER - _align(TABLES)) / (1 << 20)
    assert 480 <= per < 481


def test_info_accepts_documented_header(msdr):
    h, total = header(nch=100, frontend=True, anr=True, flags=msdr.capi.FLAG_AM_Q31)
    info = msdr.capi.snapshot_info(h)
    assert info == {"n_channels": 100, "max_taps_needed": 102,
                    "flags": msdr.capi.FLAG_AM_Q31 | msdr.capi.SNAPSHOT_FRONTEND | msdr.capi.SNAPSHOT_ANR}
    h, _ = header(nch=7, hist_len=264, frontend=False, anr=False, max_taps=256)
    assert msdr.capi.snapshot_info(h) == {"n_channels": 7, "max_taps_needed": 256, "flags": 0}


def test_info_rejects(msdr):
    E = msdr.capi
    L = E.lib()
    h, _ = header()
    cases = [
        (header(magic=b"MSDRSNAQ")[0], HEADER, E.ERR_ARGUMENT),
        (h, HEADER - 1, E.ERR_ARGUMENT),  # truncated header
        (header(version=2)[0], HEADER, E.ERR_UNSUPPORTED),
        (header(version=0)[0], HEADER, E.ERR_UNSUPPORTED),
    ]
    bad_off = h.copy()
    bad_off[64 + 16:64 + 24] = np.frombuffer(np.array([1 << 40], np.uint64).tobytes(), np.uint8)  # the history offset past the end
    cases.append((bad_off, HEADER, E.ERR_ARGUMENT))
    bad_total = h.copy()
    bad_total[16:24] = np.frombuffer(np.array([HEADER], np.uint64).tobytes(), np.uint8)
    cases.append((bad_total, HEADER, E.ERR_ARGUMENT))
    for blob, size, want in cases:
        assert L.msdr_snapshot_info(E.ptr(blob), size, None, None, None) == want
    with pytest.raises(E.MsdrError):
        E.snapshot_info(h[:200])


@pytest.mark.parametrize("total,old,new", [(1000, 3, 2), (1000, 2, 3), (1 << 20, 8, 5), (33, 1, 4), (4096, 4, 4)])
@pytest.mark.parametrize("granule", [32, 1])
def test_reshard_covers_every_channel_once(msdr, total, old, new, granule):
    sh = msdr.shard
    olds, news = sh.plan(total, old, granule=granule), sh.plan(total, new, granule=granule)
    seen = np.zeros(total, np.int32)
    for p in sh.reshard(total, old, new, granule=granule):
        o, n = olds[p.old_rank], news[p.new_rank]
        assert p.n > 0 and p.first + p.n <= o.n and p.dst_ch0 + p.n <= n.n
        assert o.ch0 + p.first == n.ch0 + p.dst_ch0  # the same global channels on both sides
        seen[o.ch0 + p.first:o.ch0 + p.first + p.n] += 1
    assert (seen == 1).all()


def test_snapshot_without_device_fails(msdr):
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(msdr.capi.MsdrError) as ei:  # no chain, so no snapshot and no restore: the chain itself cannot exist
        msdr.ReceiveChain(64).snapshot()
    assert ei.value.status == msdr.capi.ERR_CUDA and "no CPU fallback" in str(ei.value)
    L = msdr.capi.lib()
    assert L.msdr_chain_snapshot_bytes(None, 64) == 0
    h, _ = header()
    assert L.msdr_chain_restore(None, 0, msdr.capi.ptr(h), h.size, 0, 1) == msdr.capi.ERR_ARGUMENT
