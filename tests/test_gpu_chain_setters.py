"""Chain state calls run on the chain's stream: they never wait for work on other streams.  The range and list front-end presets
leave the same states.  Destroying a chain frees its cached channel-list plans."""
import os

import numpy as np
import pytest

import frontend_lib as fl
from chain_helpers import assert_same, tables_for
from test_gpu_chain_adc import _fe_state_equal
from test_gpu_update_adc_list import _adc_range, _codes
from test_gpu_update_list import USB, Layout

pytestmark = pytest.mark.gpu
SLEEP_CYCLES = 1_000_000_000  # about half a second of torch.cuda._sleep on a B200


@pytest.fixture(scope="module")
def forc():
    return fl.Orc()


# ---- 1. no device-wide wait ----------------------------------------------------------------------------------------------------

def test_state_calls_do_not_wait_for_other_streams(msdr, K):
    """Each call returns while a sleep queued on another torch stream is still running.  Every call runs once before it is timed
    (and the first ANR and front-end use on a second chain), so no timed call loads a module or grows a buffer."""
    import torch
    C_ = 4096
    lay = Layout(K, C_, seed=51)
    g, warm = lay.gpu(msdr), lay.gpu(msdr)
    warm.enable_frontend()
    warm.set_anr(1, 0, 8)
    g.enable_frontend()
    lst = np.arange(5, C_, 97, dtype=np.uint32)[::-1].copy()
    cI, cQ = tables_for(K, USB)
    st, fst, ast = g.get_state(3), g.get_frontend_state(3), warm.get_anr_state(2)
    calls = {
        "set_state": lambda: g.set_state(3, st),
        "set_frontend_state": lambda: g.set_frontend_state(3, fst),
        "enable_frontend": lambda: g.enable_frontend(),
        "frontend_preset": lambda: g.frontend_preset(1000, 10, 300),
        "frontend_preset_list": lambda: g.frontend_preset_list(1000, lst),
        "fir_init_list": lambda: g.fir_init_list(cI, cQ, lst),
        "set_anr (first use)": lambda: g.set_anr(1, 0, 16),
        "set_anr_state": lambda: g.set_anr_state(2, ast),
    }
    for name, call in calls.items():
        if not name.startswith("set_anr"):
            call()
    warm.set_anr_state(2, ast)
    torch.cuda.synchronize()
    other = torch.cuda.Stream()

    def sleep_on_other():
        with torch.cuda.stream(other):
            torch.cuda._sleep(SLEEP_CYCLES)
            ev = torch.cuda.Event()
            ev.record(other)
        return ev

    assert not sleep_on_other().query(), "the sleep ended before it could be checked"
    torch.cuda.synchronize()
    late = []
    for name, call in calls.items():
        ev = sleep_on_other()
        call()
        if ev.query():
            late.append(name)
        torch.cuda.synchronize()
    assert not late, f"returned only after the other stream's sleep had ended: {late}"
    g.synchronize()


# ---- 2. range and list presets -------------------------------------------------------------------------------------------------

def test_range_and_list_presets_agree(msdr, forc, K):
    """The range preset and the list preset of the same channels leave the front-end oracle's states, byte for byte, and the ADC
    updates after them agree."""
    C_, ch0, n, first = 300, 37, 200, 2900
    lay = Layout(K, C_, seed=41)
    a, b = lay.gpu(msdr), lay.gpu(msdr)
    a.enable_frontend()
    b.enable_frontend()
    fo = forc.frontend(C_)
    codes = _codes(C_, 128 * 3, seed=43, extreme=False)
    head = np.ascontiguousarray(codes[:, :128])
    assert_same(_adc_range(a, 0, head), _adc_range(b, 0, head), "before the presets")
    fo.run(head)
    launches = a.launch_count()
    a.frontend_preset(first, ch0, n)
    assert a.launch_count() == launches + 1, "the range preset is one kernel"
    b.frontend_preset_list(first, lay.rng.permutation(np.arange(ch0, ch0 + n)))
    for c in range(ch0, ch0 + n):
        fo.preset(c, first)
    a.synchronize()
    for c in range(C_):
        assert bytes(a.get_frontend_state(c)) == bytes(b.get_frontend_state(c)), c
        _fe_state_equal(a.get_frontend_state(c), fo.state(c), c)
    tail = np.ascontiguousarray(codes[:, 128:])
    assert_same(_adc_range(a, 0, tail), _adc_range(b, 0, tail), "after the range and the list preset")
    fo.run(tail)
    for c in range(C_):
        _fe_state_equal(a.get_frontend_state(c), fo.state(c), c)
        assert bytes(a.get_frontend_state(c)) == bytes(b.get_frontend_state(c)), c


# ---- 3. no leak at destroy -----------------------------------------------------------------------------------------------------

def _process_used_bytes():
    """This process's device memory as NVML lists it, or None when NVML lists no entry for it."""
    pynvml = pytest.importorskip("pynvml")
    try:
        pynvml.nvmlInit()
    except pynvml.NVMLError as e:
        pytest.skip(f"NVML unavailable: {e}")
    try:
        used = None
        for i in range(pynvml.nvmlDeviceGetCount()):
            for p in pynvml.nvmlDeviceGetComputeRunningProcesses(pynvml.nvmlDeviceGetHandleByIndex(i)):
                if p.pid == os.getpid() and p.usedGpuMemory is not None:
                    used = (used or 0) + p.usedGpuMemory
        return used
    finally:
        pynvml.nvmlShutdown()


def test_destroy_frees_list_plans(msdr, K):
    """Chains that cached plans of 2^20-channel lists are created and destroyed in a loop; this process's device memory must not
    grow by the lists' device copies (4 bytes a listed channel, per plan)."""
    import torch
    C_, n_chains = 1 << 20, 5
    rng = np.random.default_rng(61)
    lists = [rng.permutation(C_).astype(np.uint32)[:C_ - 4096 * i] for i in range(3)]
    d_in = torch.zeros((C_, 128), dtype=torch.int16, device="cuda")
    d_out = torch.empty_like(d_in)
    cI, cQ = tables_for(K, USB)

    def cycle():
        g = msdr.ReceiveChain(C_)
        g.set_mode(USB)
        g.fir_init(cI, cQ)
        for ch in lists:
            g.update_list_device(ch, d_in.data_ptr(), d_out.data_ptr(), 1, d_in.stride(0))
        g.synchronize()
        assert g.plan_build_count() == len(lists)
        g.close()

    cycle()  # first use: modules and the driver's own structures
    torch.cuda.synchronize()
    before = _process_used_bytes()
    if before is None:
        pytest.skip("NVML lists no entry for this process (its PID is not visible to NVML here)")
    for _ in range(n_chains):
        cycle()
    torch.cuda.synchronize()
    after = _process_used_bytes()
    lists_bytes = n_chains * sum(4 * ch.size for ch in lists)
    assert after - before < lists_bytes // 2, (before, after, lists_bytes)
