"""K3 study kernel: mix + FIR pair + demod on the tensor cores (tcgen05 kind::i8, byte-split Toeplitz form) against the oracle.
The oracle chain with identity biquads (b0 = 2^30) returns exactly the demodulated samples."""
import numpy as np
import pytest

import oracle_lib as ol
from chain_helpers import assert_same, tables_for
from conftest import adversarial_inputs, wrap_coeffs

pytestmark = pytest.mark.gpu
IDENT = np.array([1 << 30, 0, 0, 0, 0], np.int32)
KIND_TO_MODE = {0: ol.MODE_LSB, 1: ol.MODE_USB, 2: ol.MODE_AM, 3: ol.MODE_AM}


def _oracle(orc, cI, cQ, kinds, x, q31):
    o = orc.chain(x.shape[0], q31)
    for r, k in enumerate(kinds):
        o.set_mode(r, 1, KIND_TO_MODE[int(k)])
    o.fir_init(0, x.shape[0], cI, cQ)
    for obj in (0, 1):
        o.biquad_set_coefficients(obj, 0, x.shape[0], 0, IDENT)
    return o.run(x)[0]


def _tc(msdr, cI, cQ, kinds, x):
    L, p = msdr.capi.lib(), msdr.capi.ptr
    out = np.empty_like(x)
    kinds = np.ascontiguousarray(kinds, np.uint8)
    cI, cQ = np.ascontiguousarray(cI, np.int16), np.ascontiguousarray(cQ, np.int16)
    st = L.msdr_op_fir_demod_tc(0, len(cI), p(cI), p(cQ), p(kinds), 0, p(x), p(out), x.shape[0], x.shape[1], x.shape[1])
    assert st == 0, st
    return out


@pytest.mark.parametrize("q31", [False, True])
def test_tc_reference_tables(msdr, orc, K, q31):
    rng = np.random.default_rng(5)
    for mode in (ol.MODE_USB, ol.MODE_AM, ol.MODE_CW):
        cI, cQ = tables_for(K, mode)
        rows = 130  # not a multiple of the 128-row tile
        kinds = np.array([(3 if q31 else 2) if r % 3 == 2 else r % 3 for r in range(rows)], np.uint8)  # LSB, USB, envelope
        x = msdr.synth.batch([KIND_TO_MODE[int(k)] for k in kinds], 128 * 7)
        x[5] = rng.integers(-32768, 32768, x.shape[1], dtype=np.int16)
        x[6] = -32768
        assert_same(_tc(msdr, cI, cQ, kinds, x), _oracle(orc, cI, cQ, kinds, x, q31), f"tc mode {mode} q31 {q31}")


@pytest.mark.parametrize("T", [4, 38, 62, 64, 86, 102, 128, 190, 192, 254, 256])
def test_tc_wrap_and_saturation(msdr, orc, T):
    """Random full-range taps (accumulator wraps, outputs saturate) on the adversarial inputs, every tap count class, both edges of
    every FIR window (64, 96, 128, 160 and 192 words)."""
    rng = np.random.default_rng(T)
    ins = adversarial_inputs(128 * 4, rng)
    names = sorted(ins)
    x = np.stack([ins[n] for n in names for _ in range(4)])
    kinds = np.array([i % 4 for i in range(x.shape[0])], np.uint8)
    for trial in range(2):
        cI, cQ = wrap_coeffs(T, rng), wrap_coeffs(T, rng)
        got = _tc(msdr, cI, cQ, kinds, x)
        for q31 in (False, True):
            sel = np.array([k in (0, 1) or (k == 3) == q31 for k in kinds])
            exp = _oracle(orc, cI, cQ, np.where(kinds == 3, 3, kinds), x, q31)
            assert_same(got[sel], exp[sel], f"tc wrap T={T} q31={q31}")


def test_tc_is_tensor_core_code(msdr):
    """The study kernel really issues tcgen05 MMAs: SASS carries UTCIMMA and TMEM loads."""
    import shutil
    import subprocess
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run(["cuobjdump", "-sass", msdr.lib_path()], capture_output=True, text=True).stdout
    assert "UTCIMMA" in sass and "LDTM" in sass


def test_tc_envelope_sqrt_equals_sqrt_rn_everywhere(msdr):
    """The epilogue's branch-free sqrtf is bit-identical to sqrt.rn.f32 for EVERY AM envelope argument (2^31 integers)."""
    import ctypes as C
    bad = C.c_uint64(123)
    st = msdr.capi.lib().msdr_study_sqrt_check(0, C.byref(bad))
    assert st == 0
    assert bad.value == 0
