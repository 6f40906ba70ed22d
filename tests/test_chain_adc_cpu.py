"""The ADC-code input of the receive chain without a GPU: it fails loudly, there is no CPU fallback."""
import pytest


def test_update_adc_without_device_fails(msdr):
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(msdr.capi.MsdrError) as ei:
        g = msdr.ReceiveChain(64)
        g.enable_frontend()
        g.update_adc(__import__("numpy").zeros((64, 128), "uint16"))
    assert ei.value.status == msdr.capi.ERR_CUDA
    assert "no CPU fallback" in str(ei.value)
