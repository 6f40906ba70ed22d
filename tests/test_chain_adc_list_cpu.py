"""ADC-code channel-list updates without a GPU: they fail loudly, there is no CPU fallback."""
import pytest


def test_update_adc_list_without_device_fails(msdr):
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    np = pytest.importorskip("numpy")
    with pytest.raises(msdr.capi.MsdrError) as ei:
        g = msdr.ReceiveChain(64)
        g.enable_frontend()
        g.update_adc_list([3, 1, 2], np.zeros((3, 128), np.uint16))
    assert ei.value.status == msdr.capi.ERR_CUDA
    assert "no CPU fallback" in str(ei.value)
