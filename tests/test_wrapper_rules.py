"""Caller-supplied outputs and workspaces are checked by one rule for every operator (_ffi.check_out /
_ffi.use_workspace): a buffer the kernels could not use as given is refused with ValueError before any launch."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("shape", [(64, 64), (4, 64, 64)])
def test_median_refuses_an_out_on_another_device(dev, shape):
    import mie_b200 as M

    img = torch.randint(0, 65535, shape, dtype=torch.int32, device=dev).to(torch.uint16)
    with pytest.raises(ValueError):
        M.median(img, out=torch.empty(shape, dtype=img.dtype))                  # host memory
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            M.median(img, out=torch.empty(shape, dtype=img.dtype, device="cuda:1"))
    out = torch.empty_like(img)
    assert M.median(img, out=out) is out
    assert torch.equal(out, M.median(img))


def test_fused_chains_refuse_a_strided_workspace(dev):
    """numel() of a strided view passes a size check, but the library uses that many DENSE bytes from data_ptr()."""
    import mie_b200 as M

    x = torch.zeros(1, 1, 128, 128, dtype=torch.uint16, device=dev)
    for need, run in ((M.chain.bilateral_clahe_workspace_bytes(1, 128, 128, (2, 2)),
                       lambda ws: M.bilateral_clahe(x, 9, 0.1, (1.5, 1.5), 2.0, (2, 2), workspace=ws)),
                      (M.chain_workspace_bytes(1, 128, 128, (2, 2)),
                       lambda ws: M.enhance_chain(x, M.ChainConfig(grid_size=(2, 2)), workspace=ws))):
        strided = torch.empty(2 * need, dtype=torch.uint8, device=dev)[::2]
        assert strided.numel() == need and strided.data_ptr() % 256 == 0
        with pytest.raises(ValueError):
            run(strided)
        run(torch.empty(need, dtype=torch.uint8, device=dev))                    # the dense buffer is accepted
    torch.cuda.synchronize(dev)
