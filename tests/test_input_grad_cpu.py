"""The reference semantics of the input-volume gradient, pinned without the oracle's im2col: the oracle's d tokens / d x
equals that of a plain torch.nn.Conv3d + flatten(2).transpose + cls concat + position add (Embeddings.forward,
modeling.py:162-173) in fp64, including the voxels Conv3d drops (gradient 0)."""
import pytest
import torch

from oracle import vit3d_oracle as O


@pytest.mark.parametrize("size", [128, 130])
@pytest.mark.parametrize("patch", [16, 8])
def test_oracle_input_grad_equals_conv3d_embedding(size, patch):
    cfg = O.get_config(patch, 64, 1, 32, 4)
    sd = O.to_dtype(O.init_state_dict(cfg, seed=3), torch.float64)
    pre = "transformer.embeddings."
    gen = torch.Generator().manual_seed(size + patch)
    x = torch.randn(2, 1, size, size, 5, generator=gen, dtype=torch.float64)

    xa = x.clone().requires_grad_()
    tok = O.embeddings(sd, cfg, xa)
    g = torch.randn(tok.shape, generator=gen, dtype=torch.float64)
    tok.backward(g)

    w = sd[pre + "patch_embeddings.weight"]
    conv = torch.nn.Conv3d(1, w.shape[0], kernel_size=w.shape[2:], stride=w.shape[2:]).double()
    with torch.no_grad():
        conv.weight.copy_(w)
        conv.bias.copy_(sd[pre + "patch_embeddings.bias"])
    xb = x.clone().requires_grad_()
    t = conv(xb).flatten(2).transpose(-1, -2)
    t = torch.cat((sd[pre + "cls_token"].expand(2, -1, -1), t), dim=1) + sd[pre + "position_embeddings"]
    t.backward(g)

    torch.testing.assert_close(xa.grad, xb.grad, rtol=1e-12, atol=1e-12)
    if size % patch:
        assert (xa.grad[:, :, size - size % patch:] == 0).all()
