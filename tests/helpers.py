"""Shared helpers for the parity tests (test infrastructure)."""
import os

import numpy as np
import torch

from oracle import vit3d_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

CASES = {
    "tiny": ((16, 64, 2, 32, 4), 3),
    "shipped": ((16, 3072, 8, 16, 16), 2),
    "shipped_p8": ((8, 2204, 6, 8, 8), 1),
    "conf5": ((16, 2048, 6, 256, 8), 2),
    "conf9": ((16, 2048, 8, 256, 16), 2),
    "conf11": ((16, 3072, 4, 256, 8), 2),
    "conf18": ((16, 3072, 8, 256, 16), 2),
    "conf1": ((16, 2048, 4, 256, 4), 2),
}


def stats(t: torch.Tensor) -> np.ndarray:
    """Same statistic vector as oracle/gen_golden.py:stats."""
    t = t.detach().double().reshape(-1).cpu()
    head = torch.zeros(8, dtype=torch.float64)
    n = min(8, t.numel())
    head[:n] = t[:n]
    w = torch.arange(1, t.numel() + 1, dtype=torch.float64) / t.numel()
    return torch.cat([torch.stack([t.sum(), t.norm(), t.abs().max(), (t * w).sum()]), head]).numpy()


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def case_setup(name):
    """Config, seeded weights (same RNG stream as the reference ctor + token re-draw),
    inputs, labels, pos_weight of a golden case."""
    args, B = CASES[name]
    cfg = O.get_config(*args)
    sd = O.init_state_dict(cfg, seed=42, randomize_tokens=True)
    x = O.synth_volumes(B, seed=42, kind="img")
    y = O.synth_labels(B)
    w = O.balanced_pos_weight(y)
    return cfg, sd, x, y, w


def unpack_masks(g):
    masks = {}
    for k in g.files:
        if not k.startswith("mask/"):
            continue
        kn = k[len("mask/"):]
        shape = tuple(int(v) for v in g["mask_shape/" + kn])
        n = int(np.prod(shape))
        m = np.unpackbits(g[k])[:n].reshape(shape).astype(bool)
        key = "emb" if kn == "emb" else (kn.split("_")[0], int(kn.split("_")[1]))
        masks[key] = torch.from_numpy(m)
    return masks


def assert_stats_equal(got: np.ndarray, want: np.ndarray, what=""):
    """`stats` of the same tensor values.  The max and the leading elements are values of the tensor: bit exact.
    Sum, L2 norm and weighted sum are float64 reductions whose order, and so whose last bit, depends on the CPU's
    vector width: they are held to 1e-14 of the L2 norm (~45 float64 epsilons), which admits float64 rounding while
    a one-ulp change of any float32 element larger than ~2e-7 of the norm still fails."""
    np.testing.assert_array_equal(got[2:3], want[2:3], err_msg=what)
    np.testing.assert_array_equal(got[4:], want[4:], err_msg=what)
    np.testing.assert_allclose(got[[0, 1, 3]], want[[0, 1, 3]], rtol=0, atol=1e-14 * float(want[1]), err_msg=what)


def assert_stats_close(got: np.ndarray, want: np.ndarray, rtol, atol, what=""):
    scale = max(float(want[1]), 1e-30)          # L2 norm of the golden tensor
    # sum / weighted-sum are compared relative to the norm (they cancel)
    for i in (0, 3):
        assert abs(got[i] - want[i]) <= rtol * scale * 40 + atol, (what, i, got[i], want[i])
    assert abs(got[1] - want[1]) <= rtol * scale + atol, (what, "l2", got[1], want[1])
    assert abs(got[2] - want[2]) <= rtol * max(float(want[2]), 1e-30) * 4 + atol, (what, "max", got[2], want[2])
    np.testing.assert_allclose(got[4:], want[4:], rtol=rtol * 50, atol=rtol * float(want[2]) * 4 + atol, err_msg=what)
