"""CPU-side checks of the drop-in surface: constructor RNG parity with the reference, state_dict keys,
C-ABI exports, and that there is no CPU fallback."""
import ctypes
import os
import re

import pytest
import torch

import vit3d_b200
from oracle import vit3d_oracle as O
from tests.helpers import CASES, assert_stats_equal, load_golden, stats
from vit3d_b200 import _lib
from vit3d_b200.models.modeling import (Attention, Block, Embeddings, Encoder, Mlp, Transformer, TransformerEnsemble,
                                        VisionTransformer)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("name", list(CASES))
def test_constructor_matches_reference_rng_and_keys(name):
    """Same seed -> same initial weights and state_dict keys as the reference's VisionTransformer."""
    g = load_golden("init_seed42")
    args, _ = CASES[name]
    cfg = vit3d_b200.get_config(*args)
    torch.manual_seed(42)
    m = VisionTransformer(cfg, 128, zero_head=True, num_classes=1)
    sd = m.state_dict()
    keys = sorted(k[len(name) + 1:] for k in g.files if k.startswith(name + "/"))
    assert sorted(sd.keys()) == keys
    for k in keys:
        assert_stats_equal(stats(sd[k]), g[f"{name}/{k}"], k)


def test_state_dict_roundtrip_with_oracle_layout():
    cfg = vit3d_b200.north_star_config(5)
    sd = O.init_state_dict(cfg, seed=3)
    m = VisionTransformer(cfg, 128, zero_head=True, num_classes=1)
    missing, unexpected = m.load_state_dict(sd)
    assert not missing and not unexpected
    for k, v in m.state_dict().items():
        assert torch.equal(v, sd[k])
    assert sum(p.numel() for p in m.parameters()) == 8236033


def test_ensemble_keys():
    cfgs = [vit3d_b200.north_star_config(c) for c in (5, 9, 11)]
    ens = TransformerEnsemble(*[VisionTransformer(c, 128, zero_head=True, num_classes=1) for c in cfgs], in_features=1)
    assert len(ens.state_dict()) == 314       # SURVEY.md §8b [probed]
    assert ens.classifier.weight.shape == (1, 3)
    # reference default in_features=3 builds Linear(9,1) (modeling.py:348-351): same constructor behaviour
    ens3 = TransformerEnsemble(*[VisionTransformer(cfgs[0], 128, num_classes=1)], in_features=3)
    assert ens3.classifier.weight.shape == (1, 3)


def test_config_tables():
    assert vit3d_b200.parameters_config(5) == (16, 3072, 8, 16, 16)     # tools.py:60-80 as shipped
    assert vit3d_b200.parameters_config(20) == (8, 2204, 6, 8, 8)
    c = vit3d_b200.north_star_config(18)
    assert (c.hidden_size, c.transformer["mlp_dim"], c.transformer.num_layers, c.transformer["num_heads"]) == (256, 3072, 8, 16)
    assert c.patches.get("grid") is None and c.patches["size"] == (16, 16, 5) and c.classifier == "token"


def test_c_abi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "vit3d.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(vit3d_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 25
    assert os.path.exists(_lib.LIB_PATH), "libvit3d_sm100.so must be built (python -c 'import __graft_entry__ as g; g.build()')"
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(L, name), f"{name} declared in include/vit3d.h but not exported"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert _lib.lib().vit3d_version() == 100
    # ABI constants the Python side mirrors
    assert int(re.search(r"#define VIT3D_SHADOW_TILE (\d+)", hdr).group(1)) == _lib.SHADOW_TILE


def test_no_cpu_fallback():
    cfg = vit3d_b200.get_config(16, 64, 2, 32, 4)
    m = VisionTransformer(cfg, 128, zero_head=True, num_classes=1)
    with pytest.raises(vit3d_b200.Vit3dError):
        m(torch.zeros(1, 1, 128, 128, 5))
    with pytest.raises(vit3d_b200.Vit3dError):
        Mlp(cfg)(torch.zeros(1, 65, 32))


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "3d_vit_ensemble_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), f
                assert "vit3d_oracle" not in src, f


def test_reference_import_line_works_with_package_dir_on_sys_path(tmp_path):
    """`from models.modeling import VisionTransformer` (train_baseline_cv.py:14) resolves to this
    implementation when 3d_vit_ensemble_b200/ is on sys.path, with the SAME class objects."""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r); "
            "from models.modeling import VisionTransformer, TransformerEnsemble; "
            "import importlib; v = importlib.import_module('3d_vit_ensemble_b200.vit'); "
            "assert VisionTransformer is v.VisionTransformer; print('ok')") % os.path.join(ROOT, "3d_vit_ensemble_b200")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr
