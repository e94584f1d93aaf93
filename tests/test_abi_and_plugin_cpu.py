"""CPU: the C-ABI library loads and exports every symbol of include/lgb200.h; the plugin honours
the reference's plugin surface (construction, names, state_dict) and fails loudly without a GPU."""
import ast
import importlib
import importlib.util
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge

    return ge.build()


def test_library_exports_every_declared_symbol(built):
    from gluefactory_b200 import _lib

    hdr = open(os.path.join(ROOT, "include", "lgb200.h")).read()
    declared = set(re.findall(r"\b(lgb200_[a-z0-9_]+)\s*\(", hdr))
    assert declared and declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = _lib.load(check_device=False)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.lgb200_abi_version() == 2
    # pure host queries are callable without a GPU
    assert lib.lgb200_assign_ws_bytes(2, 64, 64) == 2 * 2 * 64 * 8
    assert lib.lgb200_ln_gelu_bwd_parts(1000) == 125


def test_plugin_surface_matches_reference_names():
    from gluefactory_b200 import synthetic
    from gluefactory_b200.matchers import lightglue as plug

    model = plug.__main_model__({"name": "gluefactory_b200.matchers.lightglue", "n_layers": 3, "unknown_key": 1})
    names = [n for n, _ in model.named_parameters()]
    conf = dict(synthetic.DEFAULT_CONF, n_layers=3)
    assert names == [n for n, _ in synthetic.state_dict_spec(conf)]
    for n, shape in synthetic.state_dict_spec(conf):
        assert tuple(model.state_dict()[n].shape) == tuple(shape), n
    assert "confidence_thresholds" in model.state_dict()
    assert model.required_data_keys == ["keypoints0", "keypoints1", "descriptors0", "descriptors1"]
    disk = plug.LightGlue({"input_dim": 128, "n_layers": 1})
    assert tuple(disk.input_proj.weight.shape) == (256, 128)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    from gluefactory_b200 import synthetic
    from gluefactory_b200._lib import Lgb200Error
    from gluefactory_b200.matchers.lightglue import LightGlue

    model = LightGlue({"n_layers": 1})
    data = synthetic.make_pairs(1, 64, seed=1)
    with pytest.raises(Lgb200Error, match="no CPU fallback"):
        model(data)


def test_dropin_through_reference_get_model():
    """The reference's get_model resolves a dotted module name that holds no subclass of its BaseModel to the module's
    `__main_model__` (models/__init__.py:7-30), and TwoViewPipeline builds its matcher and ground-truth components
    from plain config dicts through it (two_view_pipeline.py:48-56).  Found that way, the plugin must expose the
    reference matcher's state_dict and the reference ground-truth component's conf and inputs, as recorded from the
    unmodified reference in tests/golden/dropin_surface.npz (oracle/make_golden.py)."""
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "dropin_surface.npz"), allow_pickle=False))

    def get_model(name):
        assert importlib.util.find_spec(name) is not None, name
        return importlib.import_module(name).__main_model__

    cls = get_model("gluefactory_b200.matchers.lightglue")
    mine = cls({"n_layers": 2})
    assert list(mine.state_dict().keys()) == list(g["lightglue|keys"])
    for k in g["lightglue|keys"]:
        assert tuple(mine.state_dict()[k].shape) == tuple(g["lightglue|shape|" + k]), k
    np.testing.assert_allclose(mine.confidence_thresholds.numpy(), g["lightglue|confidence_thresholds"], rtol=1e-7)
    mine.load_state_dict({k: torch.zeros(tuple(g["lightglue|shape|" + k])) for k in g["lightglue|keys"]})  # strict
    assert isinstance(cls({"name": "gluefactory_b200.matchers.lightglue", "n_layers": 1}), cls)
    gt_cls = get_model("gluefactory_b200.matchers.homography_matcher")
    gt = gt_cls({"name": "gluefactory_b200.matchers.homography_matcher", "th_positive": 2.0})
    assert gt.conf.th_positive == 2.0
    assert sorted(gt_cls({}).required_data_keys) == list(g["homography|required_data_keys"])
    for k, v in ast.literal_eval(str(g["homography|default_conf"])).items():
        assert gt_cls.default_conf[k] == v, k
    with pytest.raises(NotImplementedError):
        gt_cls({}).loss({}, {})
    with pytest.raises(Exception):  # CPU tensors: the op refuses instead of falling back to the CPU
        gt_cls({})({"H_0to1": torch.eye(3)[None], "keypoints0": torch.zeros(1, 4, 2), "keypoints1": torch.zeros(1, 4, 2)})


def test_split_operand_host_logic():
    """Host side of the tensor-core parity mode (`precision: bf16x3`): the bf16 hi / lo split of an fp32 operand loses
    2^-16 at most, the K-concatenated products [Ah|Ah|Al] x [Bh|Bl|Bh] reproduce A B to ~1e-5, and the mode switch is
    scoped (a node's backward runs under the mode of its forward)."""
    from gluefactory_b200 import engine

    g = torch.Generator().manual_seed(0)
    a, b = torch.randn(37, 64, generator=g), torch.randn(53, 64, generator=g)
    a3, b3 = engine.split3(a, 1, "hhl"), engine.split3(b, 1, "hlh")
    assert a3.dtype == torch.bfloat16 and a3.shape == (37, 192)
    hi, lo = a3[:, :64].float(), a3[:, 128:].float()
    assert ((hi + lo) - a).abs().max() <= a.abs().max() * 2.0 ** -15
    ref = a.double() @ b.double().t()
    got = a3.double() @ b3.double().t()
    plain = a.bfloat16().double() @ b.bfloat16().double().t()
    err = lambda x: ((x - ref).norm() / ref.norm()).item()  # noqa: E731
    assert err(got) < 2e-5 and err(got) < err(plain) / 50
    assert engine.FP32_GEMM == "cublas"
    with engine.fp32_gemm("x3"):
        assert engine.FP32_GEMM == "x3"
        with engine.fp32_gemm("cublas"):
            assert engine.FP32_GEMM == "cublas"
        assert engine.FP32_GEMM == "x3"
    assert engine.FP32_GEMM == "cublas"


def test_mask_counts_host_fallback():
    from gluefactory_b200 import ops

    m = (torch.rand(2, 9, 13, generator=torch.Generator().manual_seed(1)) < 0.3)
    r, c = ops.mask_counts(m.view(torch.uint8))
    assert torch.equal(r, m.sum(2).float()) and torch.equal(c, m.sum(1).float())
