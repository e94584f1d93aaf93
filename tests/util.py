"""Shared helpers for the parity tests: golden loading and comparisons."""
import ast
import os

import numpy as np
import torch

from gluefactory_b200 import synthetic

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = ["lg_small_d128_l2_n96", "lg_small_d128_l2_m80_n112", "lg_d256_l3_n160",
         "lg_disk_d256_l2_n128", "lg_full_l9_n512"]
EXTRA_CASES = ["lg_sift_d256_l2_n96"]  # add_scale_ori (SIFT-style scale / orientation inputs), input_dim 128, M != N


def load_case(name, dtype=torch.float64):
    """Returns (golden dict, conf, weights, data) with inputs rebuilt from the stored seeds."""
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False))
    conf = ast.literal_eval(str(g["meta|conf"]))
    B, N, M, seed = (int(g["meta|" + k]) for k in ["B", "N", "M", "seed"])
    weights = {k: v.to(dtype) for k, v in synthetic.make_weights(conf, seed=seed).items()}
    data = synthetic.make_pairs(B, N, seed=seed + 1, D=conf["input_dim"], M=M, dtype=dtype)
    if conf.get("add_scale_ori"):
        data = synthetic.add_scale_ori_inputs(data, seed + 2)
    return g, conf, weights, data


def load_gluestick_attn():
    """tests/golden/gluestick_attn.npz with its inputs: the fixture stores the reference's outputs and gradients, the
    inputs are re-drawn from the generator's seeded stream (oracle/make_golden.py run_gluestick_attention)."""
    g = dict(np.load(os.path.join(GOLDEN, "gluestick_attn.npz"), allow_pickle=False))
    rs = np.random.RandomState(21)
    b, d, h, n, m = 1, 64, 4, 40, 56
    for k, shape in (("core|q", (b, d, h, n)), ("core|k", (b, d, h, m)), ("core|v", (b, d, h, m)),
                     ("core|w", (b, d, h, n)), ("mha|x", (b, 256, n)), ("mha|src", (b, 256, m)), ("mha|w", (b, 256, n))):
        g[k] = rs.standard_normal(shape)
    return g


def probe_index(n, k=512):
    return torch.from_numpy(np.random.RandomState(n % 65521).randint(0, n, size=k))


def probe_vector(n):
    return torch.from_numpy(np.random.RandomState((n * 7919) % 65521).standard_normal(n))


def check_grad_summary(g, name, grad, rtol, atol_scale=1.0):
    """Compare a gradient tensor against the summary stored by oracle/make_golden.py.
    Tolerance is relative to the gradient's own norm (||err|| <= rtol * ||g||)."""
    grad = grad.detach().double().cpu()
    ref_norm = float(g[f"grad|{name}|norm"])
    tol = rtol * max(ref_norm, 1e-12) * atol_scale
    assert abs(grad.norm().item() - ref_norm) <= tol + 1e-300, (name, grad.norm().item(), ref_norm)
    if f"grad|{name}|full" in g:
        ref = torch.from_numpy(g[f"grad|{name}|full"])
        err = (grad - ref).norm().item()
        assert err <= tol, (name, err, ref_norm)
    else:
        flat = grad.reshape(-1)
        ref = torch.from_numpy(g[f"grad|{name}|sample"])
        got = flat[probe_index(flat.numel())]
        # 512 samples of n entries carry ~sqrt(512/n) of the norm
        scale = ref_norm * (512.0 / flat.numel()) ** 0.5
        err = (got - ref).norm().item()
        assert err <= rtol * max(scale, 1e-12) * 4 * atol_scale, (name, err, scale)
        proj = (flat * probe_vector(flat.numel())).sum().item()
        assert abs(proj - float(g[f"grad|{name}|proj"])) <= 4 * tol, (name, proj, float(g[f"grad|{name}|proj"]))


def rel_err(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / b.norm().clamp(min=1e-30)).item()


def report(tag, **vals):
    """Append measured error figures to gpurun_out/parity_report.txt (when that directory exists): the numbers behind
    the tolerance table in DESIGN.md.  Never fails a test."""
    try:
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        d = os.path.join(root, "gpurun_out")
        if os.path.isdir(d):
            with open(os.path.join(d, "parity_report.txt"), "a") as f:
                f.write(tag + " " + " ".join(f"{k}={v:.4g}" if isinstance(v, float) else f"{k}={v}" for k, v in vals.items()) + "\n")
    except Exception:  # noqa: BLE001
        pass
