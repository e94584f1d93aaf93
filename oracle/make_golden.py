"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED
reference (TEST INFRASTRUCTURE ONLY; runs in the build container, where
/root/reference exists -- the GPU box only ever sees the committed .npz files).

    python oracle/make_golden.py            # writes tests/golden/*.npz

The reference modules are imported from /root/reference with the omegaconf
stand-in of oracle/_shim on sys.path (omegaconf is not installed here).
Weights and inputs come from gluefactory_b200.synthetic (numpy RandomState
streams), so tests regenerate the exact same inputs from the seeds stored in
each fixture.  Big matrices (parameter gradients) are stored as a fixed
sub-sample plus two scalar functionals, see `summarise`.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("GLUEFACTORY_REFERENCE", "/root/reference")
sys.path.insert(0, os.path.join(HERE, "_shim"))
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

from gluefactory_b200 import synthetic  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def summarise(name, g):
    """Compact, order-sensitive summary of a gradient tensor."""
    g = g.detach().double().cpu()
    out = {f"{name}|norm": np.array(g.norm().item())}
    if g.numel() <= 4096:
        out[f"{name}|full"] = g.numpy()
    else:
        flat = g.reshape(-1)
        idx = probe_index(flat.numel())
        out[f"{name}|sample"] = flat[idx].numpy()
        out[f"{name}|proj"] = np.array((flat * probe_vector(flat.numel())).sum().item())
    return out


def probe_index(n, k=512):
    return torch.from_numpy(np.random.RandomState(n % 65521).randint(0, n, size=k))


def probe_vector(n):
    return torch.from_numpy(np.random.RandomState((n * 7919) % 65521).standard_normal(n))


def build_reference(conf, weights, dtype):
    from gluefactory.models import get_model

    cls = get_model("matchers.lightglue")
    model = cls(dict(conf))
    sd = {k: v.to(dtype) for k, v in weights.items()}
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert missing == [] or missing == ["confidence_thresholds"], missing
    return model.to(dtype).train()


def run_case(name, conf, B, N, M, seed, dtype=torch.float64, sub=1):
    weights = synthetic.make_weights(conf, seed=seed)
    data = synthetic.make_pairs(B, N, seed=seed + 1, D=conf["input_dim"], M=M, dtype=dtype)
    if conf.get("add_scale_ori"):
        data = synthetic.add_scale_ori_inputs(data, seed + 2)
    model = build_reference(conf, weights, dtype)
    pred = model(data)
    losses, _ = model.loss(pred, data)
    loss = losses["total"].mean()
    loss.backward()
    out = {
        "meta|B": np.array(B), "meta|N": np.array(N), "meta|M": np.array(M), "meta|seed": np.array(seed),
        "meta|conf": np.array(repr(conf)),
    }
    for k in ["matches0", "matches1", "matching_scores0", "matching_scores1"]:
        out["pred|" + k] = pred[k].detach().cpu().numpy()
    la = pred["log_assignment"].detach()
    out["pred|log_assignment"] = la[:, ::sub, ::sub].cpu().numpy()
    out["pred|log_assignment_rowmax"] = la[:, :-1, :-1].max(2).values.cpu().numpy()
    out["pred|log_assignment_colmax"] = la[:, :-1, :-1].max(1).values.cpu().numpy()
    for k, v in losses.items():
        out["loss|" + k] = v.detach().cpu().numpy() if torch.is_tensor(v) else np.array(v)
    for k, p in model.named_parameters():
        assert p.grad is not None, k
        out.update(summarise("grad|" + k, p.grad))
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **out)
    print(f"{name}: loss={loss.item():.6f} matches={int((pred['matches0'] > -1).sum())} -> {path} "
          f"({os.path.getsize(path) / 1e6:.2f} MB)")


def _err_stats(prefix, got, ref):
    """rel. L2 error of `got` against the fp64 reference tensor `ref` (whole tensor)."""
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    return {prefix: np.array(((got - ref).norm() / ref.norm().clamp(min=1e-300)).item())}


def run_case_autocast(name, conf, B, N, M, seed):
    """How far does the UNMODIFIED reference itself move when it is run the way `train.py --mp bfloat16`
    runs it (train.py:468-472: fp32 module under torch.autocast(dtype=bfloat16))?  Both the fp64 run and the
    autocast run are the reference module on identical weights / inputs; the fixture stores, per output, per loss
    entry and per parameter gradient, the error of the autocast run against the fp64 run, measured exactly as
    tests/test_gpu_parity_bf16.py measures the CUDA bf16 path against the fp64 golden of the same case:
        whole-tensor rel. L2 for log_assignment / losses / small gradients,
        rel. L2 over the 512 probe entries (and the probe projection) for big gradient matrices.
    The CUDA bf16 path (bf16 operands, fp32 accumulate, fp32 residual stream) is required to be at least this
    close to fp64 -- the 'same autocast dtype' contract of SURVEY.md section 7, hard part 1(b)."""
    weights = synthetic.make_weights(conf, seed=seed)
    out = {"meta|B": np.array(B), "meta|N": np.array(N), "meta|M": np.array(M), "meta|seed": np.array(seed),
           "meta|conf": np.array(repr(conf)), "meta|autocast": np.array("cpu/bfloat16")}
    runs = {}
    for tag, dtype in (("f64", torch.float64), ("ac", torch.float32)):
        data = synthetic.make_pairs(B, N, seed=seed + 1, D=conf["input_dim"], M=M, dtype=dtype)
        model = build_reference(conf, weights, dtype)
        if tag == "ac":
            with torch.autocast("cpu", dtype=torch.bfloat16):
                pred = model(data)
                losses, _ = model.loss(pred, data)
                loss = losses["total"].mean()
        else:
            pred = model(data)
            losses, _ = model.loss(pred, data)
            loss = losses["total"].mean()
        loss.backward()
        runs[tag] = (pred, losses, {k: p.grad.detach().double() for k, p in model.named_parameters()})
    (p64, l64, g64), (pac, lac, gac) = runs["f64"], runs["ac"]
    la64, laac = p64["log_assignment"].detach().double(), pac["log_assignment"].detach().double()
    out.update(_err_stats("err|log_assignment", laac, la64))
    out["err|log_assignment_maxabs"] = np.array((laac - la64).abs().max().item())
    inner64, innerac = la64[:, :-1, :-1], laac[:, :-1, :-1]
    top2 = inner64.topk(2, dim=2).values
    margin = top2[..., 0] - top2[..., 1]
    agree = innerac.max(2).indices == inner64.max(2).indices
    out["idx|row_agree_frac"] = np.array(agree.double().mean().item())
    # smallest margin above which the autocast reference keeps every row argmax
    out["idx|row_safe_margin"] = np.array(margin[~agree].max().item() if (~agree).any() else 0.0)
    out["idx|matches0_agree_frac"] = np.array((pac["matches0"] == p64["matches0"]).double().mean().item())
    for k in ["total", "last", "assignment_nll", "nll_pos", "nll_neg", "confidence", "row_norm"]:
        out.update(_err_stats("err|loss|" + k, lac[k], l64[k]))
    for k in g64:
        a, r = gac[k], g64[k]
        if r.numel() <= 4096:
            out.update(_err_stats("err|grad|" + k, a, r))
        else:
            idx = probe_index(r.numel())
            out.update(_err_stats("err|grad|" + k, a.reshape(-1)[idx], r.reshape(-1)[idx]))
        out["err|gradnorm|" + k] = np.array(abs(a.norm().item() - r.norm().item()) / max(r.norm().item(), 1e-300))
    path = os.path.join(OUT, "ac_" + name + ".npz")
    np.savez_compressed(path, **out)
    worst = max(float(v) for k_, v in out.items() if k_.startswith("err|grad|"))
    print(f"ac_{name}: log_assignment rel {float(out['err|log_assignment']):.3e} (max abs "
          f"{float(out['err|log_assignment_maxabs']):.3e}), loss rel {float(out['err|loss|total']):.3e}, worst grad rel "
          f"{worst:.3e}, row argmax agreement {float(out['idx|row_agree_frac']):.4f} -> {path}")


def run_heads():
    """Golden vectors for the two other assignment heads on the path."""
    from gluefactory.models.matchers.gluestick import log_double_softmax
    from gluefactory_nonfree.superglue import log_optimal_transport

    rs = np.random.RandomState(7)
    out = {}
    for tag, (B, M, N) in {"a": (2, 37, 53), "b": (1, 128, 96)}.items():
        sim = torch.from_numpy(rs.standard_normal((B, M, N)) * 3.0)
        bin_score = torch.tensor(0.7, dtype=torch.float64)
        out[f"{tag}|sim"] = sim.numpy()
        out[f"{tag}|lds"] = log_double_softmax(sim, bin_score).numpy()
        out[f"{tag}|lot"] = log_optimal_transport(sim, bin_score, 50).numpy()
    path = os.path.join(OUT, "heads.npz")
    np.savez_compressed(path, **out)
    print("heads ->", path)


def run_heads_grad():
    """Gradients of the two other assignment heads w.r.t. the similarity (and the bin / dustbin score), from the
    reference functions under autograd -- the fixtures the backward kernels of rows a15 / a16 will be held to."""
    from gluefactory.models.matchers.gluestick import log_double_softmax
    from gluefactory_nonfree.superglue import log_optimal_transport

    rs = np.random.RandomState(9)
    out = {}
    for tag, (B, M, N) in {"a": (2, 37, 53), "b": (1, 96, 80)}.items():
        sim0 = rs.standard_normal((B, M, N)) * 3.0
        w = torch.from_numpy(rs.standard_normal((B, M + 1, N + 1)))
        out[f"{tag}|sim"], out[f"{tag}|w"] = sim0, w.numpy()
        for name, fn in (("lds", lambda s_, b_: log_double_softmax(s_, b_)),
                         ("lot", lambda s_, b_: log_optimal_transport(s_, b_, 50))):
            sim = torch.from_numpy(sim0).requires_grad_()
            beta = torch.tensor(0.7, dtype=torch.float64, requires_grad=True)
            (fn(sim, beta) * w).sum().backward()
            out[f"{tag}|{name}|dsim"] = sim.grad.numpy()
            out[f"{tag}|{name}|dbin"] = beta.grad.numpy()
    path = os.path.join(OUT, "heads_grad.npz")
    np.savez_compressed(path, **out)
    print("heads_grad ->", path)


def run_gluestick_attention():
    """Golden vectors for the GlueStick attention core and its MultiHeadedAttention wrapper
    (models/matchers/gluestick.py:524-551; SURVEY 8a row a15): forward and all gradients in fp64."""
    from gluefactory.models.matchers.gluestick import MultiHeadedAttention, attention

    rs = np.random.RandomState(21)
    out = {}
    b, d, h, n, m = 1, 64, 4, 40, 56
    q = torch.from_numpy(rs.standard_normal((b, d, h, n))).requires_grad_()
    k = torch.from_numpy(rs.standard_normal((b, d, h, m))).requires_grad_()
    v = torch.from_numpy(rs.standard_normal((b, d, h, m))).requires_grad_()
    w = torch.from_numpy(rs.standard_normal((b, d, h, n)))
    o, _ = attention(q, k, v)
    (o * w).sum().backward()
    # the inputs q, k, v, w (and x, src, w2 below) are not stored: tests re-draw them from RandomState(21)
    out.update({"core|out": o.detach().numpy(), "core|dq": q.grad.numpy(), "core|dk": k.grad.numpy(),
                "core|dv": v.grad.numpy()})
    # module level: weights drawn from the seeded stream below (the test rebuilds them), gradients summarised
    b, n, m = 1, 40, 56
    mha = MultiHeadedAttention(4, 256).double()
    wrs = np.random.RandomState(22)
    with torch.no_grad():
        for name, p_ in mha.named_parameters():  # order: merge.weight, merge.bias, proj.{0,1,2}.{weight,bias}
            p_.copy_(torch.from_numpy(wrs.uniform(-1, 1, size=tuple(p_.shape)) / 16.0))
    x = torch.from_numpy(rs.standard_normal((b, 256, n))).requires_grad_()
    src = torch.from_numpy(rs.standard_normal((b, 256, m))).requires_grad_()
    w2 = torch.from_numpy(rs.standard_normal((b, 256, n)))
    y = mha(x, src, src)
    (y * w2).sum().backward()
    out.update({"mha|out": y.detach().numpy(), "mha|dx": x.grad.numpy(), "mha|dsrc": src.grad.numpy(),
                "mha|param_names": np.array([n_ for n_, _ in mha.named_parameters()])})
    for name, p_ in mha.named_parameters():
        out.update(summarise("mha|grad|" + name, p_.grad))
    path = os.path.join(OUT, "gluestick_attn.npz")
    np.savez_compressed(path, **out)
    print("gluestick attention ->", path)


def run_gt_homography():
    """Golden labels from the reference's own gt_matches_from_homography (geometry/gt_generation.py:109-161),
    imported with the kornia stand-in of oracle/_shim (the function itself never touches kornia)."""
    from gluefactory.geometry.gt_generation import gt_matches_from_homography

    out = {}
    for tag, (B, M, N, seed) in {"a": (2, 260, 300, 5), "b": (1, 513, 200, 6)}.items():
        d = synthetic.make_pairs(B, N, seed=seed, M=M, with_gt=False)
        kp0, kp1, H = d["keypoints0"], d["keypoints1"], d["H_0to1"]  # fp32, as the pipeline passes them
        r = gt_matches_from_homography(kp0, kp1, H, pos_th=3.0, neg_th=3.0)
        out.update({f"{tag}|kp0": kp0.numpy(), f"{tag}|kp1": kp1.numpy(), f"{tag}|H": H.numpy(),
                    f"{tag}|matches0": r["matches0"].numpy(), f"{tag}|matches1": r["matches1"].numpy(),
                    f"{tag}|positives": r["assignment"].nonzero().numpy(),
                    f"{tag}|proj_0to1": r["proj_0to1"].numpy(), f"{tag}|proj_1to0": r["proj_1to0"].numpy()})
    path = os.path.join(OUT, "gt_homography.npz")
    np.savez_compressed(path, **out)
    print("gt_homography ->", path)


def run_gluestick(name="gluestick_l4_n160", n_gnn=4, B=2, N=160, L=24, seed=31):
    """Forward + loss + backward of the UNMODIFIED reference GlueStick (models/matchers/gluestick.py) in fp64, train
    mode (BatchNorm batch statistics), on the synthetic points+lines batch: predictions, all loss entries, every
    parameter gradient (summarised) and the updated BatchNorm running statistics.  Weights come from
    synthetic.make_gluestick_weights over the PLUGIN's state_dict layout and are loaded strictly into the reference --
    which also proves the two module trees carry identical names and shapes."""
    from gluefactory.models import get_model
    from gluefactory_b200.matchers.gluestick import GlueStick as Plugin

    conf = {"GNN_layers": ["self", "cross"] * (n_gnn // 2), "filter_threshold": 0.2}
    # weights are drawn in fp32 (what the CUDA plugin holds) and evaluated by the reference in fp64
    sd = synthetic.make_gluestick_weights(Plugin(dict(conf)).state_dict(), seed=seed)
    model = get_model("matchers.gluestick")(dict(conf, name="matchers.gluestick")).double()
    assert list(model.state_dict().keys()) == list(sd.keys())
    model.load_state_dict({k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}, strict=True)
    model = model.train()
    data = synthetic.make_gluestick_batch(B, N, L, seed + 1, dtype=torch.float64)
    pred = model(data)
    losses, _ = model.loss(pred, data)
    losses["total"].mean().backward()
    out = {"meta|conf": np.array(repr(conf)), "meta|B": np.array(B), "meta|N": np.array(N), "meta|L": np.array(L),
           "meta|seed": np.array(seed)}
    for k in ["matches0", "matches1", "matching_scores0", "matching_scores1", "log_assignment", "line_matches0",
              "line_matches1", "line_matching_scores0", "line_log_assignment", "raw_line_scores"]:
        out["pred|" + k] = pred[k].detach().numpy()
    for k, v in losses.items():
        out["loss|" + k] = v.detach().numpy() if torch.is_tensor(v) else np.array(v)
    for k, p in model.named_parameters():
        assert p.grad is not None, k
        out.update(summarise("grad|" + k, p.grad))
    for k, v in model.state_dict().items():
        if "running_" in k:
            out["bn|" + k] = v.numpy()
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **out)
    print(f"{name}: loss={losses['total'].mean().item():.6f} point matches={int((pred['matches0'] > -1).sum())} "
          f"line matches={int((pred['line_matches0'] > -1).sum())} params={sum(p.numel() for p in model.parameters())} -> "
          f"{path} ({os.path.getsize(path) / 1e6:.2f} MB)")


def run_gt_pose_depth():
    """Golden labels from the reference's own gt_matches_from_pose_depth (geometry/gt_generation.py:13-106) with its
    Camera / Pose wrappers, for th_epi None / 5 and th_consistency None / 3: stores the inputs of the O(M N) pass
    (reprojections and masks, as the reference computed them) and its outputs."""
    from gluefactory.geometry.gt_generation import gt_matches_from_pose_depth
    from gluefactory.geometry.wrappers import Camera, Pose

    out = {}
    for tag, (B, M, N, seed, epi, cc) in {"a": (2, 300, 260, 61, None, None), "b": (1, 513, 640, 62, 5.0, None),
                                          "c": (2, 200, 333, 63, 5.0, 3.0)}.items():
        sc = synthetic.pose_depth_scene(B, M, N, seed)
        data = {"view0": {"camera": Camera.from_calibration_matrix(sc["K0"]), "depth": sc["depth0"]},
                "view1": {"camera": Camera.from_calibration_matrix(sc["K1"]), "depth": sc["depth1"]},
                "T_0to1": Pose.from_Rt(sc["R"], sc["t"])}
        r = gt_matches_from_pose_depth(sc["kp0"], sc["kp1"], data, pos_th=3.0, neg_th=5.0, epi_th=epi, cc_th=cc)
        out[f"{tag}|meta"] = np.array([B, M, N, seed, -1 if epi is None else epi, -1 if cc is None else cc], dtype=np.float64)
        for k in ("matches0", "matches1", "proj_0to1", "proj_1to0", "visible0", "visible1", "depth_keypoints0",
                  "depth_keypoints1"):
            out[f"{tag}|{k}"] = r[k].numpy()
        out[f"{tag}|positives"] = r["assignment"].nonzero().numpy()
        from gluefactory.geometry.depth import sample_depth
        out[f"{tag}|valid0"] = sample_depth(sc["kp0"], sc["depth0"])[1].numpy()
        out[f"{tag}|valid1"] = sample_depth(sc["kp1"], sc["depth1"])[1].numpy()
        print(f"gt_pose_depth {tag}: positives={int(r['assignment'].sum())} unmatched0={int((r['matches0'] == -1).sum())} "
              f"ignored0={int((r['matches0'] == -2).sum())}")
    path = os.path.join(OUT, "gt_pose_depth.npz")
    np.savez_compressed(path, **out)
    print("gt_pose_depth ->", path, f"({os.path.getsize(path) / 1e6:.2f} MB)")


def run_adaptive():
    """Inference-time point pruning (lightglue.py:461-526, 545-558; SURVEY 8f row 4) of the unmodified reference in
    eval mode, fp32 (its pruning branch mixes default-dtype buffers with the model dtype, so fp64 fails).  The seed is
    chosen so that every pruning decision clears its threshold by a margin (checked below), i.e. the fixture does not
    hinge on fp32 rounding.  Early stopping is not recorded: the reference cannot take that branch without crashing
    (`torch.stack` of the empty `all_desc0` list after the `break`, lightglue.py:485-492, 533)."""
    from gluefactory.models import get_model

    conf = dict(synthetic.DEFAULT_CONF, n_layers=5, width_confidence=0.6, depth_confidence=-1, filter_threshold=0.0)
    N, M = 224, 200
    for seed in range(70, 90):
        w = synthetic.make_weights(conf, seed=seed)
        model = get_model("matchers.lightglue")(dict(conf, name="matchers.lightglue"))
        model.load_state_dict(w, strict=False)
        model = model.eval()
        data = synthetic.make_pairs(1, N, seed=seed + 1, M=M)
        margins = []
        orig = model.get_pruning_mask

        def spy(confidences, scores, layer_index, _orig=orig):
            margins.append((scores - (1 - conf["width_confidence"])).abs().min().item())
            return _orig(confidences, scores, layer_index)
        model.get_pruning_mask = spy
        with torch.no_grad():
            pred = model(data)
        kept = pred["log_assignment"].shape[1] - 1
        if min(margins) > 2e-4 and 20 < kept < M - 20:
            break
    else:
        raise RuntimeError("no seed with comfortable pruning margins")
    out = {"meta|conf": np.array(repr(conf)), "meta|seed": np.array(seed), "meta|M": np.array(M), "meta|N": np.array(N),
           "meta|min_margin": np.array(min(margins))}
    for k in ["matches0", "matches1", "matching_scores0", "matching_scores1", "prune0", "prune1", "log_assignment"]:
        out["pred|" + k] = pred[k].numpy()
    path = os.path.join(OUT, "adaptive_prune.npz")
    np.savez_compressed(path, **out)
    print(f"adaptive_prune: seed={seed} kept0={kept} kept1={pred['log_assignment'].shape[2] - 1} min margin={min(margins):.2e} "
          f"matches={int((pred['matches0'] > -1).sum())} -> {path}")


def run_eval_loss():
    """Validation-mode loss of the reference (train.py:92-93 do_evaluation: model.eval(), loss on the last layer only,
    lightglue.py:485 keeps one stacked layer and :588 uses log_assignment[-1]) + the matcher metrics."""
    conf = dict(synthetic.DEFAULT_CONF, n_layers=3, filter_threshold=0.1)
    B, N, seed = 2, 160, 13
    weights = synthetic.make_weights(conf, seed=seed)
    data = synthetic.make_pairs(B, N, seed=seed + 1, D=conf["input_dim"], dtype=torch.float64)
    model = build_reference(conf, weights, torch.float64).eval()
    with torch.no_grad():
        pred = model(data)
        losses, metrics = model.loss(pred, data)
    out = {"meta|conf": np.array(repr(conf)), "meta|B": np.array(B), "meta|N": np.array(N), "meta|M": np.array(N),
           "meta|seed": np.array(seed)}
    for k, v in losses.items():
        out["loss|" + k] = v.detach().cpu().numpy() if torch.is_tensor(v) else np.array(v)
    for k, v in metrics.items():
        out["metric|" + k] = v.detach().cpu().numpy()
    path = os.path.join(OUT, "eval_loss.npz")
    np.savez_compressed(path, **out)
    print("eval_loss ->", path, {k: v for k, v in out.items() if k.startswith("loss|total")})


def run_dropin_surface():
    """What a drop-in replacement of the reference's LightGlue matcher and homography ground-truth component must
    reproduce (models/matchers/lightglue.py, models/matchers/homography_matcher.py): the matcher's state_dict names,
    shapes and confidence thresholds at n_layers=2, and the ground-truth component's default_conf and
    required_data_keys."""
    from gluefactory.models import get_model

    lg = get_model("matchers.lightglue")({"n_layers": 2})
    gt = get_model("matchers.homography_matcher")
    out = {"lightglue|keys": np.array(list(lg.state_dict().keys())),
           "lightglue|confidence_thresholds": lg.confidence_thresholds.numpy(),
           "homography|required_data_keys": np.array(sorted(gt({}).required_data_keys)),
           "homography|default_conf": np.array(repr(dict(gt.default_conf)))}
    for k, v in lg.state_dict().items():
        out["lightglue|shape|" + k] = np.array(tuple(v.shape), dtype=np.int64)
    path = os.path.join(OUT, "dropin_surface.npz")
    np.savez_compressed(path, **out)
    print("dropin_surface ->", path)


def run_autocast_cases():
    torch.manual_seed(0)
    mid = dict(synthetic.DEFAULT_CONF, n_layers=3, filter_threshold=0.1)
    run_case_autocast("lg_d256_l3_n160", mid, B=2, N=160, M=160, seed=13)
    disk = dict(synthetic.DEFAULT_CONF, n_layers=2, input_dim=128)
    run_case_autocast("lg_disk_d256_l2_n128", disk, B=1, N=128, M=128, seed=14)
    run_case_autocast("lg_full_l9_n512", dict(synthetic.DEFAULT_CONF), B=1, N=512, M=512, seed=15)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    only = [a for a in sys.argv[1:] if not a.startswith("-")]  # single fixtures: gluestick_attn, gt_homography, heads_grad
    if only:
        for name in only:
            {"gluestick_attn": run_gluestick_attention, "gt_homography": run_gt_homography,
             "heads_grad": run_heads_grad, "autocast": run_autocast_cases, "eval_loss": run_eval_loss, "gluestick": run_gluestick, "gt_pose_depth": run_gt_pose_depth, "adaptive": run_adaptive,
             "dropin": run_dropin_surface,
             "sift": lambda: run_case("lg_sift_d256_l2_n96", dict(synthetic.DEFAULT_CONF, n_layers=2, input_dim=128,
                                                                  add_scale_ori=True), B=1, N=96, M=80, seed=16)}[name]()
        sys.exit(0)
    torch.manual_seed(0)
    torch.set_num_threads(8)
    small = dict(synthetic.DEFAULT_CONF, descriptor_dim=128, input_dim=128, num_heads=2, n_layers=2)
    run_case("lg_small_d128_l2_n96", small, B=2, N=96, M=96, seed=11)
    run_case("lg_small_d128_l2_m80_n112", small, B=2, N=112, M=80, seed=12)
    mid = dict(synthetic.DEFAULT_CONF, n_layers=3, filter_threshold=0.1)
    run_case("lg_d256_l3_n160", mid, B=2, N=160, M=160, seed=13)
    disk = dict(synthetic.DEFAULT_CONF, n_layers=2, input_dim=128)
    run_case("lg_disk_d256_l2_n128", disk, B=1, N=128, M=128, seed=14)
    run_case("lg_sift_d256_l2_n96", dict(synthetic.DEFAULT_CONF, n_layers=2, input_dim=128, add_scale_ori=True), B=1, N=96, M=80, seed=16)
    full = dict(synthetic.DEFAULT_CONF)
    run_case("lg_full_l9_n512", full, B=1, N=512, M=512, seed=15, sub=8)
    run_heads()
    run_heads_grad()
    run_gluestick_attention()
    run_gt_homography()
    run_autocast_cases()
    run_eval_loss()
    run_gluestick()
    run_gt_pose_depth()
    run_adaptive()
    run_dropin_surface()
