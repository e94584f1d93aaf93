"""GlueStick (points + lines, BASELINE configs[4]) training step on one B200: the plugin (bf16 and fp32) against the
unmodified reference module from oracle/_ref in PyTorch eager on the same GPU (fp32 and bf16 autocast).
Forward + loss + backward + Adam, synthetic batch, N points and L lines per image."""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gluefactory_b200 import synthetic  # noqa: E402
from gluefactory_b200.matchers.gluestick import GlueStick  # noqa: E402

B, N, L = int(os.environ.get("PB", "8")), int(os.environ.get("PN", "2048")), int(os.environ.get("PL", "512"))
dev = torch.device("cuda", 0)
data = synthetic.to_device(synthetic.make_gluestick_batch(B, N, L, 5), dev)


def timed(step, reps=5, warm=2):
    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps * 1e3


def make_step(model, autocast=None):
    opt = torch.optim.Adam(model.parameters(), lr=1e-5)

    def step():
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=autocast, enabled=autocast is not None):
            pred = model(data)
            losses, _ = model.loss(pred, data)
            loss = losses["total"].mean()
        loss.backward()
        opt.step()
        return loss

    return step


conf = dict(GlueStick.default_conf) if hasattr(GlueStick, "default_conf") else {}
rows = []
w = None
for prec in ("bf16", "fp32"):
    m = GlueStick(dict(conf, precision=prec))
    if w is None:
        w = synthetic.make_gluestick_weights(m.state_dict(), seed=3)
    m.load_state_dict(w, strict=True)
    ms = timed(make_step(m.to(dev).train()))
    rows.append((f"plugin precision={prec}", ms))
    del m
try:  # the same step captured into one CUDA graph by the library's trainer (flat parameters, flat Adam)
    from gluefactory_b200.trainer import MatcherTrainer

    m = GlueStick(dict(conf, precision="bf16"))
    m.load_state_dict(w, strict=True)
    tr = MatcherTrainer(m.to(dev).train(), lr=1e-5)
    ms_eager = timed(lambda: tr.step(data))
    rows.append(("plugin bf16, MatcherTrainer eager", ms_eager))
    tr.capture(data, dev)
    rows.append(("plugin bf16, CUDA-graph replay", timed(lambda: tr.step_graphed(data))))
    del m, tr
except Exception as e:  # noqa: BLE001
    import traceback

    tb = [ln for ln in traceback.format_exc().splitlines() if "glue-factory_b200" in ln or "gluefactory_b200" in ln]
    print("graph capture failed:", type(e).__name__, str(e)[:200].replace("\n", " "), "|", " <- ".join(t.strip() for t in tb[-6:]))
    rows.append(("graph capture failed", float("nan")))
try:
    from oracle.stage_reference import import_reference

    get_model = import_reference()
    ref_conf = {k: v for k, v in conf.items() if k not in ("precision",)}
    for ac, tag in ((None, "fp32"), (torch.bfloat16, "bf16 autocast")):
        ref = get_model("matchers.gluestick")(dict(ref_conf, name="matchers.gluestick"))
        ref.load_state_dict(w, strict=True)
        ms = timed(make_step(ref.to(dev).train(), ac))
        rows.append((f"reference eager {tag}", ms))
        del ref
except Exception as e:  # noqa: BLE001
    rows.append((f"reference unavailable: {type(e).__name__}: {e}", float("nan")))
print(f"GlueStick training step, B={B} pairs, N={N} points, L={L} lines per image")
for name, ms in rows:
    print(f"  {name:32s} {ms:9.1f} ms/step  {B / ms * 1e3:8.1f} pairs/s")

if os.environ.get("PROF"):
    from torch.profiler import ProfilerActivity, profile

    m = GlueStick(dict(conf, precision="bf16"))
    m.load_state_dict(w, strict=True)
    step = make_step(m.to(dev).train())
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    evs = sorted(prof.key_averages(), key=lambda e: -e.device_time_total)
    tot = sum(e.device_time_total for e in evs)
    print(f"plugin bf16: total device time {tot / 1e3:.2f} ms over {sum(e.count for e in evs)} launches")
    for e in evs[:32]:
        print(f"  {e.device_time_total:9.0f} us {100 * e.device_time_total / tot:5.1f}% x{e.count:4d}  {e.key[:110]}")
