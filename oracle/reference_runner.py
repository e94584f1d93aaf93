"""Drive the UNMODIFIED reference (installed under oracle/_ref by oracle/stage_reference.py) through its own public
API for the hot path: `TwoViewPipeline` with `extractor.name = None`, features supplied through `view*["cache"]`
(the cached-feature route, two_view_pipeline.py:62-70), `matcher.name = matchers.lightglue`, and the body of the
training loop restated from train.py:456-517 (zero_grad -> autocast(forward, loss) -> mean -> scaled backward ->
optimizer step).  BASELINE INFRASTRUCTURE ONLY: imported by bench.py's `--impl reference` / `gpu_eager_baseline`
legs and by tests; never by the product package.  `train.py` itself cannot be imported (h5py / kornia / matplotlib).
"""
import torch

from .stage_reference import import_reference


def available():
    return import_reference() is not None


def build_pipeline(conf, weights, device="cpu", checkpointed=False, flash=False):
    """conf: LightGlue conf (synthetic.DEFAULT_CONF keys); weights: state_dict under the reference names."""
    get_model = import_reference()
    assert get_model is not None, "reference not installed under oracle/_ref (run oracle/stage_reference.py)"
    matcher_conf = {k: v for k, v in conf.items() if k not in ("precision", "engine", "stack_ref_descriptors")}
    matcher_conf.update(name="matchers.lightglue", checkpointed=bool(checkpointed), flash=bool(flash))
    pipe = get_model("two_view_pipeline")({
        "extractor": {"name": None}, "matcher": matcher_conf, "ground_truth": {"name": None},
        "allow_no_extract": True,
    })
    missing, unexpected = pipe.matcher.load_state_dict({k: v.float() for k, v in weights.items()}, strict=False)
    assert not unexpected and missing in ([], ["confidence_thresholds"]), (missing, unexpected)
    return pipe.to(device).train()


def pipeline_batch(data):
    """Our flat synthetic batch -> the pipeline's input contract (features under view*["cache"], labels as gt_*)."""
    out = {k: v for k, v in data.items() if k.startswith("gt_") or k == "H_0to1"}
    for i in "01":
        out[f"view{i}"] = {"image_size": data[f"view{i}"]["image_size"],
                           "cache": {"keypoints": data[f"keypoints{i}"], "descriptors": data[f"descriptors{i}"]}}
    return out


class ReferenceTrainer:
    """train.py:347-367, 456-517 around the reference pipeline: Adam, optional autocast + GradScaler."""

    def __init__(self, pipe, lr=1e-4, mp_dtype=None):
        self.pipe = pipe
        self.loss_fn = pipe.loss
        self.opt = torch.optim.Adam([p for p in pipe.parameters() if p.requires_grad], lr=lr)
        self.mp_dtype = mp_dtype
        dev = next(pipe.parameters()).device
        self.device_type = dev.type
        self.scaler = torch.amp.GradScaler(self.device_type, enabled=mp_dtype is not None and dev.type == "cuda")

    def step(self, batch):
        self.pipe.train()
        self.opt.zero_grad()
        with torch.autocast(device_type=self.device_type, enabled=self.mp_dtype is not None, dtype=self.mp_dtype):
            pred = self.pipe(batch)
            losses, _ = self.loss_fn(pred, batch)
            loss = torch.mean(losses["total"])
        if torch.isnan(loss).any():
            return loss.detach()
        self.scaler.scale(loss).backward()
        self.scaler.step(self.opt)
        self.scaler.update()
        return loss.detach()
