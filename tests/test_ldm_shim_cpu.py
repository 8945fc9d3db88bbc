"""The LatentDiffusion surface (qdiff_b200/ldm_shim.py) is what the reference's sampler classes need: the reference's
UNMODIFIED PLMSSampler and DDIMSampler were run on top of the shim around a toy eps-model, reproducing the committed
reference results (tests/golden/samplers.pt), and every query they made of the shim is stored in
tests/golden/shim_sampler_trace.pt (tools/make_shim_golden.py); the shim must still answer each one the same way.  The
shim's apply_model / DiffusionWrapper dispatch is checked against ddpm.py:895-905,1426-1445 semantics."""
import os

import torch

from qdiff_b200.ldm_shim import LatentDiffusionShim
from tools.make_sampler_golden import toy_eps

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class ToyUNet:
    """Stands in for qdiff_b200.QuantModel: same call signature (x, timesteps, context=None)."""

    def __init__(self):
        self.calls = []

    def __call__(self, x, timesteps=None, context=None):
        self.calls.append(context)
        return toy_eps(x, timesteps, context)


def test_apply_model_dispatch():
    u = ToyUNet()
    m = LatentDiffusionShim(u, "crossattn", 1000, 0.00085, 0.012, device="cpu")
    x, t, c = torch.randn(2, 4, 8, 8), torch.tensor([5, 7]), torch.randn(2, 5, 16)
    ref = toy_eps(x, t, c)
    assert torch.equal(m.apply_model(x, t, c), ref)                       # tensor -> {'c_crossattn': [c]}
    assert torch.equal(m.apply_model(x, t, [c]), ref)
    assert torch.equal(m.apply_model(x, t, {"c_crossattn": [c]}), ref)
    assert u.calls[0] is c                                                # single context: the caller's tensor object is kept
    two = m.apply_model(x, t, {"c_crossattn": [c[:, :2], c[:, 2:]]})      # several contexts are concatenated on dim 1
    assert torch.allclose(two, ref)
    m0 = LatentDiffusionShim(ToyUNet(), None, device="cpu")
    assert torch.equal(m0.apply_model(x, t, None), toy_eps(x, t))
    assert m.model.diffusion_model is u and m.num_timesteps == 1000
    assert m.alphas_cumprod.dtype == torch.float32 and m.alphas_cumprod_prev[0] == 1.0


def test_reference_samplers_run_unchanged_on_the_shim():
    """The samplers are deterministic given the model's answers, so equal answers reproduce the recorded run."""
    g = torch.load(os.path.join(GOLD, "shim_sampler_trace.pt"), map_location="cpu", weights_only=False)
    for which in ("plms", "ddim"):
        u = ToyUNet()
        shim = LatentDiffusionShim(u, "crossattn", 1000, g["linear_start"], g["linear_end"], device="cpu")
        for name, v in g["attrs"].items():
            got = getattr(shim, name)
            if isinstance(v, torch.Tensor):
                assert got.dtype == v.dtype and torch.equal(got, v), (which, name)
            else:
                assert (str(got) if isinstance(got, torch.device) else got) == v, (which, name, got, v)
        tr = g[which]
        for k in range(len(tr["x"])):
            out = shim.apply_model(tr["x"][k], tr["t"][k], tr["c"])
            assert torch.equal(out, toy_eps(tr["x"][k], tr["t"][k], tr["c"])), (which, k)
            assert u.calls[-1] is tr["c"]
