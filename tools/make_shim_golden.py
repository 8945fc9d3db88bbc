"""Golden trace of the reference's PLMSSampler / DDIMSampler driving qdiff_b200.ldm_shim.LatentDiffusionShim, produced by
RUNNING THE REFERENCE's sampler code (imported read-only, see tools/make_golden.py) over a recording proxy of the shim
around the toy eps-model of tools/make_sampler_golden.py.  Build container only; the fixture is committed.

    python tools/make_shim_golden.py      -> tests/golden/shim_sampler_trace.pt

The trace holds every attribute the samplers read from the model (with its value; both samplers read the same ones)
and the inputs of every apply_model call, stacked per sampler; each call's answer was toy_eps of its inputs, which is
checked here.  The samplers are deterministic given those answers (DDIM's noise draws are replayed from
tests/golden/samplers.pt), so a shim that gives the same answers makes them reproduce the same results; the run recorded
here is checked against samplers.pt before the trace is written.
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "q-diffusion_b200")]
from tools.make_golden import OUT, _import_reference  # noqa: E402
from tools.make_sampler_golden import toy_eps  # noqa: E402


def _clone(v):
    if isinstance(v, torch.Tensor):
        return v.detach().clone()
    if isinstance(v, torch.device):
        return str(v)
    if isinstance(v, (list, tuple)):
        return type(v)(_clone(u) for u in v)
    if isinstance(v, dict):
        return {k: _clone(u) for k, u in v.items()}
    return v


def _same(a, b):
    return torch.equal(a, b) if isinstance(a, torch.Tensor) else a == b


def _stack(calls):
    """Inputs of the apply_model calls stacked along a new first axis; the conditioning is the same tensor every call."""
    for k in calls:
        assert torch.equal(k["out"], toy_eps(k["x"], k["t"], k["c"])) and torch.equal(k["c"], calls[0]["c"])
    return dict(x=torch.stack([k["x"] for k in calls]), t=torch.stack([k["t"] for k in calls]), c=calls[0]["c"])


class Recorder:
    """Forwards to the shim; records first reads of plain attributes and every apply_model call."""

    def __init__(self, shim):
        self._shim, self.attrs, self.calls = shim, {}, []

    def __getattr__(self, name):
        v = getattr(self._shim, name)
        if name == "apply_model":
            def apply_model(x, t, c, *a, **k):
                out = v(x, t, c, *a, **k)
                self.calls.append(dict(x=_clone(x), t=_clone(t), c=_clone(c), out=_clone(out)))
                return out
            return apply_model
        if name not in self.attrs:
            self.attrs[name] = _clone(v)
        return v


def main():
    _import_reference()
    from ldm.models.diffusion import ddim as ref_ddim
    from ldm.models.diffusion.plms import PLMSSampler
    from qdiff_b200.ldm_shim import LatentDiffusionShim

    class ToyUNet:
        def __call__(self, x, timesteps=None, context=None):
            return toy_eps(x, timesteps, context)

    class CpuPLMS(PLMSSampler):       # the reference's register_buffer moves everything to "cuda" (plms.py:19-23)
        def register_buffer(self, name, attr):
            setattr(self, name, attr)

    class CpuDDIM(ref_ddim.DDIMSampler):
        def register_buffer(self, name, attr):
            setattr(self, name, attr)

    g = torch.load(os.path.join(OUT, "samplers.pt"), map_location="cpu", weights_only=False)
    p = g["plms"]
    rec = Recorder(LatentDiffusionShim(ToyUNet(), "crossattn", 1000, p["linear_start"], p["linear_end"], device="cpu"))
    with torch.no_grad():
        out, _ = CpuPLMS(rec).sample(S=p["S"], batch_size=p["x_T"].shape[0], shape=tuple(p["x_T"].shape[1:]),
                                     conditioning=p["cond"], verbose=False, unconditional_guidance_scale=p["scale"],
                                     unconditional_conditioning=p["uc"], eta=0.0, x_T=p["x_T"])
    assert (out - p["out"]).abs().max().item() <= 2e-5 * max(1.0, p["out"].abs().max().item())
    trace = dict(linear_start=p["linear_start"], linear_end=p["linear_end"], attrs=rec.attrs, plms=_stack(rec.calls))

    d = g["ddim"]
    noises = list(d["noises"])
    real = ref_ddim.noise_like
    ref_ddim.noise_like = lambda shape, device, repeat=False: noises.pop(0)
    rec = Recorder(LatentDiffusionShim(ToyUNet(), "crossattn", 1000, d["linear_start"], d["linear_end"], device="cpu"))
    try:
        with torch.no_grad():
            out2, _ = CpuDDIM(rec).sample(S=d["S"], batch_size=d["x_T"].shape[0], shape=tuple(d["x_T"].shape[1:]),
                                          conditioning=d["cond"], verbose=False, unconditional_guidance_scale=d["scale"],
                                          unconditional_conditioning=d["uc"], eta=d["eta"], x_T=d["x_T"])
    finally:
        ref_ddim.noise_like = real
    assert (out2 - d["out"]).abs().max().item() <= 2e-5 * max(1.0, d["out"].abs().max().item())
    assert (d["linear_start"], d["linear_end"]) == (p["linear_start"], p["linear_end"])
    assert rec.attrs.keys() == trace["attrs"].keys()
    assert all(_same(rec.attrs[k], trace["attrs"][k]) for k in rec.attrs)
    trace["ddim"] = _stack(rec.calls)

    path = os.path.join(OUT, "shim_sampler_trace.pt")
    torch.save(trace, path)
    print(f"attributes read {sorted(trace['attrs'])}; apply_model calls: plms {len(trace['plms']['x'])}, "
          f"ddim {len(trace['ddim']['x'])}")
    print(f"{path}: {os.path.getsize(path) / 1e3:.1f} kB")


if __name__ == "__main__":
    main()
