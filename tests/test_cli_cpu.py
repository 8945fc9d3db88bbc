"""The command-line surface of scripts/{sample_diffusion_ddim,sample_diffusion_ldm,txt2img}.py must equal the
reference's (names, short options, defaults, types, nargs, choices, required, action): tests/golden/cli_surface.json was
extracted from the reference's sources by tools/make_cli_golden.py (AST walk; the scripts themselves need packages that
do not exist offline).  Reference: sample_diffusion_ddim.py:350-477, sample_diffusion_ldm.py:191-349, txt2img.py:107-331."""
import json
import os

import pytest

from qdiff_b200 import cli

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cli_surface.json")
PARSERS = {"ddim": cli.ddim_parser, "ldm": cli.ldm_parser, "txt2img": cli.txt2img_parser}
ACTION = {"_StoreAction": "store", "_StoreTrueAction": "store_true"}


def _norm_ours(s):
    return {k: dict(v, action=ACTION.get(v["action"], v["action"])) for k, v in s.items()}


@pytest.mark.parametrize("which", sorted(PARSERS))
def test_flags_match_reference(which):
    ref = json.load(open(GOLD))[which]
    ours = _norm_ours(cli.surface(PARSERS[which]()))
    missing = sorted(set(ref) - set(ours))
    assert not missing, f"flags of the reference script that are missing: {missing}"
    for dest, r in ref.items():
        o = ours[dest]
        for field in ("flags", "default", "type", "nargs", "choices", "required", "action"):
            assert o[field] == r[field], (which, dest, field, o[field], r[field])
    extra = sorted(set(ours) - set(ref))
    assert all(e.startswith("b200_") for e in extra), f"non-reference flags must carry the b200_ prefix: {extra}"


def test_reference_command_lines_parse():
    """The README command lines of the reference (SURVEY section 0) parse into the expected settings."""
    a = cli.ddim_parser().parse_args("--config configs/cifar10.yml --use_pretrained --timesteps 100 --eta 0 --skip_type quad "
                                     "--ptq --weight_bit 4 --quant_mode qdiff --split --resume -l out --cali_ckpt c.pth "
                                     "--quant_act --act_bit 8 --a_sym".split())
    assert (a.weight_bit, a.act_bit, a.split, a.a_sym, a.resume, a.skip_type, a.timesteps) == (4, 8, True, True, True, "quad", 100)
    b = cli.ldm_parser().parse_args("-r models/ldm/lsun_beds256/model.ckpt -n 20 --batch_size 10 -c 200 -e 1.0 --seed 41 "
                                    "--ptq --weight_bit 4 --quant_mode qdiff --quant_act --resume --cali_ckpt c.pth -l o".split())
    assert (b.custom_steps, b.eta, b.n_samples, b.batch_size, b.seed) == (200, 1.0, 20, 10, 41)
    c = cli.txt2img_parser().parse_args(["--prompt", "a puppy", "--plms", "--cond", "--ptq", "--weight_bit", "4",
                                         "--quant_mode", "qdiff", "--no_grad_ckpt", "--split", "--n_samples", "5",
                                         "--quant_act", "--act_bit", "8", "--sm_abit", "16", "--resume", "--cali_ckpt", "c.pth"])
    assert (c.plms, c.sm_abit, c.scale, c.ddim_steps, c.H // c.f, c.quant_mode) == (True, 16, 7.5, 50, 64, "qdiff")
    with pytest.raises(SystemExit):       # quirk Q5: the reference's default quant_mode is not a valid choice either way
        cli.txt2img_parser().parse_args(["--quant_mode", "symmetric"])


def test_scripts_refuse_what_is_out_of_scope():
    a = cli.ldm_parser().parse_args("--seed 1 --ptq --quant_act".split())
    with pytest.raises(SystemExit, match="calibration is not part of the sampling hot path"):
        cli._require_resume(a)
    b = cli.ldm_parser().parse_args("--seed 1".split())
    with pytest.raises(SystemExit, match="--ptq"):
        cli._require_resume(b)
