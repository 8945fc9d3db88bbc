"""CPU-side checks of the host mirror: state-dict key compatibility with the reference's ckpt.pth
format, the C-ABI library loads and exports every symbol the header declares, and the product path
refuses to run without CUDA (no CPU fallback)."""
import os
import re

import pytest
import torch

from tests.test_oracle_golden import CASES, ORACLE_ONLY, load_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from qdiff_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "qdiff_b200.h")).read()
    declared = set(re.findall(r"\b(qd_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    L = _lib.lib()
    for name in sorted(declared):
        assert hasattr(L, name), f"{name} declared in include/qdiff_b200.h but not exported"
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)


def test_ctypes_mirror_matches_the_header_layout(tmp_path):
    """sizeof / offsetof of every descriptor as the C compiler sees include/qdiff_b200.h == the ctypes mirror."""
    import ctypes as C
    import shutil
    import subprocess
    from qdiff_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    pairs = {"qd_qparams": _lib.QParams, "qd_gemm_desc": _lib.GemmDesc, "qd_quantize_desc": _lib.QuantizeDesc,
             "qd_groupnorm_desc": _lib.GroupNormDesc, "qd_layernorm_desc": _lib.LayerNormDesc,
             "qd_im2col_desc": _lib.Im2colDesc, "qd_attention_desc": _lib.AttentionDesc,
             "qd_sampler_desc": _lib.SamplerDesc, "qd_misc_desc": _lib.MiscDesc}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{os.path.join(ROOT, "include", "qdiff_b200.h")}"',
             'int main(void) {']
    for cname, cls in pairs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-o", str(exe), str(src)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, cls in pairs.items():
        assert int(out[cname]) == C.sizeof(cls), (cname, out[cname], C.sizeof(cls))
        for fname, _ in cls._fields_:
            assert int(out[f"{cname}.{fname}"]) == getattr(cls, fname).offset, (cname, fname)


@pytest.mark.parametrize("name", CASES + ORACLE_ONLY)
def test_checkpoint_keys_roundtrip(name):
    """Wrapping our containers + resume_cali_model must consume exactly the reference's checkpoint keys."""
    from tests.test_unet_gpu import build_qnn
    g = load_case(name)
    qnn = build_qnn(g, torch.device("cpu"))
    mods = dict(qnn.named_modules())
    n_split = sum(1 for k in g["ckpt"] if k.endswith("weight_quantizer_0.delta"))
    assert sum(1 for m in mods.values() if type(m).__name__ == "QuantModule" and m.split) == n_split
    # quantizer values landed where the graph builder reads them
    for k, v in g["ckpt"].items():
        if k.endswith(".act_quantizer.delta"):
            q = mods[k[:-len(".delta")]]
            assert float(q.delta) == float(v) and q.inited


def test_forward_without_cuda_fails_loudly():
    from tests.test_unet_gpu import build_qnn
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    g = load_case("ddim_w4a8_split")
    qnn = build_qnn(g, torch.device("cpu"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        qnn(g["x"], g["t"])
    with pytest.raises(RuntimeError):
        qnn.model.conv_in(g["x"])


def test_pack_int4_roundtrip_and_limits():
    """ops.pack_int4: unsigned nibbles + per-row zero point reproduce the zero-point-free codes; rows that do not fit
    4 bits (W8 layers) are refused so the builder falls back to the s8 layout."""
    from qdiff_b200 import ops
    gen = torch.Generator().manual_seed(3)
    ws = torch.randint(0, 16, (37, 96), generator=gen) - torch.randint(0, 16, (37, 1), generator=gen)
    packed, zero = ops.pack_int4(ws)
    assert packed.dtype == torch.uint8 and packed.shape == (37, 48) and zero.dtype == torch.int8
    assert int(zero.min()) >= 0 and int(zero.max()) <= 15
    assert torch.equal(ops.unpack_int4(packed, zero), ws.to(torch.int16))
    # nibble order: byte j of a 4-byte word = code[j] | code[4 + j] << 4 (what the unpack warps of the GEMM assume)
    wq0 = (ws[0, :8] + zero[0]).to(torch.int64)
    assert [int(b) for b in packed[0, :4]] == [int(wq0[j] | (wq0[4 + j] << 4)) for j in range(4)]
    assert ops.pack_int4(torch.randint(-128, 128, (4, 32), generator=gen)) is None     # 8-bit rows
    assert ops.pack_int4(torch.zeros(4, 36, dtype=torch.int64)) is None                 # K not a multiple of 8


def test_groupnorm_workspace_rule_is_owned_by_the_library():
    from qdiff_b200 import ops
    small = ops.gn_workspace_floats(16, 64, 1280)
    big = ops.gn_workspace_floats(16, 4096, 320)
    assert 0 < small < big
    # partial sums: doubles [B][nslab][groups][2] with nslab >= HW/64, + stats
    assert big >= 16 * (4096 // 64) * 32 * 2 * 2 + 16 * 32 * 2
    assert ops.gn_workspace_floats(0, 64, 64) == 0
