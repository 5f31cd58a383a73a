"""Grouped 3x3 conv on maps 64 or 128 wide (k_gconv3x3_tapn: the three horizontal taps stacked along N, the one-pixel shift in
the epilogue) vs fp32 PyTorch on the CPU, plus its determinism, batch invariance and agreement with the HEAL_TC_TAPN=0 paths."""
import os
import subprocess
import sys
import tempfile

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CASES = [
    # name, N, C, H, W: a unit is 128 pixels = 1 row at W 128, 2 rows at W 64
    ("w64_c128_n3_h37", 3, 128, 37, 64),      # odd H: the last unit's second row lies below the image; several segments
    ("w64_c256_n2_h1", 2, 256, 1, 64),        # one half-filled unit, fewer rows than the ring
    ("w64_c512_n5_h64", 5, 512, 64, 64),      # the pyramid's 64x64 level
    ("w128_c128_n2_h3", 2, 128, 3, 128),      # fewer rows than the ring
    ("w128_c256_n5_h33", 5, 256, 33, 128),    # ragged last segment
    ("w128_c512_n1_h130", 1, 512, 130, 128),  # 8 strips x many segments
]


def _conv(name, C, bias=True):
    gen = torch.Generator().manual_seed(abs(hash(name)) % 10000)
    conv = torch.nn.Conv2d(C, C, 3, padding=1, groups=32, bias=False)
    bnm = torch.nn.BatchNorm2d(C, eps=1e-5).eval() if bias else None
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=gen) * (1.0 / (C // 32 * 9)) ** 0.5)
        if bnm is not None:
            bnm.weight.copy_(torch.rand(C, generator=gen) + 0.5)
            bnm.bias.copy_(torch.randn(C, generator=gen) * 0.1)
            bnm.running_mean.copy_(torch.randn(C, generator=gen) * 0.1)
            bnm.running_var.copy_(torch.rand(C, generator=gen) + 0.5)
    return conv, bnm, gen


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("planes", [2, 1], ids=["tc32", "bf16"])
@pytest.mark.parametrize("relu", [True, False], ids=["relu", "linear"])
def test_grouped_tapn(case, planes, relu):
    """Against fp32 PyTorch; input read from a channel slice of a wider tensor and output written into a channel slice of a wider
    buffer whose neighbours must stay untouched."""
    from heal_b200 import ops
    name, N, C, H, W = case
    conv, bnm, gen = _conv(name, C)
    x = torch.randn(N, C, H, W, generator=gen)
    with torch.no_grad():
        y = bnm(conv(x))
        if relu:
            y = F.relu(y)
    fmt = "split" if planes == 2 else "bf16"
    pc = ops.pack_conv_tc(conv, bnm, relu, planes=2).to("cuda")
    xs = ops.convert(ops.to_act(x.cuda()), fmt)
    o, _ = ops.conv2d_tc(xs, pc)
    wide = torch.cat([torch.randn(N, 64, H, W, generator=gen), x, torch.randn(N, 64, H, W, generator=gen)], dim=1)
    xw = ops.convert(ops.to_act(wide.cuda()), fmt)
    buf = torch.zeros((planes, N, H, W, C + 128), dtype=torch.bfloat16, device="cuda")
    ops.conv2d_tc(xw, pc, out=ops.Act(buf, fmt), out_coffset=64, in_coffset=64)
    torch.cuda.synchronize()
    got = ops.act_to_nchw(o).cpu()
    scale = max(y.abs().max().item(), 1.0)
    err = (got - y).abs().max().item()
    print(f"{name} planes={planes} relu={relu}: max|y|={scale:.3f} err={err:.3e}")
    assert err < (1e-3 if planes == 2 else 1.4e-2 * scale)
    assert torch.equal(buf[..., 64:64 + C], o.t) and torch.all(buf[..., :64] == 0) and torch.all(buf[..., 64 + C:] == 0)


@pytest.mark.parametrize("W", [64, 128])
@pytest.mark.parametrize("planes", [2, 1], ids=["tc32", "bf16"])
def test_grouped_tapn_deterministic_and_batch_invariant(W, planes):
    """Bitwise: two calls agree, and image i of an N-image call equals that image run alone (the segment grid differs)."""
    from heal_b200 import ops
    N, C, H = 4, 256, 29
    conv, bnm, gen = _conv(f"inv{W}", C)
    x = torch.randn(N, C, H, W, generator=gen)
    fmt = "split" if planes == 2 else "bf16"
    pc = ops.pack_conv_tc(conv, bnm, True, planes=2).to("cuda")
    xs = ops.convert(ops.to_act(x.cuda()), fmt)
    a, _ = ops.conv2d_tc(xs, pc)
    b, _ = ops.conv2d_tc(xs, pc)
    singles = [ops.conv2d_tc(ops.convert(ops.to_act(x[i:i + 1].cuda()), fmt), pc)[0] for i in range(N)]
    torch.cuda.synchronize()
    assert torch.equal(a.t, b.t)
    for i in range(N):
        assert torch.equal(a.t[:, i], singles[i].t[:, 0]), i


def test_grouped_tapn_runs_the_kernel():
    from heal_b200 import ops
    conv, bnm, gen = _conv("prof", 128)
    xs = ops.convert(ops.to_act(torch.randn(1, 128, 8, 64, generator=gen).cuda()), "split")
    pc = ops.pack_conv_tc(conv, bnm, True, planes=2).to("cuda")
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        ops.conv2d_tc(xs, pc)
        torch.cuda.synchronize()
    assert any("k_gconv3x3_tapn" in e.key for e in prof.key_averages())


def test_grouped_tapn_equals_previous_path():
    """HEAL_TC_TAPN=0 (row ring at W 128, tile kernel at W 64) in a child process: same results within the fp32-equivalent
    tolerance (the horizontal taps are summed in a different order, so not bit for bit)."""
    code = (
        "import sys, torch\n"
        "from heal_b200 import ops\n"
        "g = torch.Generator().manual_seed(11)\n"
        "outs = []\n"
        "for C, H, W in ((512, 21, 64), (256, 13, 128)):\n"
        "    conv = torch.nn.Conv2d(C, C, 3, padding=1, groups=32, bias=False)\n"
        "    conv.weight.data.copy_(torch.randn(conv.weight.shape, generator=g) / (C // 32 * 9) ** 0.5)\n"
        "    x = torch.randn(2, C, H, W, generator=g)\n"
        "    pc = ops.pack_conv_tc(conv, None, True, planes=2).to('cuda')\n"
        "    o, _ = ops.conv2d_tc(ops.convert(ops.to_act(x.cuda()), 'split'), pc)\n"
        "    outs.append(ops.act_to_nchw(o).cpu())\n"
        "torch.cuda.synchronize()\n"
        "torch.save(outs, sys.argv[1])\n")
    res = []
    with tempfile.TemporaryDirectory() as td:
        for tapn in ("1", "0"):
            path = os.path.join(td, f"o{tapn}.pt")
            env = dict(os.environ, HEAL_TC_TAPN=tapn, PYTHONPATH=ROOT)
            subprocess.run([sys.executable, "-c", code, path], check=True, env=env, timeout=300, cwd=ROOT)
            res.append(torch.load(path))
    for new, old in zip(*res):
        err = (new - old).abs().max().item()
        print(f"tapn vs previous path: max|y|={old.abs().max().item():.3f} err={err:.3e}")
        assert err < 1e-4 * max(old.abs().max().item(), 1.0)
