"""conv1's epilogue accumulates the squeeze-excitation channel totals of its output on every level: per thread on the 32-channel
layers, and with a transposed ownership (each epilogue warp re-reads its stored 32 x 16 block column-wise from shared memory)
on the 64-, 128- and 256-channel layers.  SKB_NO_FUSED_SUMS=1 (read once per process -> subprocesses) runs the separate
plane_sum pass on every level instead.  Both add the same 2^-15 fixed-point integers, so embeddings and block outputs must
agree bit for bit: with activations beyond 128 on the deep levels, with utterances shorter than a conv tile, with utterance
boundaries inside a 32-row block, whatever the packing, on every trunk that runs this forward."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CODE = r"""
import sys, torch
from sidekit_b200 import synth, _lib
from tests.models import make_xtractor

archi, dtype, path = sys.argv[1], sys.argv[2], sys.argv[3]
scaled = ("layer3.1", "layer4.0")
out = {}
with torch.no_grad():
    sets = {
        # lengths not aligned to anything: utterance boundaries fall at every offset inside the 32-row blocks
        "mixed": [(16000, 2), (9000, 3), (40321, 4), (8000, 5), (25000, 6), (4321, 7), (12345, 8), (6000, 9), (30017, 10)],
        # fewer pixels than one conv tile on the deep levels (the shortest has no frame left after pooling: NaN by design)
        "short": [(800, 11), (1200, 12), (3000, 13), (2600, 14), (5100, 15)],
    }
    ws = [synth.synth_wave(1, L, seed=s)[0].cuda() for L, s in sets["mixed"]]
    sd = make_xtractor(archi, 32, 256, compute_dtype=dtype).state_dict()
    blocks = sorted({k.split(".bn1.")[0][len("sequence_network."):] for k in sd if ".bn1." in k and ".layer" in k},
                    key=lambda n: (int(n[len("layer"):].split(".")[0]), int(n.split(".")[1])))

    def model():
        m = make_xtractor(archi, 32, 256, compute_dtype=dtype)
        m.load_state_dict(sd)
        return m.cuda()

    def y1max(m, st):
        # largest conv1 output of block st (what the totals add), recomputed in fp32 from the block input
        x = m.debug_stage(ws, blocks[blocks.index(st) - 1]).float().cpu()
        blk = dict(m.named_modules())["sequence_network." + st]
        bn = blk.bn1
        y1 = torch.nn.functional.conv2d(x, blk.conv1.weight.float().cpu(), stride=blk.conv1.stride, padding=1)
        y1 = torch.nn.functional.batch_norm(y1, bn.running_mean.cpu(), bn.running_var.cpu(), bn.weight.cpu(), bn.bias.cpu(), False, 0.0, bn.eps)
        return torch.relu(y1).max().item()

    # conv1 of one block on each of the two deepest levels scaled (bn1) so that its outputs peak at 160: beyond 128, and
    # far enough from the fp16 range that nothing after it saturates
    for st in scaled:
        s = 160.0 / y1max(model(), st)
        for k in ("weight", "bias"):
            sd["sequence_network.%s.bn1.%s" % (st, k)] *= s
    m = model()
    for st in scaled:
        out["y1max/" + st] = y1max(m, st)
        out["stage/" + st] = m.debug_stage(ws, st).cpu()
    for name, spec in sets.items():
        wl = [synth.synth_wave(1, L, seed=s)[0].cuda() for L, s in spec]
        out[name] = m.extract_varlen(wl).cpu()
        out[name + "/solo"] = torch.cat([m.extract_varlen([w]) for w in wl]).cpu()
        out[name + "/reversed"] = m.extract_varlen(wl[::-1]).flip(0).cpu()
    lib = _lib.lib()
    n0 = lib.skb_kernel_launches()
    m.extract_varlen(ws)
    torch.cuda.synchronize()
    out["launches"] = lib.skb_kernel_launches() - n0
    out["blocks"] = len(blocks)
torch.save(out, path)
print("totals ok")
"""


def _run(tmp_path, archi, dtype, env):
    path = os.path.join(tmp_path, "%s_%s_%d.pt" % (archi, dtype, len(env)))
    r = subprocess.run([sys.executable, "-c", CODE, archi, dtype, path], cwd=ROOT, env=dict(os.environ, **env),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "totals ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
    return torch.load(path)


@pytest.mark.parametrize("archi,dtype", [("halfresnet34", "fp16"), ("halfresnet34", "bf16"), ("resnet34", "fp16"),
                                         ("fastresnet34", "bf16")])
def test_channel_totals_in_conv1_equal_the_separate_pass(tmp_path, archi, dtype):
    fused = _run(tmp_path, archi, dtype, {})
    ref = _run(tmp_path, archi, dtype, {"SKB_NO_FUSED_SUMS": "1"})
    bits = lambda t: t.contiguous().view(torch.int32)                      # bit for bit, NaN included
    for k, v in ref.items():
        if isinstance(v, torch.Tensor):
            assert torch.equal(bits(fused[k]), bits(v)), k
    assert torch.isfinite(ref["mixed"]).all()
    for st in ("layer3.1", "layer4.0"):
        assert ref["y1max/" + st] > 128.0, (st, ref["y1max/" + st])          # the scaled conv1 outputs do reach beyond 128
    for name in ("mixed", "short"):
        for other in ("/solo", "/reversed"):
            assert torch.equal(bits(fused[name]), bits(fused[name + other])), name + other      # packing invariance
    # one plane_sum launch less per block: conv1 produces the totals on every level
    assert fused["blocks"] > 0 and ref["launches"] - fused["launches"] == fused["blocks"]
