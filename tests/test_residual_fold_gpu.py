"""conv2 of a block with a 1x1 shortcut computes that shortcut itself, in a second tensor-memory accumulator, on the 32- and
64-channel layers.  SKB_UNFUSED_SHORTCUT=1 (read once per process -> subprocesses) runs the shortcut as its own launch
through a 16-bit buffer instead.  conv2 rounds the folded shortcut exactly as that buffer stores it, so everything must agree
bit for bit: embeddings, the activations after every block with a shortcut, and the fp16 range guard."""
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
out = {}
with torch.no_grad():
    m = make_xtractor(archi, 32, 256, compute_dtype=dtype).cuda()
    sets = {
        "one": [(16000, 1)],
        "mixed": [(16000, 2), (9000, 3), (40321, 4), (8000, 5), (25000, 6)],
        # fewer pixels than one conv tile on the deep levels (the shortest has no frame left after pooling: NaN by design)
        "short": [(800, 7), (1200, 8), (3000, 9)],
    }
    for name, spec in sets.items():
        ws = [synth.synth_wave(1, L, seed=s)[0].cuda() for L, s in spec]
        out[name] = m.extract_varlen(ws).cpu()
        out[name + "/solo"] = torch.cat([m.extract_varlen([w]) for w in ws]).cpu()
    ws = [synth.synth_wave(1, L, seed=s)[0].cuda() for L, s in sets["mixed"]]
    if archi == "halfresnet34":
        for st in ("layer1.0", "layer2.0", "layer3.0", "layer4.0"):
            out["stage/" + st] = m.debug_stage(ws, st).cpu()
    lib = _lib.lib()
    n0 = lib.skb_kernel_launches()
    m.extract_varlen(ws)
    torch.cuda.synchronize()
    out["launches"] = lib.skb_kernel_launches() - n0
    # fp16 range guard: a shortcut whose outputs saturate must be reported whichever path computes it.  Its BN shift goes
    # to 1e5 (every output beyond 65504) while the folded weights stay in range: scaled weights that themselves overflow
    # fp16 make the accumulators inf / NaN, which the guard does not see on either path.
    sd = m.state_dict()
    first = sorted(k for k in sd if k.endswith(".shortcut.1.bias"))[0]
    sd[first] += 1e5
    m.load_state_dict(sd)
    try:
        m.extract_varlen(ws)
        out["overflow"] = False
    except OverflowError:
        out["overflow"] = True
torch.save(out, path)
print("fold ok")
"""


def _run(tmp_path, archi, dtype, env):
    path = os.path.join(tmp_path, "%s_%s_%d.pt" % (archi, dtype, len(env)))
    r = subprocess.run([sys.executable, "-c", CODE, archi, dtype, path], cwd=ROOT, env=dict(os.environ, **env),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "fold ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
    return torch.load(path)


@pytest.mark.parametrize("archi,dtype,folded", [("halfresnet34", "fp16", 2), ("halfresnet34", "bf16", 2),
                                                ("resnet34", "fp16", 0), ("fastresnet34", "bf16", 2)])
def test_folded_shortcut_equals_the_standalone_launch(tmp_path, archi, dtype, folded):
    fold = _run(tmp_path, archi, dtype, {})
    ref = _run(tmp_path, archi, dtype, {"SKB_UNFUSED_SHORTCUT": "1"})
    bits = lambda t: t.contiguous().view(torch.int32)                      # bit for bit, NaN included
    for k, v in ref.items():
        if isinstance(v, torch.Tensor):
            assert torch.equal(bits(fold[k]), bits(v)), k
    assert torch.isfinite(ref["mixed"]).all()
    for name in ("one", "mixed", "short"):
        assert torch.equal(bits(fold[name]), bits(fold[name + "/solo"])), name          # packing invariance
    assert fold["overflow"] == ref["overflow"] == (dtype == "fp16")
    # one launch less per folded shortcut (layer1.0 and layer2.0 of halfresnet34; resnet34's 128-channel levels keep theirs)
    assert ref["launches"] - fold["launches"] == folded
