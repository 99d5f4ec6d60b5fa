"""Where the squeeze-excitation channel totals cost time in one HalfResNet34 config-4 step, per setting:
  default               conv1's epilogue accumulates the totals on every level (no plane_sum launch)
  SKB_NO_FUSED_SUMS=1   the separate plane_sum pass after conv1 on every level

Each setting runs in its own process (the engine reads its switches once per process) through tools/residual_probe.py's
child, the same step (96 utterances of 2-20 s, ~1050 audio-s, fp16): step time from CUDA events with the profiler off, then
one step under torch.profiler.  Printed per level: conv1 time (sum and mean per launch), plane_sum time, and the launch
counts; then each setting's full kernel totals.  The device name and power limit head the report.

    python tools/se_totals_probe.py [--steps 20] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SETTINGS = [("fused", {}), ("separate", {"SKB_NO_FUSED_SUMS": "1"})]
LEVEL_BLOCKS = (3, 4, 6, 3)          # HalfResNet34 blocks per level (32, 64, 128, 256 channels)


def per_level(launches):
    """{level: [conv1 us list, plane_sum us list]}: a block starts at the first unfused conv after a fused conv2 or the stem."""
    bounds = [sum(LEVEL_BLOCKS[:i + 1]) for i in range(len(LEVEL_BLOCKS))]
    out = {l: ([], []) for l in range(len(LEVEL_BLOCKS))}
    block, in_block = -1, False
    for name, us in launches:
        if name.startswith("conv_umma_kernel"):
            fused = name.split(",")[3] == "true"
            if not fused and not in_block:
                block, in_block = block + 1, True
                level = next(l for l, b in enumerate(bounds) if block < b)
                out[level][0].append(us)
            elif fused:
                in_block = False
        elif name.startswith("plane_sum_kernel") and block >= 0:
            out[next(l for l, b in enumerate(bounds) if block < b)][1].append(us)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    import torch
    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    lines = ["device: %s | nvidia-smi: %s" % (props.name, smi)]
    res = {}
    child = os.path.join(ROOT, "tools", "residual_probe.py")
    for name, env in SETTINGS:
        r = subprocess.run([sys.executable, child, "--child", "--steps", str(args.steps)], cwd=ROOT,
                           env=dict(os.environ, **env), capture_output=True, text=True, timeout=900)
        row = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
        if r.returncode != 0 or not row:
            raise RuntimeError("%s failed:\n%s" % (name, r.stdout[-2000:] + r.stderr[-2000:]))
        res[name] = json.loads(row[0][len("RESULT "):])
    lines.append("")
    lines.append("per level (one profiled step): conv1 launches, total us, mean us | plane_sum launches, total us")
    lv = {name: per_level(res[name]["launches"]) for name, _ in SETTINGS}
    for l in range(len(LEVEL_BLOCKS)):
        for name, _ in SETTINGS:
            c, s = lv[name][l]
            lines.append("  level %d (%3d ch) %-9s conv1 %2d %8.1f %7.1f | plane_sum %2d %7.1f" % (
                l + 1, 32 << l, name, len(c), sum(c), sum(c) / max(len(c), 1), len(s), sum(s)))
        (cf, sf), (cs, ss) = lv["fused"][l], lv["separate"][l]
        lines.append("  level %d           conv1 + plane_sum: fused %.1f us, separate %.1f us (%+.1f us)" % (
            l + 1, sum(cf) + sum(sf), sum(cs) + sum(ss), sum(cf) + sum(sf) - sum(cs) - sum(ss)))
    for name, _ in SETTINGS:
        d = res[name]
        t = d["step_ms"]
        lines.append("")
        lines.append("== %s: %.1f audio-s per step, step %.3f ms mean (min %.3f, max %.3f) over %d steps, profiler off"
                     % (name, d["audio_s"], sum(t) / len(t), min(t), max(t), len(t)))
        lines.append("   one profiled step: %d launches, %.1f us of kernel time" % (len(d["launches"]), sum(x[1] for x in d["launches"])))
        tot = {}
        for n, us in d["launches"]:
            c, s = tot.get(n, (0, 0.0))
            tot[n] = (c + 1, s + us)
        lines.append("   per kernel: launches, total us")
        for n, (c, s) in sorted(tot.items(), key=lambda kv: -kv[1][1]):
            lines.append("     %-60s %4d %10.1f" % (n, c, s))
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
