"""Where the time of one HalfResNet34 config-4 step goes, per switch setting of the residual path.

Each setting runs in its own process (the engine reads its switches once per process):
  default                  shortcut folded into conv2 on the 32- / 64-channel layers
  SKB_UNFUSED_SHORTCUT=1   every 1x1 shortcut as its own launch through a 16-bit buffer

Per setting: the step time from CUDA events (profiler off, mean / min / max over --steps steps after warm-up), then one
step under torch.profiler (CUDA activities, a separate pass): every kernel launch in order with its device time, and the
totals per kernel.  The step is bench.py's shape: 96 utterances of 2-20 s (~1050 audio-s), HalfResNet34, fp16.

    python tools/residual_probe.py [--steps 20] [--out FILE]
"""
import argparse
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SETTINGS = [("default", {}), ("unfused_shortcut", {"SKB_UNFUSED_SHORTCUT": "1"})]


def short_name(name):
    m = re.match(r"(?:void )?(?:skb::)?(\w+)(<[^(]*>)?", name)
    if not m:
        return name[:60]
    args = (m.group(2) or "").replace("(int)", "").replace("(bool)", "").replace(" ", "")
    return m.group(1) + args


def child(steps):
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from torch.profiler import ProfilerActivity, profile
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    with torch.no_grad():
        m = bench.build_model("halfresnet34", 256, dev)
        b = bench.make_batches(1, 96, 500, 2.0, 20.0, dev)[0]
        for _ in range(3):
            m.extract_packed(b[1], b[2])
        torch.cuda.synchronize()
        times = []
        for _ in range(steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            m.extract_packed(b[1], b[2])
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            m.extract_packed(b[1], b[2])
            torch.cuda.synchronize()
    kernels = [(e.time_range.start, short_name(e.name), e.device_time) for e in prof.events()
               if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith("Memcpy") and not e.name.startswith("Memset")]
    kernels.sort()
    audio_s = float(sum(b[2])) / 16000.0
    print("RESULT " + json.dumps({"audio_s": audio_s, "step_ms": times, "launches": [(n, t) for _, n, t in kernels]}))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.child:
        return child(args.steps)
    import torch
    lines = []
    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    lines.append("device: %s | nvidia-smi: %s" % (props.name, smi))
    res = {}
    for name, env in SETTINGS:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--steps", str(args.steps)], cwd=ROOT,
                           env=dict(os.environ, **env), capture_output=True, text=True, timeout=900)
        row = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
        if r.returncode != 0 or not row:
            raise RuntimeError("%s failed:\n%s" % (name, r.stdout[-2000:] + r.stderr[-2000:]))
        res[name] = json.loads(row[0][len("RESULT "):])
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
        lines.append("   launch list (in order): us, kernel")
        for i, (n, us) in enumerate(d["launches"]):
            lines.append("     %3d %9.1f  %s" % (i, us, n))
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
