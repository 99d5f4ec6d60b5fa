"""Every kernel of the library is launched through ``launch_kernel`` (csrc/common.cuh), the one place that counts launches
for ``skb_kernel_launches`` and synchronises after each one under SKB_SYNC_CHECK=1.  A source scan keeps it that way."""
import os
import re

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "sidekit_b200", "csrc")


def _sources():
    """{file name: code with comments and string literals removed}"""
    out = {}
    for name in sorted(os.listdir(CSRC)):
        if name.endswith((".cu", ".cuh")):
            with open(os.path.join(CSRC, name)) as f:
                text = f.read()
            text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
            text = re.sub(r"//[^\n]*", "", text)
            out[name] = re.sub(r'"(\\.|[^"\\\n])*"', '""', text)
    return out


def _lines(pattern):
    return [(name, line.strip()) for name, text in _sources().items() for line in text.splitlines() if re.search(pattern, line)]


def test_sources_are_found():
    assert {"common.cuh", "engine.cu", "scoring.cu", "layers.cu"} <= set(_sources())


def test_no_triple_chevron_launch():
    assert _lines(r"<<<") == []


def test_cuda_launch_kernel_ex_only_in_the_helper():
    assert [name for name, _ in _lines(r"\bcudaLaunchKernelEx\b")] == ["common.cuh"]


def test_launch_counter_only_in_the_helper_its_definition_and_the_abi_getter():
    hits = _lines(r"\bg_launches\b")
    assert sorted(name for name, _ in hits) == ["common.cuh", "common.cuh", "engine.cu", "engine.cu"], hits
    engine = [line for name, line in hits if name == "engine.cu"]
    assert any(line.startswith("std::atomic<long long> g_launches") for line in engine), engine
    assert any(line.startswith("int64_t skb_kernel_launches(") for line in engine), engine
