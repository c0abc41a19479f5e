"""CPU suite: the throughput search kernel fits the occupancy it is compiled for.

search_tile_kernel<16, HS, SP, MINB> is launched with MINB one-warp CTAs per SM.  Its pop loop must fit the
register cap that __launch_bounds__ implies without spilling to local memory, and MINB warps must fit the
register file.  The shared-memory side of the same budget is a static_assert in pdmpc_capi.cu.
"""
import os
import re
import shutil
import subprocess


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "p-dmpc_b200", "csrc", "libpdmpc_b200.so")
REGS_PER_SM = 65536


def cuobjdump():
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    tool = os.path.join(os.path.dirname(nvcc), "cuobjdump")
    if os.path.exists(tool):
        return tool
    tool = shutil.which("cuobjdump")
    assert tool, "cuobjdump not found next to nvcc or on PATH"
    return tool


def resource_usage():
    out = subprocess.run([cuobjdump(), "--dump-resource-usage", LIB], check=True, capture_output=True,
                         text=True).stdout
    usage, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
            continue
        if name and "REG:" in line:
            usage[name] = {k: int(v) for k, v in re.findall(r"(\w+):(\d+)", line)}
            name = None
    return usage


def tile_instances(usage, tile):
    pat = re.compile(rf"_ZN5pdmpc18search_tile_kernelILi{tile}ELi(\d+)ELi(\d+)ELi(\d+)E")
    return [(int(m.group(3)), r) for n, r in usage.items() if (m := pat.match(n))]


def test_tile16_kernel_fits_its_occupancy_without_spills(built):
    inst = tile_instances(resource_usage(), 16)
    assert len(inst) == 1, inst
    ctas, r = inst[0]
    assert r["STACK"] == 0 and r["LOCAL"] == 0, r
    assert r["REG"] * 32 * ctas <= REGS_PER_SM, (r["REG"], ctas)


def test_tile8_kernel_does_not_spill(built):
    inst = tile_instances(resource_usage(), 8)
    assert len(inst) == 1, inst
    assert inst[0][1]["STACK"] == 0 and inst[0][1]["LOCAL"] == 0, inst[0][1]
