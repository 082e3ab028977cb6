"""The two-network entry points are exported, and their kernels (the CTA-pair-split input convolution and tower, the CTA-split
heads) run on tcgen05 with TMA like the single-network kernels.  Runs on the CPU box (cuobjdump reads the sm_100a code)."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

import alphazero_chess_b200 as az

LIB = os.path.join(os.path.dirname(az.__file__), "libaz_b200.so")


def test_network_entry_points_are_exported():
    L = az.lib()
    for name in ("az_load_network", "az_forward_networks", "az_search_networks"):
        assert isinstance(getattr(L, name), ctypes._CFuncPtr), name


@pytest.mark.parametrize("needle", ["conv_tower_nets_kernelILi2E", "conv3x3_tc2_nets_kernelILi1ELi64E", "k_heads_tc_nets"])
def test_network_kernels_are_tcgen05(needle):
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    az.lib()
    out = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    kernels, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            kernels[cur] = []
        elif cur is not None:
            kernels[cur].append(line)
    hits = [k for k in kernels if needle in k]
    assert hits, needle
    for k in hits:
        s = "\n".join(kernels[k])
        assert re.search(r"\bUTC[A-Z]*MMA", s) and "UTMALDG" in s and "LDTM" in s, k
