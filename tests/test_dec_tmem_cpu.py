"""The persistent decoder's default instantiation keeps P in tensor memory when the window is the whole utterance
(no GPU needed: cuobjdump on the in-tree .so).  tcgen05.st / tcgen05.ld read STTM / LDTM in SASS."""
import os
import re
import shutil
import subprocess

import pytest

from helpers import package

CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


@pytest.fixture(scope="module")
def dec_scan_sass():
    lib = package()._lib.LIB_PATH
    if not os.path.exists(lib) or not os.path.exists(CUOBJDUMP):
        pytest.skip("library or cuobjdump missing")
    out = subprocess.run([CUOBJDUMP, "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name and "/*" in line:
            funcs[name].append(line)
    # dec_scan_kernel<false>: the default (non-compact) instantiation, the only one that stages P in TMEM
    hits = {k: v for k, v in funcs.items() if "dec_scan_kernel" in k and "ILb0E" in k}
    assert hits, "no dec_scan_kernel<false> in the library"
    return hits


def test_p_is_staged_and_read_through_tensor_memory(dec_scan_sass):
    for name, lines in dec_scan_sass.items():
        body = "\n".join(lines)
        assert "STTM" in body, name                            # one-time staging of P
        assert "LDTM" in body, name                            # energy loop reads P back
        assert "HMMA" in body, name                            # handler product still on mma.sync


def test_tensor_memory_energy_loop_does_not_touch_local_memory(dec_scan_sass):
    """One energy tile -- from each LDTM.xN (N = 4 * NTW P values per thread) through its 3 * NTW MMAs, the tanh
    chain and the four shuffles that reduce the two row sums -- holds no local-memory access.  The kernel as a whole
    does have local-memory traffic elsewhere (the dense-tile descriptors of the non-inlined dense_tile calls live on
    the stack); the energy loop is the part that runs per position."""
    for name, lines in dec_scan_sass.items():
        ld = [i for i, l in enumerate(lines) if "LDTM" in l]
        assert ld, name
        for i in ld:
            ntw = int(re.search(r"LDTM\.x(\d+)", lines[i]).group(1)) // 4
            mma = [j for j in range(i, len(lines)) if "HMMA" in lines[j]][:3 * ntw]
            assert len(mma) == 3 * ntw, (name, lines[i])
            shfl = [j for j in range(mma[-1], len(lines)) if "SHFL.BFLY" in lines[j]][:4]
            assert len(shfl) == 4, (name, lines[i])
            window = lines[i:shfl[-1] + 1]
            assert not any(re.search(r"\bLDL\b|\bSTL\b", l) for l in window), (name, lines[i])
