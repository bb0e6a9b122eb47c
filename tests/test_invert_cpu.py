"""CPU suite: the parts of the device inversion that need no device (tool usage, argument checks of invert_rl_bwt)."""
import os
import subprocess

import numpy as np
import pytest

import grlbwt_b200 as G

IMAGE = (1).to_bytes(8, "little") + (1).to_bytes(8, "little") + bytes([10, 1, 65, 1])   # "A\n" as a BWT: runs (\n,1) (A,1)


def test_reverse_bwt_gpu_usage():
    r = subprocess.run([os.path.join(G.LIB_DIR, "reverse_bwt_gpu")], capture_output=True, text=True)
    assert r.returncode == 0 and "usage:" in r.stdout


@pytest.mark.parametrize("kw", [dict(cell_bytes=3), dict(cell_bytes=0), dict(n_seqs=-1), dict(out=np.zeros(8, np.uint16)),
                                dict(out=np.zeros((2, 8), np.uint8)), dict(out=np.zeros(16, np.uint8)[::2]), dict(out=b"\0" * 8)])
def test_invert_rl_bwt_argument_checks(kw):
    """rejected before the library is asked for a device (which this machine may not have)"""
    with pytest.raises(G.GrlGpuError) as e:
        G.invert_rl_bwt(IMAGE, **kw)
    assert e.value.status == -1


def test_invert_rl_bwt_reads_a_path(tmp_path):
    """a path is read like parse_rl_bwt reads it: the argument checks see the file's bytes"""
    p = tmp_path / "x.rl_bwt"
    p.write_bytes(IMAGE)
    with pytest.raises(G.GrlGpuError) as e:
        G.invert_rl_bwt(str(p), cell_bytes=5)
    assert e.value.status == -1
