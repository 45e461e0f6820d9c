"""The algebraic pressure multigrid with PressureBCs on several ranks: every rank gathers the Dirichlet flags of all
owned rows with the global Ap, builds the same mask and hierarchy, and keeps its owned rows of level 1.  Runs
tests/amg_pbc_mr_worker.py under torch.distributed.run (partition, slab-local provider and adapter routes; the outlet
lies in the last slab, so the other ranks hold no outlet dof) and is skipped on boxes with fewer GPUs."""
import os
import subprocess
import sys

import pytest

from oasisx_b200 import _lib as L

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.parametrize("nranks,peer", [(2, "1"), (2, "0"), (4, "1"), (4, "0")])
def test_amg_with_pressure_bcs_on_several_ranks(nranks, peer):
    if L.load_library().b2_device_count() < nranks:
        pytest.skip(f"needs {nranks} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nranks}", "--master-addr",
           "127.0.0.1", "--master-port", str(29900 + 10 * nranks + int(peer)), os.path.join(HERE, "amg_pbc_mr_worker.py"),
           "partition", "slab", "adapter"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, env=dict(os.environ, B200_PEER=peer))
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-4000:]
    assert res.stdout.count("MR_OK") == nranks
    print(res.stdout[-3000:])
