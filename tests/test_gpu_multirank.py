"""BASELINE config 3 ("mesh-3D-5 ... 1 vs 2 GPUs") as a -m gpu test: tools/gpu_multi.py under torchrun with one
process per visible GPU (2, 4 or 8): peer-store halo (CUDA IPC over NVLink, separate push / wait kernels) and the NCCL
send/recv halo.  Skipped on a single-GPU box.

Asserted per rank: pattern of the owned rows bit-exact against the oracle (reference cpp:256-273), A and b
relative 1e-12 against the oracle AND bit-exact against a single-GPU assembly (SURVEY 8c pin 6), the
tight-tolerance field within 1e-8 of a sparse direct solve, the same GMRES count at the reference tolerance as on
one GPU; then three steps of NavierStokes<3>(make_3D_2Z): C_D, C_L, dP within 1e-6 of the oracle's trajectory
(which the 1-GPU run matches to the same bar in test_gpu_parity.py), and one VTU piece per rank."""
import json
import os
import socket
import subprocess
import sys

import pytest

from tests.conftest import ROOT

pytestmark = pytest.mark.gpu


def _ngpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("halo", ["p2p", "nccl"])
def test_multi_gpu_matches_oracle_and_single_gpu(tmp_path, halo):
    n = _ngpus()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (run with gpurun --gpus 2)")
    world = 8 if n >= 8 else 4 if n >= 4 else 2
    out = str(tmp_path / "multi.json")
    env = dict(os.environ, NSB200_HALO=halo, OMP_NUM_THREADS="4")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tools", "gpu_multi.py"), "--json", out, "--lc", "0.05"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    s = json.load(open(out))
    keep = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(keep):
        json.dump(s, open(os.path.join(keep, "multirank_n%d_%s.json" % (world, halo)), "w"), indent=1)
    assert s["world"] == world and len(s["ranks"]) == world
    assert sum(r_["rows"] for r_ in s["ranks"]) == s["n_dofs"]
    for r_ in s["ranks"]:
        assert r_["pattern_ok"] and r_["A_relerr"] < 1e-12 and r_["b_relerr"] < 1e-12, r_
        assert r_["A_bitexact_vs_1gpu"] and r_["b_bitexact_vs_1gpu"], r_
        assert r_["gmres_ok"] and r_["tight_ok"] and r_["field_relerr_vs_direct"] < 1e-8, r_
        assert abs(r_["gmres_its"] - r_["gmres_its_1gpu"]) <= 1, r_      # partition-independent preconditioner (up to rounding)
    for st in s["host_class_steps"]:
        assert st["err_cd"] < 1e-6 and st["err_dp"] < 1e-6, st
        assert st["err_cl"] < 1e-6 or st["err_cl"] * st["cl_abs"] < 1e-10, st       # C_L ~ 0 in 3D-2Z
    assert s["host_class_field_relerr"] < 1e-8
    assert s["vtu_pieces"] == ["solution_0003.%d.vtu" % k for k in range(world)]
    assert s["vtu_cells_total"] == s["mesh_cells"]
