"""Restart files: a run saved after step k and resumed by a new solver continues bit for bit like the run that was never
interrupted (solution bytes, every StepInfo field but the two timings, forces.txt bytes), across the CN / BE first step
and the first-order u* of step 2, for Newton, for SUPG in 3-D and with a forcing source; the library's sticky cycle flag
crosses the file; forces.txt is cut back to the saved step after a crash; the driver's --restart-every / --resume; and
every mismatch or damaged file is refused before anything is changed.  The two-rank checks are tools/gpu_multi.py
--restart (skipped below two GPUs)."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from tests import restart_format as rf
from tests.conftest import PKG_DIR, ROOT
from tests.forcing_sources import SMOOTH

pytestmark = pytest.mark.gpu

TIMINGS = ("wall_seconds", "forcing_seconds")


def _out(path):
    os.makedirs(path, exist_ok=True)
    return str(path) + "/"


def _solver(nsb, case, mesh, out, **kw):
    return nsb.HostSolver(case, mesh, output_dir=out, **kw)


def _steps(s, n):
    return [{k: v for k, v in s.step().items() if k not in TIMINGS} for _ in range(n)]


def _mesh_path(request, msh_file, tmp_path, name):
    if name == "small-3D":
        from tools import msh
        p = str(tmp_path / "m3.bin")
        msh.write_bin(p, request.getfixturevalue("small_3d_mesh"))
        return p
    return msh_file(name)


def _straight_and_resumed(nsb, case, mesh, tmp_path, k, setup=lambda s: None, **kw):
    """Run A: 2k steps.  Run B: k steps, save_restart, a new solver resumes, k more.  Returns both."""
    a_dir, b_dir = _out(tmp_path / "a"), _out(tmp_path / "b")
    a = _solver(nsb, case, mesh, a_dir, **kw)
    setup(a)
    a.initialize()
    infos_a = _steps(a, 2 * k)
    xa = a.solution()
    a.close()
    b = _solver(nsb, case, mesh, b_dir, **kw)
    setup(b)
    b.initialize()
    infos_b = _steps(b, k)
    b.save_restart(b_dir + "restart.nsb")
    b.close()
    b = _solver(nsb, case, mesh, b_dir, **kw)
    setup(b)
    b.resume(b_dir + "restart.nsb")
    infos_b += _steps(b, k)
    xb = b.solution()
    b.close()
    return dict(infos_a=infos_a, infos_b=infos_b, xa=xa, xb=xb, forces_a=open(a_dir + "forces.txt", "rb").read(),
                forces_b=open(b_dir + "forces.txt", "rb").read(), file=open(b_dir + "restart.nsb", "rb").read())


def _assert_same(r):
    assert r["infos_a"] == r["infos_b"]
    assert r["xa"].tobytes() == r["xb"].tobytes()
    assert r["forces_a"] == r["forces_b"]


@pytest.mark.parametrize("case,mesh,k", [("2D-2", "mesh-2D", 1), ("2D-2", "mesh-2D", 2), ("2D-1", "mesh-2D", 2),
                                         ("3D-2Z", "small-3D", 2)])
def test_continuation_is_bit_identical(nsb, request, msh_file, tmp_path, case, mesh, k):
    r = _straight_and_resumed(nsb, case, _mesh_path(request, msh_file, tmp_path, mesh), tmp_path, k)
    _assert_same(r)
    f = rf.unpack(r["file"])                    # the file the C++ class wrote, read by the Python restatement
    assert (f["case"], f["step"], f["dim"]) == (case, k, 2 if case.startswith("2D") else 3)
    assert f["time"] == r["infos_a"][k - 1]["time"]
    assert (f["first_step"], f["second_step"]) == (0, int(k == 1))
    assert len(r["forces_a"].decode().strip().split("\n")) == 2 * k + 1


def test_continuation_with_forcing_source(nsb, msh_file, tmp_path):
    r = _straight_and_resumed(nsb, "2D-2", msh_file("mesh-2D"), tmp_path, 2, setup=lambda s: s.set_forcing_source(SMOOTH))
    _assert_same(r)


def test_cycle_flag_crosses_the_file(nsb, msh_file, tmp_path):
    k = 2
    mesh = msh_file("mesh-2D")
    a_dir, b_dir = _out(tmp_path / "a"), _out(tmp_path / "b")
    a = _solver(nsb, "2D-2", mesh, a_dir)
    a.initialize()
    _steps(a, k)
    assert a.device().velocity_pc_info()["two_level"]          # the flag decides something here
    a.device().set_run_state(True)
    a.save_restart(b_dir + "restart.nsb")
    infos_a = _steps(a, 2)
    pc_a = a.device().velocity_pc_info()["two_level"]
    xa = a.solution()
    a.close()
    assert rf.unpack(open(b_dir + "restart.nsb", "rb").read())["cycle_disabled"] == 1
    b = _solver(nsb, "2D-2", mesh, b_dir)
    b.resume(b_dir + "restart.nsb")
    assert b.device().run_state() == dict(cycle_disabled=True)
    infos_b = _steps(b, 2)
    pc_b = b.device().velocity_pc_info()["two_level"]
    xb = b.solution()
    b.close()
    assert pc_a is False and pc_b is False
    assert infos_a == infos_b and xa.tobytes() == xb.tobytes()


def test_device_run_state_round_trip(nsb, golden_mesh):
    from oracle import dofs as odofs
    m = golden_mesh("mesh-2D")
    dm = odofs.enumerate_dofs(m)
    d = nsb.Device(2, 0)
    with pytest.raises(nsb.NsbError, match="no mesh uploaded"):
        d.run_state()
    with pytest.raises(nsb.NsbError, match="no mesh uploaded"):
        d.set_run_state(True)
    d.upload_mesh(m.points, m.cells, dm.cell_dofs, dm.n_u, dm.n_p)
    assert d.run_state() == dict(cycle_disabled=False)
    d.set_run_state(True)
    assert d.run_state() == dict(cycle_disabled=True)
    d.set_run_state(**d.run_state())
    assert d.run_state() == dict(cycle_disabled=True)
    d.set_run_state(False)
    assert d.run_state() == dict(cycle_disabled=False)
    d.set_run_state(True)
    d.set_solver_opts()                                          # new options reset the flag
    assert d.run_state() == dict(cycle_disabled=False)
    d.set_run_state(True)
    d.upload_mesh(m.points, m.cells, dm.cell_dofs, dm.n_u, dm.n_p)   # so does a new mesh
    assert d.run_state() == dict(cycle_disabled=False)
    d.close()


def test_forces_after_a_crash(nsb, msh_file, tmp_path):
    """Saved at step 3, the run went on to step 5 and died; resuming from the step-3 file in the same directory and running
    3 steps gives the forces.txt of a 6-step run (rows 4 and 5 of the dead run are dropped, not duplicated)."""
    mesh = msh_file("mesh-2D")
    c_dir, d_dir = _out(tmp_path / "c"), _out(tmp_path / "d")
    s = _solver(nsb, "2D-2", mesh, c_dir)
    s.initialize()
    _steps(s, 3)
    s.save_restart(c_dir + "restart.nsb")
    _steps(s, 2)
    s.close()
    assert len(open(c_dir + "forces.txt").read().strip().split("\n")) == 6
    s = _solver(nsb, "2D-2", mesh, c_dir)
    s.resume(c_dir + "restart.nsb")
    _steps(s, 3)
    s.close()
    s = _solver(nsb, "2D-2", mesh, d_dir)
    s.initialize()
    _steps(s, 6)
    s.close()
    assert open(c_dir + "forces.txt", "rb").read() == open(d_dir + "forces.txt", "rb").read()


def test_driver_restart_every_and_resume(msh_file, tmp_path):
    exe = os.path.join(PKG_DIR, "navier_stokes")
    mesh = msh_file("mesh-2D")
    split, whole = tmp_path / "split", tmp_path / "whole"
    split.mkdir()
    whole.mkdir()

    def drive(cwd, *args):
        r = subprocess.run([exe, "2D-2", mesh, *args], cwd=str(cwd), capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        return r.stdout

    drive(split, "--steps", "3", "--restart-every", "3")
    assert (split / "restart.nsb").exists() and not (split / "restart.nsb.tmp").exists()
    assert rf.unpack((split / "restart.nsb").read_bytes())["step"] == 3
    for f in split.iterdir():
        if f.suffix in (".vtu", ".pvtu"):
            f.unlink()
    out = drive(split, "--resume", str(split / "restart.nsb"), "--steps", "3")
    assert "Resuming from %s: step 3, t=" % (split / "restart.nsb") in out
    drive(whole, "--steps", "6")
    assert (split / "forces.txt").read_bytes() == (whole / "forces.txt").read_bytes()
    pvtu = sorted(f.name for f in split.iterdir() if f.suffix == ".pvtu")
    assert pvtu == ["solution_%04d.pvtu" % k for k in (4, 5, 6)]


def test_mismatches_and_damaged_files_are_refused(nsb, msh_file, tmp_path):
    mesh = msh_file("mesh-2D")
    files = {}
    for name, case, m, kw in (("base", "2D-2", mesh, {}), ("newton", "2D-1", mesh, {}),
                              ("coarse", "2D-2", msh_file("mesh-2D-40"), {})):
        s = _solver(nsb, case, m, _out(tmp_path / name), **kw)
        s.initialize()
        _steps(s, 1)
        files[name] = str(tmp_path / name / "restart.nsb")
        s.save_restart(files[name])
        s.close()
    raw = open(files["base"], "rb").read()
    (tmp_path / "truncated.nsb").write_bytes(raw[:len(raw) // 2])
    flipped = bytearray(raw)
    flipped[rf.unpack(raw)["payload_offset"] + 8 * 100 + 3] ^= 0x10
    (tmp_path / "flipped.nsb").write_bytes(bytes(flipped))
    out = _out(tmp_path / "target")
    sentinel = b"Time\tCd\tCl\tDeltaP\nsentinel row\n"
    cases = [(files["coarse"], {}, "n_u"),
             (files["newton"], {}, "the test case is '2D-1' in the file but '2D-2'"),
             (files["base"], dict(deltat=0.01), "the time step dt is 0.02"),
             (str(tmp_path / "truncated.nsb"), {}, "truncated"),
             (str(tmp_path / "flipped.nsb"), {}, "checksum mismatch"),
             (str(tmp_path / "missing.nsb"), {}, "cannot open restart file")]
    for path, kw, expect in cases:
        open(out + "forces.txt", "wb").write(sentinel)
        s = _solver(nsb, "2D-2", mesh, out, **kw)
        with pytest.raises(nsb.NsbError) as e:
            s.resume(path)
        s.close()
        assert expect in str(e.value), (path, str(e.value))
        assert open(out + "forces.txt", "rb").read() == sentinel, path


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


def test_multi_gpu_restart(tmp_path):
    """Two ranks save at step 2 and go on; fresh two-rank solvers resume and match per rank, bit for bit; one GPU resuming
    the two-rank file follows the two-rank continuation within the tight-tolerance bars."""
    if _ngpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    out = str(tmp_path / "restart.json")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tools", "gpu_multi.py"), "--restart", "--json", out, "--lc", "0.05"]
    r = subprocess.run(cmd, env=dict(os.environ, OMP_NUM_THREADS="4"), capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    s = json.load(open(out))
    assert s["world"] == 2 and len(s["ranks"]) == 2
    for r_ in s["ranks"]:
        assert r_["solution_bitexact"] and r_["steps_equal"], r_
    assert s["forces_rows_equal"]
    assert s["one_gpu_field_relerr"] < 1e-8, s
    assert s["one_gpu_force_relerr"] < 1e-6, s
