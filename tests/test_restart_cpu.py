"""CPU: HostSolver.resume checks a restart file's magic, size and checksum before it sets anything up, so a missing,
foreign, truncated or corrupted file is rejected with a message that says which, without a GPU.  The files are built
with the Python restatement of the format (tests/restart_format.py); a well-formed one passes these checks and only then
fails (no device here, or it does not describe the solver's mesh)."""
import numpy as np
import pytest

from tests import restart_format as rf


def _file(tmp_path, name="r.nsb"):
    n_u, n_p = 10, 3
    rng = np.random.default_rng(7)
    raw = rf.pack(2, n_u, n_p, 4, 5, 0x1234, "2D-2", 100.0, 1.5, 0.02, 1, 1, 0, 8.0, 0.04, 2, 0, 0, 0,
                  [rng.standard_normal(n_u + n_p) for _ in range(3)])
    p = tmp_path / name
    p.write_bytes(raw)
    return p, raw


def _resume_error(nsb, msh_file, path):
    s = nsb.HostSolver("2D-2", msh_file("mesh-2D"))
    try:
        with pytest.raises(nsb.NsbError) as e:
            s.resume(str(path))
    finally:
        s.close()
    return str(e.value)


def test_format_round_trip(tmp_path):
    p, raw = _file(tmp_path)
    f = rf.unpack(raw)
    assert (f["case"], f["step"], f["time"], f["n_u"], f["n_p"]) == ("2D-2", 2, 0.04, 10, 3)
    assert len(raw) == f["payload_offset"] + 3 * 8 * 13 + 8


def test_missing_file(nsb, msh_file, tmp_path):
    assert "cannot open restart file" in _resume_error(nsb, msh_file, tmp_path / "none.nsb")


def test_not_a_restart_file(nsb, msh_file, tmp_path):
    p = tmp_path / "x.nsb"
    p.write_bytes(b"Time\tCd\tCl\tDeltaP\n")
    assert "not a restart file" in _resume_error(nsb, msh_file, p)


def test_truncated_file(nsb, msh_file, tmp_path):
    p, raw = _file(tmp_path)
    p.write_bytes(raw[:-20])
    assert "truncated" in _resume_error(nsb, msh_file, p)
    p.write_bytes(raw[:30])
    assert "truncated" in _resume_error(nsb, msh_file, p)


def test_flipped_payload_byte(nsb, msh_file, tmp_path):
    p, raw = _file(tmp_path)
    b = bytearray(raw)
    b[rf.unpack(raw)["payload_offset"] + 17] ^= 0x01
    p.write_bytes(bytes(b))
    assert "checksum mismatch" in _resume_error(nsb, msh_file, p)


def test_well_formed_file_passes_the_integrity_checks(nsb, msh_file, tmp_path):
    p, _ = _file(tmp_path)
    msg = _resume_error(nsb, msh_file, p)
    assert "checksum" not in msg and "truncated" not in msg and "not a restart file" not in msg, msg
