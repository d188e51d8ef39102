"""Reader and writer of the restart file format of NavierStokes::save_restart (DESIGN.md section 12), restated in Python
so that the tests can check the files the C++ class writes and build files the C++ class must reject."""
import struct

import numpy as np

MAGIC = b"NSBRST01"
FNV_OFFSET, FNV_PRIME = 14695981039346656037, 1099511628211


def fnv1a(data):
    h = FNV_OFFSET
    for b in data:
        h = ((h ^ b) * FNV_PRIME) & 0xFFFFFFFFFFFFFFFF
    return h


def pack(dim, n_u, n_p, n_cells, n_vertices, mesh_hash, case, Re, U_m, dt, scheme, method, use_supg, T, time, step,
         first_step, second_step, cycle_disabled, vectors):
    body = struct.pack("<iqqqqQ", dim, n_u, n_p, n_cells, n_vertices, mesh_hash)
    body += struct.pack("<I", len(case)) + case.encode()
    body += struct.pack("<dddiiid", Re, U_m, dt, scheme, method, use_supg, T)
    body += struct.pack("<dqiii", time, step, first_step, second_step, cycle_disabled)
    for v in vectors:
        body += np.ascontiguousarray(v, "<f8").tobytes()
    return MAGIC + body + struct.pack("<Q", fnv1a(body))


def unpack(raw, check_sum=True):
    """The fields of a restart file as a dict; asserts the magic, the size and (check_sum) the checksum."""
    assert raw[:8] == MAGIC
    o = 8
    dim, n_u, n_p, n_cells, n_vertices, mesh_hash = struct.unpack_from("<iqqqqQ", raw, o)
    o += struct.calcsize("<iqqqqQ")
    (ln,) = struct.unpack_from("<I", raw, o)
    o += 4
    case = raw[o:o + ln].decode()
    o += ln
    Re, U_m, dt, scheme, method, use_supg, T = struct.unpack_from("<dddiiid", raw, o)
    o += struct.calcsize("<dddiiid")
    time, step, first_step, second_step, cycle_disabled = struct.unpack_from("<dqiii", raw, o)
    o += struct.calcsize("<dqiii")
    n = n_u + n_p
    assert len(raw) == o + 3 * 8 * n + 8, (len(raw), o + 3 * 8 * n + 8)
    vecs = [np.frombuffer(raw, "<f8", n, o + 8 * n * k) for k in range(3)]
    (stored,) = struct.unpack_from("<Q", raw, len(raw) - 8)
    if check_sum:
        assert fnv1a(raw[8:-8]) == stored
    return dict(dim=dim, n_u=n_u, n_p=n_p, n_cells=n_cells, n_vertices=n_vertices, mesh_hash=mesh_hash, case=case, Re=Re,
                U_m=U_m, dt=dt, scheme=scheme, method=method, use_supg=use_supg, T=T, time=time, step=step,
                first_step=first_step, second_step=second_step, cycle_disabled=cycle_disabled, vectors=vecs,
                payload_offset=o)
