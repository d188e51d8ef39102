"""The producer of the streamed velocity operator (k_vel_stream) loads tile headers a batch ahead and neighbour offsets one
tile ahead, so its edge cases are the first and last tiles of a CTA and the wrap of its ring of stages.  NSB200_VS_CTAS caps
the grid: with one CTA the ring wraps hundreds of times, with a cap above the tile count of a level some CTAs own a single
tile.  A tile is always reduced by one consumer group in a fixed order, whichever CTA takes it, so y and poly must be
bit-identical for every cap.

The GPU tests run on the mesh-2D-100 and mesh-3D-5 systems of test_gpu_preconditioner.py, both levels, fp16 and fp32,
MODE 2 / 3 / 4; the CPU tests check that the variable is parsed when a handle is created."""
import contextlib
import os

import numpy as np
import pytest

CAPS = (1, 2, 3, 7)
KEYS = ("2d100", "3d5")


@contextlib.contextmanager
def vs_ctas(cap):
    """NSB200_VS_CTAS = cap (None: unset) while handles are created"""
    old = os.environ.get("NSB200_VS_CTAS")
    if cap is None:
        os.environ.pop("NSB200_VS_CTAS", None)
    else:
        os.environ["NSB200_VS_CTAS"] = str(cap)
    try:
        yield
    finally:
        if old is None:
            os.environ.pop("NSB200_VS_CTAS", None)
        else:
            os.environ["NSB200_VS_CTAS"] = old


@pytest.mark.parametrize("bad", ["0", "-3", "abc", "4x", "", " ", "1.5", "99999999999999999999"])
def test_cap_rejects_non_positive_integers(nsb, bad):
    with vs_ctas(bad), pytest.raises(nsb.NsbError, match="NSB200_VS_CTAS must be a positive integer"):
        nsb.Device(3)


@pytest.mark.parametrize("good", ["1", "7", "148"])
def test_cap_accepts_positive_integers(nsb, good):
    # without a GPU creation fails later, on the device; with one it succeeds
    try:
        with vs_ctas(good):
            dev = nsb.Device(3)
        dev.close()
    except nsb.NsbError as e:
        assert "NSB200_VS_CTAS" not in str(e), e


def _apply_all(dev, n_fine, n_coarse):
    """MODE 2 / 3 / 4 on both levels, fixed random vectors: {(level, mode): arrays}"""
    out = {}
    for level, n in ((0, n_fine), (1, n_coarse)):
        rng = np.random.default_rng(23 + level)
        x, u, p = rng.standard_normal((3, n))
        for mode in (2, 3, 4):
            r = dev.apply_velocity_operator(level, mode, x, u, p, (0.7, -1.3, 0.4, 0.9))
            out[(level, mode)] = r if mode == 3 else (r,)
    return out


@pytest.fixture(scope="module")
def stream_outputs(nsb, golden_mesh):
    """Outputs of every (mesh, precision, cap) on a device of its own, created with that cap."""
    from tests.test_gpu_preconditioner import MESHES, System
    from tools import meshgen
    meshes = {}
    made = {}

    def get(key, prec, cap):
        if (key, prec, cap) not in made:
            name, case = MESHES[key]
            if key not in meshes:
                meshes[key] = meshgen.mesh_3d(5) if key == "3d5" else golden_mesh(name)
            with vs_ctas(cap):
                s = System(nsb, meshes[key], case)
            try:
                s.assemble("lin", pressure=False, precond_precision=prec)
                tiles = (s.dev.velocity_operator_info()["tiles"], s.dev.velocity_operator(1)["tiles"])
                made[(key, prec, cap)] = (tiles, _apply_all(s.dev, s.n_u, s.dim * s.n_p))
            finally:
                s.dev.close()
        return made[(key, prec, cap)]

    return get


@pytest.mark.gpu
@pytest.mark.parametrize("cap", CAPS)
@pytest.mark.parametrize("prec", [16, 32])
@pytest.mark.parametrize("key", KEYS)
def test_stream_bit_identical_for_every_grid_cap(stream_outputs, key, prec, cap):
    tiles, ref = stream_outputs(key, prec, None)
    tiles_c, got = stream_outputs(key, prec, cap)
    assert tiles_c == tiles
    print(f"[{key} fp{prec} cap {cap}] fine {tiles[0]} tiles, coarse {tiles[1]} tiles: up to "
          f"{-(-tiles[0] // min(cap, tiles[0]))} / {-(-tiles[1] // min(cap, tiles[1]))} tiles per CTA")
    for k, want in ref.items():
        for a, b in zip(got[k], want):
            assert np.all(np.isfinite(b)), (key, prec, cap, k)
            assert np.array_equal(a, b), (key, prec, cap, k, float(np.max(np.abs(a - b))))
