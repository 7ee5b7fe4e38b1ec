"""Pins oracle/prog_oracle.cpp (the restatement of the reference's program-side functions) to the reference's OWN text of
src/prog/integrate.cpp (meshToFaceCloud, flattenVertices, cleanupMesh, reprojectPoint, lines 63-222; the per-cloud preparation
+ z-buffer re-organisation of main(), lines 559-635).

Each test compares what the restatement computes with what the same inputs gave through that text, compiled from the source
where it lies (oracle/Makefile `refprog`).  Those results (SHA-256 digests of every compared array, and the counts) are stored in
tests/golden/ref_pins.json; tools/make_ref_pins.py regenerates them where the reference sources are available."""
import numpy as np
import pytest

from oracle import oracle_py
from tests.common import sha
from tests.test_ref_pin import golden


def _cloud(rng, n, spread=1.0):
    z = rng.uniform(0.4, 3.0, n).astype(np.float32)
    x = (rng.uniform(-0.7, 0.7, n) * z * spread).astype(np.float32)
    y = (rng.uniform(-0.55, 0.55, n) * z * spread).astype(np.float32)
    pts = np.zeros((n, 8), np.float32)
    pts[:, 0], pts[:, 1], pts[:, 2], pts[:, 3] = x, y, z, 1.0
    pts.view(np.uint32)[:, 4] = rng.integers(0, 2**32, n, dtype=np.uint64).astype(np.uint32)
    return pts


ORGANISE_CASES = [(1, 1.0, False, False), (2, 0.001, True, False), (3, 1.0, True, True), (4, 2.5, False, True)]


def observe_organise(kind, seed, units, zero_nans, world):
    rng = np.random.default_rng(seed)
    W, H = 160, 120
    intr = (131.25, 131.25, 79.5, 59.5)
    pts = _cloud(rng, 60000, spread=1.2)
    pts[:, :3] /= units                                            # the program scales by cloud_units first (:559-568)
    pts[rng.random(len(pts)) < 0.03, :3] = 0.0                     # (0,0,0) = NaN under --zero-nans
    pts[rng.random(len(pts)) < 0.02, 2] = np.nan
    pts[rng.random(len(pts)) < 0.02, 2] *= -1                      # behind the camera
    dup = rng.integers(0, len(pts), 4000)                          # exact depth ties: the earlier point must win (:603-606)
    pts[dup[:2000]] = pts[dup[2000:]]
    tf = None
    if world:
        a = 0.3 * seed
        tf = np.array([[np.cos(a), 0, np.sin(a), 0.1], [0, 1, 0, -0.05], [-np.sin(a), 0, np.cos(a), 0.2], [0, 0, 0, 1]], np.float64)
    out, filled = oracle_py.organize(pts, intr, W, H, rgba_off=16, cloud_units=units, zero_nans=zero_nans, world_to_camera=tf, kind=kind)
    assert filled > 500
    # x, y, z and the colour word; the padding float and the bytes after the colour are whatever the default point holds
    return {"filled": filled, "xyz": sha(out.view(np.uint32)[..., :3]), "rgba": sha(out.view(np.uint32)[..., 4])}


@pytest.mark.parametrize("seed,units,zero_nans,world", ORGANISE_CASES)
def test_organise_block_matches_the_reference_text(seed, units, zero_nans, world):
    assert observe_organise("port", seed, units, zero_nans, world) == golden(f"organise[{seed}]")


def _mc_like_mesh(rng, n_quads, jitter):
    """A bumpy sheet of quads split into triangles, as a soup (every triangle has its own three vertices, like marching cubes
    output), plus a few small stray islands for cleanupMesh."""
    g = int(np.sqrt(n_quads))
    xs, ys = np.meshgrid(np.arange(g + 1), np.arange(g + 1), indexing="ij")
    P = np.stack([xs * 0.01, ys * 0.01, 0.02 * np.sin(xs * 0.3) * np.cos(ys * 0.2)], -1).astype(np.float32)
    tris = []
    for i in range(g):
        for j in range(g):
            a, b, c, d = P[i, j], P[i + 1, j], P[i + 1, j + 1], P[i, j + 1]
            tris += [(a, b, c), (a, c, d)]
    for k in range(12):                                            # islands of 1..6 triangles far from the sheet
        o = np.array([0.5 + 0.2 * k, 1.0, 0.3], np.float32)
        for t in range(1 + k % 6):
            tris.append((o + [0.004 * t, 0, 0], o + [0.004 * t + 0.003, 0, 0], o + [0.004 * t, 0.003, 0]))
    soup = np.asarray(tris, np.float32).reshape(-1, 3)
    soup = soup + (rng.normal(scale=jitter, size=soup.shape)).astype(np.float32)
    return soup, np.arange(len(soup), dtype=np.int32).reshape(-1, 3)


def mesh_digests(v, t):
    return {"n_verts": len(v), "n_tris": len(t), "verts": sha(v.view(np.uint32)), "tris": sha(t)}


FLATTEN_CASES = [(1, 0.0, 1e-4), (2, 3e-5, 1e-4), (3, 2e-4, 2e-3), (4, 0.0, 0.0)]


def observe_flatten(kind, seed, jitter, min_dist):
    rng = np.random.default_rng(seed)
    v, t = _mc_like_mesh(rng, 900, jitter)
    fv, ft = oracle_py.flatten_vertices(v, t, min_dist, kind=kind)
    assert min_dist == 0.0 or len(fv) < len(v)
    return mesh_digests(fv, ft)


@pytest.mark.parametrize("seed,jitter,min_dist", FLATTEN_CASES)
def test_flatten_vertices_matches_the_reference_text(seed, jitter, min_dist):
    assert observe_flatten("port", seed, jitter, min_dist) == golden(f"flatten[{seed}]")


CLEANUP_CASES = [(1, 0.02, 5), (2, 0.008, 3), (3, 0.05, 40)]


def observe_cleanup(kind, seed, face_dist, min_neighbors):
    rng = np.random.default_rng(seed)
    v, t = _mc_like_mesh(rng, 400, 0.0)
    v, t = oracle_py.flatten_vertices(v, t, 1e-4, kind="port")       # cleanupMesh runs on the welded mesh in the program (:707-712)
    cv, ct = oracle_py.cleanup_mesh(v, t, face_dist, min_neighbors, kind=kind)
    assert len(ct) < len(t)
    return mesh_digests(cv, ct)


@pytest.mark.parametrize("seed,face_dist,min_neighbors", CLEANUP_CASES)
def test_cleanup_mesh_matches_the_reference_text(seed, face_dist, min_neighbors):
    assert observe_cleanup("port", seed, face_dist, min_neighbors) == golden(f"cleanup[{seed}]")


def observe_all(kind):
    """Every observation above, keyed as in tests/golden/ref_pins.json."""
    out = {}
    for c in ORGANISE_CASES:
        out[f"organise[{c[0]}]"] = observe_organise(kind, *c)
    for c in FLATTEN_CASES:
        out[f"flatten[{c[0]}]"] = observe_flatten(kind, *c)
    for c in CLEANUP_CASES:
        out[f"cleanup[{c[0]}]"] = observe_cleanup(kind, *c)
    return out
