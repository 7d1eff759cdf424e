"""Deterministic synthetic scenes for the BASELINE.json configs (SURVEY.md section 8d).

Each generator returns (verts float32[v,3], corners int32[3t,4], norms
float32[k,3] or None): the three lists the reference's OBJ glue hands to
build_kd (src/model.c:109-133).  Geometry is single-sided -- the kernel culls
back faces (src/kernel.cl:239) -- so triangles wind toward where the camera is.

Coordinates are passed through a 6-decimal text round trip ("%.6f" then parse),
so an OBJ written from these arrays loads back to the same floats.
"""
from __future__ import annotations

import numpy as np

from . import corners_from_faces

# The canonical camera of SURVEY.md section 8d / BASELINE.md section 4.
CANONICAL_CAMERA = dict(near=0.1, far=1.0, fov=np.pi / 3, position=(0.0, 0.9, -1.7),
                        forward=(0.0, -0.42, 0.9075))
# Default camera of the reference application (src/game.c:275-277).
REFERENCE_CAMERA = dict(near=0.1, far=1.0, fov=np.pi / 3, position=(0.0, 0.1, -0.2),
                        forward=(0.0, 0.0, 1.0))
# Slightly off-axis on purpose: a centred camera sends pixel rays exactly through
# the mesh edges of the axis-aligned walls (exact u/v ties between neighbours).
CORNELL_CAMERA = dict(near=0.1, far=1.0, fov=np.pi / 3, position=(0.031, 0.047, -2.6),
                      forward=(-0.012, -0.018, 0.99976599))


def _six_decimals(a: np.ndarray) -> np.ndarray:
    """float64 -> '%.6f' text -> float32, exactly what an OBJ round trip does."""
    flat = np.asarray(a, dtype=np.float64).reshape(-1)
    # Fast path: rint(x * 1e6) / 1e6 is the same double the text round trip gives
    # unless x * 1e6 sits within rounding error of a .5 tie; those few values (and
    # anything large) take the literal text path.
    scaled = flat * 1e6
    out = np.rint(scaled) / 1e6
    frac = scaled - np.floor(scaled)
    slow = (np.abs(frac - 0.5) < 1e-4) | (np.abs(flat) > 1e6) | ~np.isfinite(flat)
    if slow.any():
        out[slow] = np.char.mod("%.6f", flat[slow]).astype(np.float64)
    return out.astype(np.float32).reshape(np.shape(a))


def heightfield(n: int, with_normals: bool = False, seed: int = 0):
    """(n+1)^2 vertices over x,z in [-1,1], y = 0.15 sin(3x) cos(2z) + 0.02 N(0,1);
    2 n^2 upward-facing triangles.  n = 22 / 224 / 707 / 2236 gives
    968 / 100,352 / 999,698 / 9,999,392 triangles."""
    g = np.linspace(-1.0, 1.0, n + 1)
    x, z = np.meshgrid(g, g, indexing="ij")  # vertex (i, j) -> index i*(n+1)+j
    rng = np.random.default_rng(seed)
    y = 0.15 * np.sin(3 * x) * np.cos(2 * z) + 0.02 * rng.standard_normal(x.shape)
    verts = _six_decimals(np.stack([x, y, z], axis=-1).reshape(-1, 3))
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    a = (i * (n + 1) + j).reshape(-1)
    b = ((i + 1) * (n + 1) + j).reshape(-1)
    c = ((i + 1) * (n + 1) + j + 1).reshape(-1)
    d = (i * (n + 1) + j + 1).reshape(-1)
    faces = np.empty((2 * n * n, 3), dtype=np.int64)
    faces[0::2] = np.stack([a, c, b], axis=1)
    faces[1::2] = np.stack([a, d, c], axis=1)
    norms = None
    if with_normals:
        norms = np.zeros((len(verts), 3), dtype=np.float32)
        norms[:, 1] = 1.0
    return verts, corners_from_faces(faces, with_normals), norms


def _grid_quad(origin, du, dv, n):
    """n x n quads spanning origin + s*du + t*dv; triangles wind so that the
    geometric normal is du x dv."""
    s = np.linspace(0.0, 1.0, n + 1)
    S, T = np.meshgrid(s, s, indexing="ij")
    P = origin[None, None, :] + S[..., None] * du[None, None, :] + T[..., None] * dv[None, None, :]
    verts = P.reshape(-1, 3)
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    a = (i * (n + 1) + j).reshape(-1)
    b = ((i + 1) * (n + 1) + j).reshape(-1)
    c = ((i + 1) * (n + 1) + j + 1).reshape(-1)
    d = (i * (n + 1) + j + 1).reshape(-1)
    faces = np.empty((2 * n * n, 3), dtype=np.int64)
    faces[0::2] = np.stack([a, b, c], axis=1)
    faces[1::2] = np.stack([a, c, d], axis=1)
    nrm = np.cross(du, dv)
    nrm = nrm / np.linalg.norm(nrm)
    return verts, faces, np.tile(nrm, (len(verts), 1))


def _box(lo, hi):
    """Axis-aligned box, outward faces, 12 triangles, per-face normals."""
    lo, hi = np.asarray(lo, float), np.asarray(hi, float)
    e = hi - lo
    ex, ey, ez = np.array([e[0], 0, 0]), np.array([0, e[1], 0]), np.array([0, 0, e[2]])
    quads = [
        (lo, ez, ey),                 # -x face: normal ez x ey = -x
        (lo + ex, ey, ez),            # +x
        (lo, ex, ez),                 # -y
        (lo + ey, ez, ex),            # +y
        (lo, ey, ex),                 # -z
        (lo + ez, ex, ey),            # +z
    ]
    return [_grid_quad(o, du, dv, 1) for (o, du, dv) in quads]


def cornell(n: int = 10):
    """Cornell-style box: 5 inward-facing walls of n x n quads and two boxes,
    with vertex normals; 10 n^2 + 24 triangles (1024 at n = 10).  The open face
    is z = -1; use CORNELL_CAMERA.  Returns also a per-triangle material id
    (0 white, 1 red, 2 green, 3 light) for the stochastic mode."""
    X, Y, Z = np.eye(3)
    parts, mats = [], []
    walls = [
        (np.array([-1.0, -1.0, -1.0]), 2 * Z, 2 * X, 0),  # floor, normal +y
        (np.array([-1.0, 1.0, -1.0]), 2 * X, 2 * Z, 3),   # ceiling, normal -y (the light)
        (np.array([-1.0, -1.0, 1.0]), 2 * Y, 2 * X, 0),   # back wall, normal -z
        (np.array([-1.0, -1.0, -1.0]), 2 * Y, 2 * Z, 1),  # left wall, normal +x
        (np.array([1.0, -1.0, -1.0]), 2 * Z, 2 * Y, 2),   # right wall, normal -x
    ]
    for (o, du, dv, m) in walls:
        parts.append(_grid_quad(o, du, dv, n))
        mats.append(m)
    for q in _box([-0.65, -1.0, -0.1], [-0.05, 0.2, 0.5]) + _box([0.15, -1.0, -0.6], [0.7, -0.4, -0.05]):
        parts.append(q)
        mats.append(0)
    verts, faces, norms, tri_mat, base = [], [], [], [], 0
    for (v, f, nn), m in zip(parts, mats):
        verts.append(v)
        norms.append(nn)
        faces.append(f + base)
        tri_mat.append(np.full(len(f), m, dtype=np.int32))
        base += len(v)
    verts = _six_decimals(np.concatenate(verts))
    norms = _six_decimals(np.concatenate(norms))
    faces = np.concatenate(faces)
    return verts, corners_from_faces(faces, True), norms, np.concatenate(tri_mat)


CORNELL_MATERIALS = np.array([
    # albedo r g b, kind, emission r g b, pad
    [0.73, 0.73, 0.73, 0, 0, 0, 0, 0],
    [0.65, 0.05, 0.05, 0, 0, 0, 0, 0],
    [0.12, 0.45, 0.15, 0, 0, 0, 0, 0],
    [0.78, 0.78, 0.78, 0, 4.0, 4.0, 4.0, 0],
], dtype=np.float32)
CORNELL_MATERIALS.view(np.int32)[:, 3] = 0


def cornell_small_light(n: int = 10, side: float = 0.4, drop: float = 0.005):
    """cornell(n) with the ceiling's emission moved to a small square lamp: the ceiling takes the
    white material, and a side x side quad facing -y hangs `drop` below its centre with material 3
    (emitter).  10 n^2 + 26 triangles; use CORNELL_SMALL_LIGHT_MATERIALS, whose lamp emits as much
    power as the ceiling of CORNELL_MATERIALS does at side 0.4."""
    verts, corners, norms, tri_mat = cornell(n)
    tri_mat = np.where(tri_mat == 3, 0, tri_mat).astype(np.int32)
    X, Z = np.eye(3)[0], np.eye(3)[2]
    h = side / 2
    v, f, nn = _grid_quad(np.array([-h, 1.0 - drop, -h]), side * X, side * Z, 1)
    base = len(verts)
    verts = np.concatenate([verts, _six_decimals(v)])
    norms = np.concatenate([norms, _six_decimals(nn)])
    corners = np.concatenate([corners, corners_from_faces(f + base, True)])
    return verts, corners, norms, np.concatenate([tri_mat, np.full(len(f), 3, dtype=np.int32)])


CORNELL_SMALL_LIGHT_MATERIALS = CORNELL_MATERIALS.copy()
CORNELL_SMALL_LIGHT_MATERIALS[3, 4:7] = 100.0  # 4 * (2 x 2 ceiling) / (0.4 x 0.4 lamp)


def soup(n_tris: int, size: float = 0.02, seed: int = 1):
    """Incoherent stress scene: n_tris small random triangles in the unit cube
    (centred on the origin), no normals."""
    rng = np.random.default_rng(seed)
    centre = rng.uniform(-0.5, 0.5, size=(n_tris, 1, 3))
    offs = rng.uniform(-size, size, size=(n_tris, 3, 3))
    verts = _six_decimals((centre + offs).reshape(-1, 3))
    faces = np.arange(3 * n_tris, dtype=np.int64).reshape(-1, 3)
    return verts, corners_from_faces(faces, False), None


def write_obj_text(path: str, verts, corners, norms=None) -> None:
    """Minimal OBJ writer ('v', 'vn', 'f a//a' or 'f a')."""
    with open(path, "w") as f:
        for v in np.asarray(verts)[:, :3]:
            f.write("v %.6f %.6f %.6f\n" % tuple(v))
        if norms is not None:
            for v in np.asarray(norms)[:, :3]:
                f.write("vn %.6f %.6f %.6f\n" % tuple(v))
        c = np.asarray(corners).reshape(-1, 3, 4)
        for tri in c:
            if tri[0, 1] >= 0:
                f.write("f %d//%d %d//%d %d//%d\n" % (tri[0, 0] + 1, tri[0, 1] + 1, tri[1, 0] + 1,
                                                       tri[1, 1] + 1, tri[2, 0] + 1, tri[2, 1] + 1))
            else:
                f.write("f %d %d %d\n" % (tri[0, 0] + 1, tri[1, 0] + 1, tri[2, 0] + 1))


def sun_sky(n: int = 64, sun_dir=(0.3, 0.8, 0.2), half_angle: float = 0.0047, sun_radiance=50000.0,
            sky_radiance=(0.5, 0.7, 1.0), ground_radiance=(0.3, 0.25, 0.2)) -> np.ndarray:
    """A sun-and-sky environment cube, float32 [6, n, n, 3] (envmap.py): texels whose centre lies
    above the horizon (y > 0) take sky_radiance, the others ground_radiance, and the sun -- the
    texels whose centre lies within half_angle of sun_dir, and always the texel sun_dir looks up --
    takes sun_radiance.  n must be even, so that the horizon is a texel boundary on the four side
    faces.  Radiances are scalars or RGB triples; the result is deterministic."""
    from .envmap import lookup, texel_directions

    if n < 2 or n % 2:
        raise ValueError("sun_sky: n must be even")
    d = texel_directions(n)[:, :, :, 0]
    s = np.asarray(sun_dir, dtype=np.float64)
    s = s / np.linalg.norm(s)
    out = np.where((d[..., 1] > 0)[..., None], np.broadcast_to(np.asarray(sky_radiance, np.float64), (3,)),
                   np.broadcast_to(np.asarray(ground_radiance, np.float64), (3,)))
    sun = (d @ s) >= np.cos(half_angle)
    sun.reshape(-1)[lookup(s, n)] = True
    out[sun] = np.broadcast_to(np.asarray(sun_radiance, np.float64), (3,))
    return out.astype(np.float32)
