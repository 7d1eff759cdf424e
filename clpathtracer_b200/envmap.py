"""Cube-map environments for modes 2 and 3 (CLSetEnvironment, DESIGN.md "Environment light").

A cube is float32 [6][n][n][3] linear RGB radiance.  Faces are +X, -X, +Y, -Y, +Z, -Z and follow the
OpenGL cube-map convention: a direction d picks the face of its largest component, and its face
coordinates are a = sc / |ma|, b = tc / |ma| from the table below.  Column i of a face covers
a in [2i/n - 1, 2(i+1)/n - 1), row j covers b likewise, so a skybox made for GL_TEXTURE_CUBE_MAP
looks the same here.

    face  sc   tc   ma        face  sc   tc   ma
    +X    -z   -y   x         -X    +z   -y   x
    +Y    +x   +z   y         -Y    +x   -z   y
    +Z    +x   -y   z         -Z    -x   -y   z
"""
from __future__ import annotations

import numpy as np


def face_points(face: int, a, b) -> np.ndarray:
    """The point of face `face` with face coordinates (a, b) on the unit cube (its (sc, tc, ma) is
    (a, b, +-1)), float64 [..., 3]."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    one = np.ones_like(a + b)
    a, b = a * one, b * one
    return np.stack({0: (one, -b, -a), 1: (-one, -b, a), 2: (a, one, b), 3: (a, -one, -b),
                     4: (a, -b, one), 5: (-a, -b, -one)}[face], axis=-1)


def texel_directions(n: int, sub: int = 1) -> np.ndarray:
    """Unit directions through a sub x sub grid of points centred in every texel, float64
    [6, n, n, sub * sub, 3]; sub = 1 gives the texel centres."""
    k = (np.arange(n)[:, None] + (np.arange(sub)[None, :] + 0.5) / sub).reshape(-1) / n * 2 - 1  # [n * sub]
    b, a = np.meshgrid(k, k, indexing="ij")
    out = np.stack([face_points(f, a, b) for f in range(6)])  # [6, n*sub, n*sub, 3]
    out /= np.linalg.norm(out, axis=-1, keepdims=True)
    out = out.reshape(6, n, sub, n, sub, 3).transpose(0, 1, 3, 2, 4, 5)
    return out.reshape(6, n, n, sub * sub, 3)


def lookup(d: np.ndarray, n: int) -> np.ndarray:
    """The texel index (face * n + row) * n + col that each direction d [..., 3] looks up, in float64
    (the fp32 definition of CLSetEnvironment may differ from this within rounding of a texel edge)."""
    d = np.asarray(d, dtype=np.float64)
    x, y, z = d[..., 0], d[..., 1], d[..., 2]
    ax, ay, az = np.abs(x), np.abs(y), np.abs(z)
    fx = (ax >= ay) & (ax >= az)
    fy = ~fx & (ay >= az)
    face = np.where(fx, np.where(x > 0, 0, 1), np.where(fy, np.where(y > 0, 2, 3), np.where(z > 0, 4, 5)))
    ma = np.where(fx, ax, np.where(fy, ay, az))
    sc = np.choose(face, [-z, z, x, x, x, -x])
    tc = np.choose(face, [-y, -y, z, -z, -y, -y])
    col = np.clip(((sc / ma + 1) * 0.5 * n).astype(np.int64), 0, n - 1)
    row = np.clip(((tc / ma + 1) * 0.5 * n).astype(np.int64), 0, n - 1)
    return (face * n + row) * n + col


def latlong_to_cube(img: np.ndarray, n: int, sub: int = 4) -> np.ndarray:
    """Resample an equirectangular image img [H, W, 3] (the format most HDR environments ship in)
    to a cube [6, n, n, 3]: each texel is the float64 mean of the image's nearest pixels at
    sub x sub points spread over the texel (a box filter).

    Convention: row 0 of the image is straight up (+y) and row H - 1 straight down; pixel (i, j)
    looks along theta = pi (i + 0.5) / H from +y and azimuth phi = 2 pi (j + 0.5) / W,
    d = (sin theta sin phi, cos theta, -sin theta cos phi): the left edge looks along -z, the
    quarter column along +x, the centre column along +z and the three-quarter column along -x."""
    img = np.asarray(img, dtype=np.float64)
    H, W = img.shape[:2]
    d = texel_directions(n, sub)
    theta = np.arccos(np.clip(d[..., 1], -1.0, 1.0))
    phi = np.mod(np.arctan2(d[..., 0], -d[..., 2]), 2 * np.pi)
    i = np.clip((theta / np.pi * H).astype(np.int64), 0, H - 1)
    j = np.clip((phi / (2 * np.pi) * W).astype(np.int64), 0, W - 1)
    return img[i, j].mean(axis=3).astype(np.float32)
