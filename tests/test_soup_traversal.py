"""Triangle-soup traversal against a topology-free reference: every soup builder, both trace entry points.

The reference is a numpy float32 restatement of the device's triangle test (csrc/dtraverse.cuh tri_test, ray_setup; the library is
built without contraction, so IEEE float32 in numpy reproduces it bit for bit) and of the reference's slab test (tests/bvh_checks.py).
For every ray and every triangle of a soup:
  A = the triangles the triangle test accepts with the ray's t_max,
  L = the members of A whose OWN box min/max(v0, v1, v2) passes the slab test with t_max.
A leaf box contains the boxes of its triangles and the slab test is monotone in the box, so whatever the builder, the candidates C a
traversal has to consider satisfy L <= C <= A.  Hence, for every builder:
  closest hit: a hit names a member of A with that triangle's (t, b0, b1, b2) bits; min t(A) <= t <= min t(L); L not empty => a hit
               (ties in t may name any tied triangle);
  any hit:     L not empty => 1, A empty => 0;
and for the reference SAH topology the device equals the oracle bit for bit, tie-break included (same topology, same candidates)."""
import ctypes as C

import numpy as np
import pytest
from bvh_checks import check_collapse, reference_leaves, slab_reference

import toy_cpu_pathtracing_b200 as tp
from toy_cpu_pathtracing_b200 import assets, capi, scenes
from toy_cpu_pathtracing_b200.assets import MeshData

f32, f64 = np.float32, np.float64
FMAX = float(np.finfo(f32).max)
STACK = 96                                     # TCPT_TRAVERSAL_STACK


# ---------------------------------------------------------------------------------------------------------- the restatement
def _gamma(n):                                 # gamma(n) = n eps / (1 - n eps), evaluated in float32 like the kernel's constants
    eps = f32(5.9604644775390625e-8)
    return float((f32(n) * eps) / (f32(1) - f32(n) * eps))


G2, G3, G5 = _gamma(2), _gamma(3), _gamma(5)


class _Numpy:
    where, fmax, abs = staticmethod(np.where), staticmethod(np.fmax), staticmethod(np.abs)

    @staticmethod
    def via_f64(a, b, c, d):                  # (float)(a * b - c * d) in double: the products are exact, one rounding to double, one to float
        return (a.astype(f64) * b.astype(f64) - c.astype(f64) * d.astype(f64)).astype(f32)


class _Torch:
    def __init__(self, torch):
        self.t = torch
        self.where, self.fmax, self.abs = torch.where, torch.fmax, torch.abs

    def via_f64(self, a, b, c, d):
        T = self.t
        return (a.to(T.float64) * b.to(T.float64) - c.to(T.float64) * d.to(T.float64)).to(T.float32)


def degenerate_flags(tris):
    """|e1 x e2|^2 == 0 with the host's float32 arithmetic (host_math.h cross3 / dot3)."""
    a, b = tris[:, 1] - tris[:, 0], tris[:, 2] - tris[:, 0]
    n = np.stack([a[:, 1] * b[:, 2] - b[:, 1] * a[:, 2], a[:, 2] * b[:, 0] - b[:, 2] * a[:, 0], a[:, 0] * b[:, 1] - b[:, 0] * a[:, 1]], 1)
    with np.errstate(under="ignore", over="ignore"):
        return ((n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2]) == 0


def instance_ray(rays):
    """The ray in the soup's own space: the identity instance transform applied with the kernel's arithmetic (xf_point / xf_vector:
    1 * x + 0 * y turns a -0.0 into +0.0, so the reciprocal direction the triangle test sees can differ from the Render-space one)."""
    one, zero = f32(1), f32(0)

    def xf(p, translate):                     # ((m0 x + m3 y) + m6 z) + m9, row by row, with m = identity
        rows = []
        for k in range(3):
            m = [one if a == k else zero for a in range(3)]
            v = (m[0] * p[:, 0] + m[1] * p[:, 1]) + m[2] * p[:, 2]
            rows.append(v + zero if translate else v)
        return np.stack(rows, 1).astype(f32)
    return xf(rays[:, :3], True), xf(rays[:, 3:6], False)


def tri_test(xp, v, deg, o, d, t_max):
    """tri_test + ray_setup of dtraverse.cuh for rays [R] x triangles [N]: v [1, N, 3 vertices, 3], deg [1, N], o / d [R, 1, 3], t_max [R, 1].
    Returns (accepted, t, b0, b1, b2), each [R, N]."""
    ax, ay, az = xp.abs(d[..., 0]), xp.abs(d[..., 1]), xp.abs(d[..., 2])
    kz = xp.where(ay > ax, 1, 0)
    kz = xp.where(az > xp.where(ay > ax, ay, ax), 2, kz)                  # strict '>': the first of equal components wins

    def pick(a, k):                                                         # component k (per ray) of a [..., 3]
        return xp.where(k == 0, a[..., 0], xp.where(k == 1, a[..., 1], a[..., 2]))
    kx, ky = (kz + 1) % 3, (kz + 2) % 3
    dz = pick(d, kz)
    sx, sy, sz = -pick(d, kx) / dz, -pick(d, ky) / dz, 1.0 / dz
    P = [v[:, :, i, :] - o for i in range(3)]                               # [R, N, 3]
    px = [pick(p, kx) for p in P]
    py = [pick(p, ky) for p in P]
    pz = [pick(p, kz) for p in P]
    px = [px[i] + sx * pz[i] for i in range(3)]
    py = [py[i] + sy * pz[i] for i in range(3)]
    e0 = px[2] * py[1] - py[2] * px[1]
    e1 = px[0] * py[2] - py[0] * px[2]
    e2 = px[1] * py[0] - py[1] * px[0]
    zero = (e0 == 0) | (e1 == 0) | (e2 == 0)
    e0 = xp.where(zero, xp.via_f64(px[2], py[1], py[2], px[1]), e0)
    e1 = xp.where(zero, xp.via_f64(px[0], py[2], py[0], px[2]), e1)
    e2 = xp.where(zero, xp.via_f64(px[1], py[0], py[1], px[0]), e2)
    ok = ~(((e0 < 0) | (e1 < 0) | (e2 < 0)) & ((e0 > 0) | (e1 > 0) | (e2 > 0)))
    det = (e0 + e1) + e2
    ok = ok & ~(det == 0)
    pz = [p * sz for p in pz]
    t_scaled = (e0 * pz[0] + e1 * pz[1]) + e2 * pz[2]
    tmd = t_max * det
    ok = ok & ~((det < 0) & ((t_scaled >= 0) | (t_scaled < tmd))) & ~((det > 0) & ((t_scaled <= 0) | (t_scaled > tmd)))
    inv_det = 1.0 / det
    t = t_scaled * inv_det
    max_zt = xp.fmax(xp.abs(pz[0]), xp.fmax(xp.abs(pz[1]), xp.abs(pz[2])))
    max_xt = xp.fmax(xp.abs(px[0]), xp.fmax(xp.abs(px[1]), xp.abs(px[2])))
    max_yt = xp.fmax(xp.abs(py[0]), xp.fmax(xp.abs(py[1]), xp.abs(py[2])))
    delta_z, delta_x, delta_y = G3 * max_zt, G5 * max_xt, G5 * max_yt
    delta_e = 2.0 * ((G2 * max_xt * max_yt + delta_y * max_xt) + delta_x * max_yt)
    max_e = xp.fmax(xp.abs(e0), xp.fmax(xp.abs(e1), xp.abs(e2)))
    delta_t = 3.0 * ((G3 * max_e * max_zt + delta_e * max_zt) + delta_z * max_e) * xp.abs(inv_det)
    ok = ok & ~(t < delta_t) & ~deg
    return ok, t, e0 * inv_det, e1 * inv_det, e2 * inv_det


def accepted_pairs_numpy(tris, rays, chunk=None):
    """All (ray, triangle) pairs in A: ray index, triangle index, (t, b0, b1, b2) as float32."""
    ol, dl = instance_ray(rays)
    deg = degenerate_flags(tris)[None]
    v = tris[None]
    chunk = chunk or max(1, (1 << 18) // max(1, len(tris)))
    out = []
    with np.errstate(all="ignore"):
        for lo in range(0, len(rays), chunk):
            sl = slice(lo, lo + chunk)
            ok, t, b0, b1, b2 = tri_test(_Numpy, v, deg, ol[sl, None], dl[sl, None], rays[sl, 6:7])
            r, j = np.nonzero(ok)
            out.append((r + lo, j, t[r, j], b0[r, j], b1[r, j], b2[r, j]))
    return [np.concatenate(c) for c in zip(*out)] if out else [np.zeros(0, np.int64)] * 2 + [np.zeros(0, f32)] * 4


def accepted_pairs_torch(tris, rays, device, chunk=8):
    """The same restatement in eager torch float32 / float64 on the GPU (one operation per kernel: nothing to contract)."""
    import torch
    xp = _Torch(torch)
    ol, dl = instance_ray(rays)
    v = torch.from_numpy(tris).to(device)[None]
    deg = torch.from_numpy(degenerate_flags(tris)).to(device)[None]
    O, D, TM = (torch.from_numpy(np.ascontiguousarray(a)).to(device) for a in (ol, dl, rays[:, 6:7]))
    out = []
    for lo in range(0, len(rays), chunk):
        ok, t, b0, b1, b2 = tri_test(xp, v, deg, O[lo:lo + chunk, None], D[lo:lo + chunk, None], TM[lo:lo + chunk])
        r, j = torch.nonzero(ok, as_tuple=True)
        out.append([x.cpu().numpy() for x in (r + lo, j, t[r, j], b0[r, j], b1[r, j], b2[r, j])])
    return [np.concatenate(c) for c in zip(*out)]


class Bracket:
    """A and L of every ray, and the checks of the module docstring."""

    def __init__(self, tris, rays, pairs):
        self.rays, self.n = rays, len(tris)
        r, j, t, b0, b1, b2 = pairs
        lo, hi = tris.min(axis=1), tris.max(axis=1)
        with np.errstate(divide="ignore"):
            ol, dl = instance_ray(rays)
            inv_l, inv_r = f32(1) / dl, f32(1) / rays[:, 3:6]
        # the triangle's own box passes with the ray in the soup's space and with the Render-space ray (the top-level box test)
        in_l = slab_reference(lo[j], hi[j], ol[r], inv_l[r], rays[r, 6]) & slab_reference(lo[j], hi[j], rays[r, :3], inv_r[r], rays[r, 6])
        R = len(rays)
        self.min_a = np.full(R, np.inf, f32); np.minimum.at(self.min_a, r, t)
        self.min_l = np.full(R, np.inf, f32); np.minimum.at(self.min_l, r[in_l], t[in_l])
        self.any_a = np.isfinite(self.min_a)
        self.any_l = np.isfinite(self.min_l)
        self.key = r.astype(np.int64) * self.n + j
        order = np.argsort(self.key)
        self.key = self.key[order]
        self.bits = np.stack([t, b0, b1, b2], 1).astype(f32).view(np.int32)[order]

    def check_closest(self, hits, what):
        hit = hits[:, 0] >= 0
        assert np.all(hits[hit, 0] == 0), f"{what}: a soup has one primitive"
        assert not np.any(self.any_l & ~hit), f"{what}: {np.count_nonzero(self.any_l & ~hit)} rays miss although a triangle's own box and test accept them: rays {np.nonzero(self.any_l & ~hit)[0][:8]}"
        idx = np.nonzero(hit)[0]
        k = idx.astype(np.int64) * self.n + hits[idx, 1]
        pos = np.minimum(np.searchsorted(self.key, k), max(len(self.key) - 1, 0))
        in_a = (len(self.key) > 0) & (self.key[pos] == k) if len(self.key) else np.zeros(len(k), bool)
        assert in_a.all(), f"{what}: hits name triangles the triangle test rejects: rays {idx[~in_a][:8]}"
        assert np.array_equal(self.bits[pos], hits[idx, 2:6]), f"{what}: t / barycentric bits differ from the restatement: rays {idx[np.any(self.bits[pos] != hits[idx, 2:6], 1)][:8]}"
        t = hits[idx, 2].view(f32)
        low, high = t < self.min_a[idx], t > self.min_l[idx]
        assert not low.any(), f"{what}: a hit nearer than every accepted triangle: rays {idx[low][:8]}"
        assert not high.any(), f"{what}: the true closest hit was dropped (t above min t of L): rays {idx[high][:8]}, t {t[high][:4]} vs {self.min_l[idx][high][:4]}"

    def check_any(self, flags, what):
        got = flags[:, 0]
        assert set(np.unique(got)) <= {0, 1}
        assert np.all(got[self.any_l] == 1), f"{what}: any-hit misses a triangle whose own box and test accept it: rays {np.nonzero(self.any_l & (got != 1))[0][:8]}"
        assert np.all(got[~self.any_a] == 0), f"{what}: any-hit reports a hit no triangle accepts: rays {np.nonzero(~self.any_a & (got != 0))[0][:8]}"


# ---------------------------------------------------------------------------------------------------------- soups
def _uniform(n, seed=42):
    m = assets.triangle_soup(n, seed)
    return m.positions[m.indices.reshape(-1)].reshape(-1, 3, 3).astype(f32)


def _rotated(n, seed=3):
    """One triangle shape turned about the origin: v2 = -(v0 + v1) exactly, so every centroid (v0 + v1 + v2) / 3 is exactly 0 and every
    Morton key is equal."""
    rng = np.random.default_rng(seed)
    q, _ = np.linalg.qr(rng.normal(size=(n, 3, 3)))
    a, b = (q @ np.array([0.4, 0.1, 0.0])).astype(f32), (q @ np.array([-0.1, 0.3, 0.05])).astype(f32)
    return np.stack([a, b, -(a + b)], 1).astype(f32)


def _duplicates(permute):
    base = _uniform(200, seed=11)
    if not permute:
        return np.concatenate([base] * 4)
    return np.concatenate([base, base[:, [1, 2, 0]], base[:, [0, 2, 1]], base[:, [2, 1, 0]]])


def _coplanar(n=1000, seed=5):
    rng = np.random.default_rng(seed)
    c = rng.uniform(-1, 1, (n, 1, 3)) + rng.uniform(-0.25, 0.25, (n, 3, 3))
    c[..., 2] = 0.0
    return c.astype(f32)


def _geometric(n, axes=1):
    """Triangle k of axis a in the plane (axis a) = 2^-k, over the unit square centred on that axis: box centres at geometric spacing.
    Each level of the binned builder peels a few planes off the chain, so its depth grows with the planes of all axes together: with
    axes = 3, 126 planes per axis (every one a normal float) give a stack bound of 95, just under the traversal stack, and 140 (the last
    ones subnormal) are refused.  With n = 200 the planes past 2^-126 are subnormal and those past 2^-149 round to x = 0: exact
    duplicates, whose tied t values sit in one SAH leaf of more than 16 items that the wide layout cuts into ranges (the cut-leaf
    tie-break, checked against the oracle)."""
    x = np.ldexp(1.0, -np.arange(n))
    out = []
    for a in range(axes):
        v = np.zeros((n, 3, 3))
        v[:, :, a] = x[:, None]
        b, c = (a + 1) % 3, (a + 2) % 3
        v[:, :, b] = [-0.5, 0.5, -0.5]
        v[:, :, c] = [-0.5, -0.5, 0.5]
        out.append(v)
    return np.concatenate(out).astype(f32)


def _degenerate(seed=9):
    """A uniform soup with exactly degenerate triangles (a repeated vertex, three points on an axis-parallel line) and tiny triangles
    near the origin whose |e1 x e2|^2 underflows to 0 in float32 (the triangle test would accept them; the degenerate flag must not)."""
    rng = np.random.default_rng(seed)
    t = _uniform(600, seed=seed)
    t[0::6, 1] = t[0::6, 0]
    line = t[3::6].copy()
    line[:, 1], line[:, 2] = line[:, 0], line[:, 0]
    line[:, 1, 0] += f32(0.1); line[:, 2, 0] += f32(0.25)
    t[3::6] = line
    s = 3e-13
    c = rng.uniform(-4e-12, 4e-12, (200, 1, 3))
    tiny = (c + np.array([[0, 0, 0], [s, 0, 0], [0, s, 0]]) @ _rot(rng, 200)).astype(f32)
    assert degenerate_flags(tiny).all()
    return np.concatenate([t, tiny])


def _rot(rng, n):
    q, _ = np.linalg.qr(rng.normal(size=(n, 3, 3)))
    return q


def _big_over_small():
    big = np.array([[[-3, -3, 0.5], [3, -3, 0.5], [0, 3, 0.5]]], f32)
    return np.concatenate([_uniform(999, seed=13) * f32(0.4), big])


SOUPS = {
    **{f"uniform{n}": (lambda n=n: _uniform(n)) for n in (1, 2, 3, 17, 1000, 4099)},
    **{f"rotated{n}": (lambda n=n: _rotated(n)) for n in (64, 65, 1000)},
    "duplicates": lambda: _duplicates(False), "duplicates_permuted": lambda: _duplicates(True),
    "coplanar": _coplanar, "geometric40": lambda: _geometric(40), "geometric200": lambda: _geometric(200),
    "geometric3x126": lambda: _geometric(126, 3), "geometric3x140": lambda: _geometric(140, 3),
    "degenerate": _degenerate, "big_over_small": _big_over_small,
    "scaled_1e-3": lambda: (_uniform(1000) * f32(1e-3)).astype(f32), "scaled_1e3": lambda: (_uniform(1000) * f32(1e3)).astype(f32),
    "translated": lambda: (_uniform(1000) + np.array([1e4, -1e4, 1e4], f32)).astype(f32),
}


# ---------------------------------------------------------------------------------------------------------- rays
def _unit(v):
    return (v / np.linalg.norm(v, axis=-1, keepdims=True)).astype(f32)


def _rays(o, d, t_max=FMAX):
    return np.concatenate([np.asarray(o, f32), np.asarray(d, f32), np.broadcast_to(np.asarray(t_max, f32), (len(o),))[:, None]], 1).astype(f32)


def first_rays(name, tris, seed=0):
    """Ray families that need no hit to start from: from a sphere, bench.py's pinhole grid, axis-parallel (with -0.0 components),
    from inside the soup, aimed at random triangles from close by, and (coplanar soup) grazing at 1e-3 .. 1e-6 rad."""
    import bench
    rng = np.random.default_rng(seed)
    lo, hi = tris.reshape(-1, 3).min(0).astype(f64), tris.reshape(-1, 3).max(0).astype(f64)
    c, ext = (lo + hi) / 2, max(float((hi - lo).max()), 1e-30)
    fam = {}
    o = c + 2 * ext * _unit(rng.normal(size=(768, 3)))
    fam["sphere"] = _rays(o, _unit(rng.uniform(lo, hi, (768, 3)) - o))
    _, d = bench.soup_rays_numpy(16)
    fam["bench"] = _rays(np.broadcast_to(c + np.array([0, 0, 1.5 * ext]), d.shape), d)
    n = 384
    d = np.zeros((n, 3), f32)
    axis, sign = rng.integers(0, 3, n), rng.choice([-1.0, 1.0], n)
    d[np.arange(n), axis] = sign
    d[rng.random((n, 3)) < 0.5] *= -1                                       # -0.0 in the other components
    d[np.arange(n), axis] = sign
    o = rng.uniform(lo, hi, (n, 3))
    o[: n // 2] -= d[: n // 2] * 2 * ext                                    # half start outside, half inside
    fam["axis"] = _rays(o, d)
    fam["inside"] = _rays(rng.uniform(lo, hi, (512, 3)), _unit(rng.normal(size=(512, 3))))
    j = rng.integers(0, len(tris), 512)
    w = rng.dirichlet([1, 1, 1], 512)
    p = np.einsum("nk,nkc->nc", w, tris[j].astype(f64))
    size = np.linalg.norm(tris[j, 1].astype(f64) - tris[j, 0], axis=1) + np.linalg.norm(tris[j, 2].astype(f64) - tris[j, 0], axis=1)
    d = _unit(rng.normal(size=(512, 3)))
    fam["aimed"] = _rays(p - d * (2 * size + 1e-30)[:, None], d)
    if name == "coplanar":
        g = []
        for theta in (1e-3, 1e-4, 1e-5, 1e-6):
            phi = rng.uniform(0, 2 * np.pi, 128)
            d = np.stack([np.cos(theta) * np.cos(phi), np.cos(theta) * np.sin(phi), -np.sin(theta) * np.ones(128)], 1)
            p = np.concatenate([rng.uniform(-0.9, 0.9, (128, 2)), np.zeros((128, 1))], 1)
            g.append(_rays(p - d * 1.5, d))
        fam["grazing"] = np.concatenate(g)
    return fam


def second_rays(first, tris, bracket):
    """Ray families built from the first ones' reference hits: bench.py's bounce rays, and the sphere rays again with t_max = 0, a
    short t_max, and t_max = exactly the bits of their closest accepted t."""
    import bench
    fam, off = {}, 0
    starts = {}
    for k, r in first.items():
        starts[k] = off; off += len(r)
    b = first["bench"]
    s = slice(starts["bench"], starts["bench"] + len(b))
    hit = bracket.any_a[s]
    o2, d2 = bench.soup_bounce_numpy(b[:, :3], b[:, 3:6], np.where(hit, bracket.min_a[s], 0), hit, seed=1)
    if len(o2):
        fam["bounce"] = _rays(o2, d2)
    sp = first["sphere"]
    s = slice(starts["sphere"], starts["sphere"] + len(sp))
    lo, hi = tris.reshape(-1, 3).min(0), tris.reshape(-1, 3).max(0)
    fam["tmax0"] = _rays(sp[:, :3], sp[:, 3:6], 0.0)
    fam["tmax_short"] = _rays(sp[:, :3], sp[:, 3:6], np.linalg.norm(sp[:, :3] - (lo + hi) / 2, axis=1))
    hit = bracket.any_a[s]
    if hit.any():
        fam["tmax_exact"] = _rays(sp[hit, :3], sp[hit, 3:6], bracket.min_a[s][hit])
    return fam


_CASES = {}


def case(name, pairs_fn=None):
    """(triangles, rays, Bracket) of a soup: all ray families of the soup in one array, the reference computed once."""
    if name not in _CASES:
        tris = SOUPS[name]()
        first = first_rays(name, tris)
        r1 = np.concatenate(list(first.values()))
        p1 = accepted_pairs_numpy(tris, r1)
        r2 = np.concatenate(list(second_rays(first, tris, Bracket(tris, r1, p1)).values()))
        p2 = accepted_pairs_numpy(tris, r2)
        p2[0] = p2[0] + len(r1)
        rays = np.concatenate([r1, r2])
        _CASES[name] = (tris, rays, Bracket(tris, rays, [np.concatenate([a, b]) for a, b in zip(p1, p2)]))
    return _CASES[name]


# ---------------------------------------------------------------------------------------------------------- scenes
def _mesh(tris):
    n = len(tris)
    return MeshData(tris.reshape(-1, 3), np.tile(np.array([[0, 0, 1]], f32), (3 * n, 1)), None, np.arange(3 * n, dtype=np.uint32).reshape(n, 3))


def host_scene(tris, binned, require_gpu=True):
    """The soup as one mesh primitive (identity transform, camera at the origin: Render space = world space), BVH built on the host."""
    s = tp.Scene(device=0, require_gpu=require_gpu)
    if binned:
        s.ctx.set_option("binned_builder", 1)
    s.create_primitive(tp.CreatePrimitiveDesc.GeometryPrimitive(s.load_obj(_mesh(tris)), scenes._lambert(0.5, 0.5, 0.5), tp.Transform.identity()))
    s.build(tp.Camera(45.0, 8, 8))
    return s


def device_soup(tris, leaf):
    s = tp.Scene(device=0)
    s.ctx.set_option("soup_leaf", leaf)
    s.build_soup(tris)
    return s


BUILDERS = ["lbvh1", "lbvh2", "lbvh4", "lbvh16", "binned", "sah"]


def build(tris, builder):
    """The scene, or None when the build is refused with TCPT_ERR_LIMIT (a BVH deeper than the traversal stack): nothing else is accepted."""
    try:
        if builder.startswith("lbvh"):
            return device_soup(tris, int(builder[4:]))
        return host_scene(tris, builder == "binned")
    except capi.TcptError as e:
        assert e.code == capi.TCPT_ERR_LIMIT, str(e)
        return None


@pytest.fixture(scope="module")
def oracle_of(tables):
    from oracle import oracle
    cache = {}

    def get(name):
        if name not in cache:
            tris = case(name)[0]
            s = tp.Scene(device=0, describe_only=True)
            s.create_primitive(tp.CreatePrimitiveDesc.GeometryPrimitive(s.load_obj(_mesh(tris)), scenes._lambert(0.5, 0.5, 0.5), tp.Transform.identity()))
            cache[name] = oracle.scene_from_description(s.desc, np.zeros(3, f32), tables[0], tables[1])
        return cache[name]
    return get


# ---------------------------------------------------------------------------------------------------------- CPU tests
@pytest.mark.parametrize("name", list(SOUPS))
def test_the_restatement_brackets_the_oracle(oracle_of, name):
    """The oracle (reference topology) satisfies the bracket, and on its hit triangle the restatement has its t / barycentric bits."""
    tris, rays, br = case(name)
    orc = oracle_of(name)
    closest, _, _ = orc.trace(rays)
    any_hit, _, _ = orc.trace(rays, any_hit=True)
    br.check_closest(closest, f"oracle {name}")
    br.check_any(any_hit, f"oracle {name}")
    assert br.any_l.any() and (closest[:, 0] >= 0).any()


def test_restatement_details():
    """Hand-checked corners: -0.0 through the identity transform, the strict '>' of the shear axis, the degenerate flag."""
    o, d = instance_ray(_rays([[1, 2, 3]], [[-0.0, 0.0, -1.0]]))
    assert np.signbit(d[0, 0]) == False and d[0, 2] == -1          # noqa: E712  1 * -0 + 0 * 0 = +0
    tri = np.array([[[-1, -1, 0], [1, -1, 0], [0, 1, 0]]], f32)
    pairs = accepted_pairs_numpy(tri, _rays([[0, 0, 1], [0, 0, 1], [0.2, 0.1, -2]], [[0, 0, -1], [0.6, 0.6, -0.6], [0, 0, 1]]))
    r, j, t = pairs[0], pairs[1], pairs[2]
    assert list(r) == [0, 2] and t[0] == 1.0 and t[1] == 2.0
    assert degenerate_flags(np.array([[[0, 0, 0], [1, 1, 1], [2, 2, 2]], [[1, 0, 0], [0, 1, 0], [0, 0, 1]]], f32)).tolist() == [True, False]


def _dump_tree(ref):
    """Reference-order dump -> list of nodes (kind, box lo/hi float32, children / items)."""
    nodes, i, index = [], 0, {}
    while i < len(ref):
        index[i] = len(nodes)
        kind, value = int(ref[i, 0]), int(ref[i, 1])
        box = ref[i, 2:8].view(f32)
        if kind == 1:
            nodes.append((1, box, [int(ref[i + 1 + k, 1]) for k in range(value)], i))
            i += 1 + value
        else:
            nodes.append((0, box, (i + 1, i + value), i))
            i += 1
    return nodes, index


@pytest.mark.parametrize("name,n_expect_leaf", [("uniform1000", None), ("rotated1000", None), ("duplicates", None), ("coplanar", None),
                                                ("geometric40", None), ("geometric200", None), ("geometric3x126", None), ("geometric3x140", None),
                                                ("degenerate", None), ("big_over_small", None),
                                                ("translated", None), ("same_box40", 40), ("same_box100", None)])
def test_binned_builder_structure(tables, name, n_expect_leaf):
    """BinnedBuilder (option binned_builder) on a host-only context: a partition of the triangles into leaves, exact boxes, leaves that
    survive the 4-wide collapse, and a stack bound under the traversal stack or TCPT_ERR_LIMIT."""
    if name.startswith("same_box"):      # every box centre equal: the split-by-count branch (one leaf up to 64 items, halves above)
        tris = np.repeat(_uniform(1, seed=2), int(name[8:]), axis=0)
    else:
        tris = SOUPS[name]()
    try:
        s = host_scene(tris, True, require_gpu=False)
    except capi.TcptError as e:
        assert e.code == capi.TCPT_ERR_LIMIT, str(e)
        return
    depth = s.ctx.stats()["max_bvh_depth"]
    assert 0 < depth < STACK
    ref = s.get_bvh(0)
    leaves = reference_leaves(ref)
    items = np.concatenate([np.array(it, np.int64) for _, it in leaves])
    assert np.array_equal(np.sort(items), np.arange(len(tris))), "every triangle in exactly one leaf"
    tlo, thi = tris.min(axis=1), tris.max(axis=1)
    nodes, index = _dump_tree(ref)
    def bounds(k):
        kind, box, x, _ = nodes[k]
        if kind == 1:
            return np.concatenate([tlo[x].min(0), thi[x].max(0)])
        a, b = nodes[index[x[0]]][1], nodes[index[x[1]]][1]
        return np.concatenate([np.minimum(a[:3], b[:3]), np.maximum(a[3:], b[3:])])
    for k, (kind, box, x, _) in enumerate(nodes):
        assert np.array_equal(box, bounds(k).astype(f32)), f"node {k}: box is not the exact bound of its {'items' if kind else 'children'}"
    check_collapse(s, 0, len(tris))
    if n_expect_leaf:
        assert len(leaves) == 1 and len(leaves[0][1]) == n_expect_leaf
    if name == "same_box100":
        assert sorted(len(it) for _, it in leaves) == [50, 50]


def test_the_deep_soups_are_deep(tables):
    """What the deep soups exercise on the host builders: a binned stack bound just under the traversal stack, a binned build refused
    with TCPT_ERR_LIMIT, and a reference-topology leaf of tied duplicates cut into ranges."""
    s = host_scene(SOUPS["geometric3x126"](), True, require_gpu=False)
    assert s.ctx.stats()["max_bvh_depth"] == STACK - 1
    with pytest.raises(capi.TcptError) as e:
        host_scene(SOUPS["geometric3x140"](), True, require_gpu=False)
    assert e.value.code == capi.TCPT_ERR_LIMIT
    tris = SOUPS["geometric200"]()
    s = host_scene(tris, False, require_gpu=False)
    big = max((it for _, it in reference_leaves(s.get_bvh(0))), key=len)
    assert len(big) > 16 and np.count_nonzero(tris[big, 0, 0] == 0) > 1


def test_build_soup_refusals_need_no_device():
    """Malformed soup builds are refused before the device is touched: n = 0 and a leaf size outside [1, 16] are TCPT_ERR_INVALID."""
    ctx = capi.Context(0, require_gpu=False)
    tri = np.zeros(9, f32)
    p = capi.as_ptr(tri, C.c_float)
    assert ctx.lib.tcpt_scene_build_soup(ctx.handle, p, 0) == capi.TCPT_ERR_INVALID
    for leaf in (0, 17, -1):
        ctx.set_option("soup_leaf", leaf)
        assert ctx.lib.tcpt_scene_build_soup(ctx.handle, p, 1) == capi.TCPT_ERR_INVALID
        assert "soup_leaf" in ctx.last_error()
    ctx.set_option("soup_leaf", 4)
    if not ctx.has_gpu:
        assert ctx.lib.tcpt_scene_build_soup(ctx.handle, p, 1) == capi.TCPT_ERR_CUDA


# ---------------------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("builder", BUILDERS)
@pytest.mark.parametrize("name", list(SOUPS))
def test_soup_traversal_satisfies_the_bracket(oracle_of, name, builder):
    tris, rays, br = case(name)
    sc = build(tris, builder)
    if sc is None:
        assert name.startswith("geometric"), f"{name} / {builder}: only the deep soups may be refused"
        return
    closest, flags = sc.trace(rays), sc.trace(rays, any_hit=True)
    br.check_closest(closest, f"{name} / {builder}")
    br.check_any(flags, f"{name} / {builder}")
    if builder == "sah":
        orc = oracle_of(name)
        oc, _, _ = orc.trace(rays)
        oa, _, _ = orc.trace(rays, any_hit=True)
        assert np.array_equal(closest, oc), f"{name}: the device and the oracle disagree on rays {np.nonzero(np.any(closest != oc, 1))[0][:8]}"
        assert np.array_equal(flags, oa)


def _soa(rays, torch, dev):
    n = len(rays)
    q = np.zeros((2 * n, 4), f32)
    q[:n, :3], q[:n, 3], q[n:, :3] = rays[:, :3], rays[:, 6], rays[:, 3:6]
    return torch.from_numpy(q).to(dev)


def _records(hits, n):
    """tcpt_trace_device's hit buffer -> {prim, tri, t, b0, b1, b2} int32 rows."""
    h = hits.cpu().numpy()
    tb = h[: n * 16].view(np.int32).reshape(n, 4)
    pt = h[n * 16: n * 24].view(np.int32).reshape(n, 2)
    return np.concatenate([pt, tb], 1)


@pytest.mark.gpu
def test_trace_device_on_its_own_stream():
    """tcpt_trace_device in the SoA layout bench.py packs, on a non-default torch stream, gives tcpt_trace's records for ray counts that
    leave partial warps and chunks; n = 0 writes nothing; any hit leaves prim 0 / -1; a second call into the same buffer wins."""
    import torch
    tris, rays, br = case("uniform4099")
    sc = device_soup(tris, 4)
    ctx, dev = sc.ctx, "cuda:0"
    stream = torch.cuda.Stream(device=dev)

    def trace_dev(r_t, n, any_hit, hits):
        ctx.check(ctx.lib.tcpt_trace_device(ctx.handle, C.c_void_p(r_t.data_ptr()), n, int(any_hit), C.c_void_p(hits.data_ptr()), C.c_void_p(stream.cuda_stream)))

    for n in (1, 31, 32, 33, 127, 129, 4097):
        sub = rays[np.random.default_rng(n).choice(len(rays), n, replace=False)]
        with torch.cuda.stream(stream):
            r_t = _soa(sub, torch, dev)
            hits = torch.full((n * 24,), 0xAB, dtype=torch.uint8, device=dev)
            trace_dev(r_t, n, False, hits)
            stream.synchronize()
            got = _records(hits, n)
            want = sc.trace(sub)
            miss = want[:, 0] < 0
            assert np.array_equal(got[:, 0], want[:, 0]), n
            assert np.array_equal(got[~miss], want[~miss]), n
            trace_dev(r_t, n, True, hits)
            stream.synchronize()
            got = _records(hits, n)
            assert set(np.unique(got[:, 0])) <= {0, -1}
            assert np.array_equal(got[:, 0] == 0, sc.trace(sub, any_hit=True)[:, 0] == 1), n
    # n = 0: TCPT_OK, nothing written
    hits = torch.full((64,), 0x5A, dtype=torch.uint8, device=dev)
    r_t = _soa(rays[:1], torch, dev)
    trace_dev(r_t, 0, False, hits)
    stream.synchronize()
    assert bool((hits == 0x5A).all())
    # two calls back to back into one buffer: the second call's records
    a, b = rays[:1000], rays[1000:2000]
    with torch.cuda.stream(stream):
        ra, rb = _soa(a, torch, dev), _soa(b, torch, dev)
        hits = torch.empty(1000 * 24, dtype=torch.uint8, device=dev)
        trace_dev(ra, 1000, False, hits)
        trace_dev(rb, 1000, False, hits)
        stream.synchronize()
    got, want = _records(hits, 1000), sc.trace(b)
    hit = want[:, 0] >= 0
    assert np.array_equal(got[:, 0], want[:, 0]) and np.array_equal(got[hit], want[hit])


@pytest.mark.gpu
@pytest.mark.parametrize("builder", ["lbvh1", "binned"])
def test_count_tests(builder):
    """count_tests = 1: the same records; box / triangle test totals identical across runs and across the two entry points (each ray's
    walk is independent of scheduling); at least one triangle test per hit."""
    import torch
    tris, rays, br = case("uniform4099")
    sc = build(tris, builder)
    ctx = sc.ctx
    plain = {ah: sc.trace(rays, any_hit=ah) for ah in (False, True)}
    ctx.set_option("count_tests", 1)
    try:
        for ah in (False, True):
            counts = []
            for _ in range(2):
                assert np.array_equal(sc.trace(rays, any_hit=ah), plain[ah])
                st = ctx.stats()
                counts.append((st["box_tests"], st["tri_tests"]))
            n = len(rays)
            r_t = _soa(rays, torch, "cuda:0")
            hits = torch.empty(n * 24, dtype=torch.uint8, device="cuda:0")
            stream = torch.cuda.Stream()
            ctx.check(ctx.lib.tcpt_trace_device(ctx.handle, C.c_void_p(r_t.data_ptr()), n, int(ah), C.c_void_p(hits.data_ptr()), C.c_void_p(stream.cuda_stream)))
            st = ctx.stats()
            counts.append((st["box_tests"], st["tri_tests"]))
            assert counts[0] == counts[1] == counts[2], counts
            n_hits = int((plain[ah][:, 0] >= 0).sum()) if not ah else int(plain[ah][:, 0].sum())
            assert counts[0][1] >= n_hits > 0 and counts[0][0] > 0
    finally:
        ctx.set_option("count_tests", 0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["geometric200", "geometric3x126", "geometric3x140"])
def test_device_soup_depth_on_the_deep_soups(name):
    """The device LBVH quantises centroids to 21 bits per axis, so geometric spacing ends in equal Morton keys after about 21 planes per
    axis; the stack bound it reports is 3 levels + 4, and a build either stays under the traversal stack or is refused with TCPT_ERR_LIMIT."""
    sc = build(SOUPS[name](), "lbvh1")
    if sc is None:
        return
    levels, depth = sc.soup_build_info()["levels"], sc.ctx.stats()["max_bvh_depth"]
    print(f"{name}: {levels} wide levels, stack bound {depth}")
    assert depth == 3 * levels + 4 < STACK
    assert levels >= 12


@pytest.mark.gpu
def test_build_soup_refusals_leave_a_working_context():
    tris, rays, br = case("uniform1000")
    sc = device_soup(tris, 2)
    ctx = sc.ctx
    with pytest.raises(capi.TcptError) as e:
        sc.build_soup(tris[:0])
    assert e.value.code == capi.TCPT_ERR_INVALID
    for leaf in (0, 17):
        ctx.set_option("soup_leaf", leaf)
        with pytest.raises(capi.TcptError) as e:
            sc.build_soup(tris)
        assert e.value.code == capi.TCPT_ERR_INVALID
        br.check_closest(sc.trace(rays), f"the scene built before the refusal (leaf {leaf})")
    ctx.set_option("soup_leaf", 16)
    sc.build_soup(tris)
    br.check_closest(sc.trace(rays), "after the refusals")
    br.check_any(sc.trace(rays, any_hit=True), "after the refusals")


@pytest.mark.gpu
def test_torch_restatement_matches_numpy():
    """The eager-torch restatement (used for the bench-scale soup) gives the numpy restatement's pairs bit for bit."""
    for name in ("uniform1000", "coplanar", "degenerate", "translated"):
        tris, rays, _ = case(name)
        a, b = accepted_pairs_numpy(tris, rays), accepted_pairs_torch(tris, rays, "cuda:0")
        oa, ob = np.lexsort((a[1], a[0])), np.lexsort((b[1], b[0]))
        assert np.array_equal(a[0][oa], b[0][ob]) and np.array_equal(a[1][oa], b[1][ob]), name
        for x, y in zip(a[2:], b[2:]):
            assert np.array_equal(x[oa].view(np.int32), y[ob].view(np.int32)), name


@pytest.mark.gpu
def test_bench_scale_soup():
    """The 1 M soup of bench.py's soup_1M (LBVH leaf 1 and 4, binned builder) on a seeded subsample of its coherent and bounce rays.
    Every builder here gets the soup in world space and the rays from the camera at (0, 0, 3), which is what bench.py traces with the
    device builder.  With --soup-builder host, bench.py builds the soup and its light quad in Render space (camera at the origin), so
    its binned tree and rays are a translated copy of these: the binned builder is checked on the soup's triangles, not on those bits."""
    import bench
    tris = _uniform(1_000_000, seed=42)                         # scenes.load_soup's soup
    _, d = bench.soup_rays_numpy(4096)
    rng = np.random.default_rng(2024)
    sel = rng.choice(len(d), 1024, replace=False)
    prim = _rays(np.broadcast_to(np.array([0, 0, 3], f32), (1024, 3)), d[sel])          # the camera at (0, 0, 3): world space
    bp = Bracket(tris, prim, accepted_pairs_torch(tris, prim, "cuda:0"))
    o2, d2 = bench.soup_bounce_numpy(prim[:, :3], prim[:, 3:6], np.where(bp.any_a, bp.min_a, 0), bp.any_a, seed=1)
    rays = np.concatenate([prim, _rays(o2, d2)])
    br = Bracket(tris, rays, accepted_pairs_torch(tris, rays, "cuda:0"))
    assert br.any_l.mean() > 0.1
    for builder in ("lbvh1", "lbvh4", "binned"):
        sc = build(tris, builder)
        br.check_closest(sc.trace(rays), f"soup_1M / {builder}")
        br.check_any(sc.trace(rays, any_hit=True), f"soup_1M / {builder}")
        del sc
