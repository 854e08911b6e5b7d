"""The 4-wide quantised BVH walk (yart_b200/csrc/wide_bvh.cuh, the TRAVERSAL_AUTO default for scenes without
alpha-tested materials) against a float64 brute force, on the scenes where a box test goes wrong: tiny nodes seen
from far away, meshes far from the world origin (in their vertices or through node transforms), flat meshes, grazing
rays, huge extents and wide trees deep enough to reach the stack limit.

Checks per scene (`check_scene`):
  * closest hit: on every ray with a robust float64 hit (below) the wide walk returns that triangle, t within 1e-6;
    the wide walk never loses a hit the reference-order walk finds (didHit includes it, t no larger); where the two
    walks differ the wide walk's hit is a float64 hit of that triangle within 1e-5;
  * any hit at tMax = 0.5x, 1x, 2x the hit distance and one float ulp below / above it: every robustly occluded ray is
    occluded, and the wide walk's occlusions include the reference-order walk's.
The robust hits the reference-order walk misses are printed, not asserted: that is the reference's own slab test.

CPU part: the product sources compiled for the CPU (tests/hostsim).  `-m gpu`: the CUDA library, plus the wide
kernels' spill path and randomised scenes rendered with the default walk."""
import types

import numpy as np
import pytest

import harness as H
import yart_b200 as Y
from yart_b200 import scenes

U = 2.0 ** -24    # float32 unit roundoff
KTMIN = 0.001     # kTMin (traverse.cuh): testTriangle accepts t > kTMin
# Bound on the float32 rounding of one of testTriangle's products, relative to the product of its operands' norms:
# s = o - p0 (1 rounding), a cross product (2), a three-term dot product (3), the product by 1 / det (2).
GAMMA = 8 * U


# ------------------------------------------------------------------------------------------
# float64 brute force
# ------------------------------------------------------------------------------------------
def _pairs(o, d, v, o_err):
    """Möller–Trumbore in float64 for rays (o, d) x triangles v (m, 3, 3), with the float32 error bounds of
    testTriangle's arithmetic on the same inputs.

    The float32 evaluation of u = (s . (d x e2)) / det, v = (d . (s x e1)) / det, t = (e2 . (s x e1)) / det differs from
    the exact value by at most
        du, dv <= GAMMA |s| |d| (|e1| + |e2|) / |det| + 3 rd,   dt <= GAMMA |s| |e1| |e2| / |det| + |t| (rd + 3 U)
    with rd = GAMMA |e1| |d| |e2| / |det| the relative error of det (each rounding of a product or sum is relative to
    its operands, and |a . b| <= |a| |b|, |a x b| <= |a| |b|).  `o_err` (per ray) is an absolute uncertainty of the
    origin, e.g. the rounding of a node transform; it enters like the rounding of s.  A barycentric at least `du` from
    its edge therefore has the same sign in float32 and in float64: that is the margin delta of a robust hit."""
    e1, e2 = v[None, :, 1] - v[None, :, 0], v[None, :, 2] - v[None, :, 0]
    s = o[:, None] - v[None, :, 0]
    dd = d[:, None]
    pv = np.cross(dd, e2)
    det = np.einsum("rtk,rtk->rt", e1, pv)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        inv = 1.0 / det
        q = np.cross(s, e1)
        bu = np.einsum("rtk,rtk->rt", s, pv) * inv
        bv = np.einsum("rtk,rtk->rt", np.broadcast_to(dd, q.shape), q) * inv
        t = np.einsum("rtk,rtk->rt", e2, q) * inv
        n1, n2, nd = np.linalg.norm(e1, axis=-1), np.linalg.norm(e2, axis=-1), np.linalg.norm(dd, axis=-1)
        ns = np.linalg.norm(s, axis=-1) + o_err[:, None] / GAMMA
        ad = np.abs(det)
        rd = GAMMA * n1 * nd * n2 / ad
        delta = GAMMA * ns * nd * (n1 + n2) / ad + 3 * rd + 4 * U
        dt = GAMMA * ns * n1 * n2 / ad + np.abs(t) * (rd + 3 * U)
        bad = ~(rd < 0.5) | ~np.isfinite(t)
        delta, dt = np.where(bad, np.inf, delta), np.where(bad, np.inf, dt)
        possible = (bu >= -delta) & (bv >= -delta) & (bu + bv <= 1 + delta) & (t + dt > KTMIN) & (ad * (1 + rd) >= 1e-12)
        # float32 products that overflow (edges of ~1e13 and more) give testTriangle a NaN t, which it accepts: such a
        # triangle may "hit" any ray, at no distance the bound can place
        overflow = np.maximum(ns, nd) * n1 * n2 > 1e37
        possible, dt = possible | overflow, np.where(overflow, np.inf, dt)
        robust = ((bu >= delta) & (bv >= delta) & (bu + bv <= 1 - delta) & (t - dt > KTMIN * 1.001) & (ad * (1 - rd) > 1e-12)
                  & (dt <= 1e-5 * np.abs(t)) & ~overflow)
    return t, dt, possible, robust


def brute_force(o, d, v, o_err=None, chunk=1 << 21):
    """Per ray: (robust, prim, t).  A ray is robust when its nearest float64 hit is a robust hit (barycentrics at
    least delta inside, t - dt > kTMin, the float32 t within 1e-5) and no other triangle that float32 rounding could make a
    hit lies nearer than that hit's t (1 + 1e-5) plus the rounding of both."""
    o, d, v = (np.asarray(a, np.float64) for a in (o, d, v))
    n, m = len(o), len(v)
    o_err = np.zeros(n) if o_err is None else np.asarray(o_err, np.float64)
    best_t, best_p, best_dt = np.full(n, np.inf), np.full(n, -1), np.zeros(n)
    low = np.full((n, 2), np.inf)      # two smallest t - dt over possible hits, and their triangles
    low_p = np.full((n, 2), -1)
    rc = max(1, chunk // max(m, 1))
    tc = max(1, chunk // rc)
    for r0 in range(0, n, rc):
        rs = slice(r0, r0 + rc)
        for t0 in range(0, m, tc):
            t, dt, possible, robust = _pairs(o[rs], d[rs], v[t0:t0 + tc], o_err[rs])
            tr = np.where(robust, t, np.inf)
            j = tr.argmin(1)
            tj = tr[np.arange(len(j)), j]
            better = tj < best_t[rs]
            best_t[rs] = np.where(better, tj, best_t[rs])
            best_p[rs] = np.where(better, t0 + j, best_p[rs])
            best_dt[rs] = np.where(better, dt[np.arange(len(j)), j], best_dt[rs])
            key = np.where(possible, t - dt, np.inf)
            k2 = min(2, key.shape[1])
            idx = np.argpartition(key, k2 - 1, axis=1)[:, :k2]
            cand = np.concatenate([low[rs], np.take_along_axis(key, idx, 1)], 1)
            cand_p = np.concatenate([low_p[rs], t0 + idx], 1)
            order = np.argsort(cand, 1)[:, :2]
            low[rs], low_p[rs] = np.take_along_axis(cand, order, 1), np.take_along_axis(cand_p, order, 1)
    other = np.where(low_p[:, 0] == best_p, low[:, 1], low[:, 0])
    robust = np.isfinite(best_t) & (other > best_t * (1 + 1e-5) + best_dt)
    return robust, best_p, best_t, best_dt


def float64_hit(o, d, v, prim, t32, o_err=None):
    """True where (prim, t32) is a float64 hit of that triangle (possible within the float32 bounds), t within 1e-5."""
    o, d = np.asarray(o, np.float64), np.asarray(d, np.float64)
    o_err = np.zeros(len(o)) if o_err is None else o_err
    out = np.zeros(len(o), bool)
    for i in range(len(o)):
        t, dt, possible, _ = _pairs(o[i:i + 1], d[i:i + 1], np.asarray(v[prim[i]:prim[i] + 1], np.float64), o_err[i:i + 1])
        out[i] = possible[0, 0] and abs(float(t32[i]) - t[0, 0]) <= 1e-5 * abs(t[0, 0]) + dt[0, 0]
    return out


# ------------------------------------------------------------------------------------------
# scenes and rays (seeded numpy data written through yart_b200.scenes.Scene)
# ------------------------------------------------------------------------------------------
def mesh_scene(v, transforms=()):
    """One mesh of triangles v (m, 3, 3) under a chain of node transforms (outermost first)."""
    v = np.asarray(v, np.float32)
    m = len(v)
    e1, e2 = (v[:, 1] - v[:, 0]).astype(np.float64), (v[:, 2] - v[:, 0]).astype(np.float64)
    nrm = np.cross(e1, e2)
    nrm /= np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-300)
    faces = np.zeros((m, 4), np.uint32)
    faces[:, :3] = np.arange(3 * m).reshape(m, 3)
    s = scenes.Scene()
    s.materials = [scenes.Material(base=(0.7, 0.7, 0.7), roughness=1.0)]
    s.meshes = [scenes.Mesh(v.reshape(-1, 3), np.repeat(nrm, 3, 0), None, None, faces)]
    s.nodes = [scenes.Node(-1, -1)]
    for xf in transforms:
        s.nodes.append(scenes.Node(len(s.nodes) - 1, -1, xf))
    s.nodes[-1].mesh = 0
    return s


def cluster(rng, m, centre, half, size):
    """m random triangles of edge ~`size` with vertices in a cube of half-size `half` around `centre`."""
    c = np.asarray(centre, np.float64) + rng.uniform(-half, half, (m, 1, 3))
    return c + rng.uniform(-size, size, (m, 3, 3))


def aimed_rays(rng, v, n, dist, centre=None, grazing=None):
    """n float32 rays {o, tmin, d, tmax} from `dist` away, each aimed at a random interior point of a random triangle.
    grazing=(normal, lo, hi): directions at an angle in [lo, hi] radians to the plane with that normal."""
    v = np.asarray(v, np.float64)
    k = rng.integers(0, len(v), n)
    b = rng.dirichlet((1.0, 1.0, 1.0), n)
    target = np.einsum("ri,rik->rk", b, v[k])
    if grazing is None:
        w = rng.normal(size=(n, 3))
    else:
        nrm, lo, hi = grazing
        nrm = np.asarray(nrm, np.float64)
        tang = rng.normal(size=(n, 3))
        tang -= np.outer(tang @ nrm, nrm)
        tang /= np.linalg.norm(tang, axis=1, keepdims=True)
        a = rng.uniform(lo, hi, n) * rng.choice([-1.0, 1.0], n)
        w = np.cos(a)[:, None] * tang + np.sin(a)[:, None] * nrm
    w /= np.linalg.norm(w, axis=1, keepdims=True)
    o = (target + dist * w).astype(np.float32)
    d = (target - o.astype(np.float64)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.zeros((n, 8), np.float32)
    rays[:, :3], rays[:, 3], rays[:, 4:7], rays[:, 7] = o, KTMIN, d, np.inf
    return rays


def write(sc, tmp_path, name):
    path = str(tmp_path / f"{name}.ysc")
    sc.write(path)
    return path


def open_ctx(path, traversal):
    ctx = Y.Context(max_depth=1, traversal=traversal)
    ctx.upload_scene(Y.Scene(path))
    return ctx


def wide_active(ctx):
    """True when the context's scene runs the wide walk (TRACE_WIDE raises STATE otherwise)."""
    try:
        ctx.trace(np.zeros((1, 8), np.float32), Y.TRACE_CLOSEST | Y.TRACE_WIDE)
        return True
    except Y.YartError as e:
        assert "STATE" in str(e), e
        return False


def object_rays(rays, transforms):
    """The rays in the mesh's object space (float64 inverse of the node chain) and the absolute uncertainty of
    the float32 object-space origins the library forms (xformRows per level: one rounding per product and sum)."""
    o, d = rays[:, :3].astype(np.float64), rays[:, 4:7].astype(np.float64)
    err = np.zeros(len(rays))
    for xf in transforms:
        inv = np.linalg.inv(np.asarray(xf, np.float64))
        mag = np.abs(inv[:3, :3]) @ np.abs(o.T) + np.abs(inv[:3, 3:4])
        o, d = (inv[:3, :3] @ o.T + inv[:3, 3:4]).T, (inv[:3, :3] @ d.T).T
        err = err * np.abs(inv[:3, :3]).sum(1).max() + 4 * U * mag.max(0)
    return o, d, err


# ------------------------------------------------------------------------------------------
# the checks
# ------------------------------------------------------------------------------------------
def check_scene(tag, path, v, rays, transforms=()):
    """All checks of the module docstring on one scene; returns (robust rays, robust hits the reference-order walk
    misses, robust hits the wide walk misses)."""
    ctx = open_ctx(path, Y.TRAVERSAL_WIDE)
    o, d, o_err = object_rays(rays, transforms)
    robust, prim, t64, dt64 = brute_force(o, d, v, o_err)
    wide, _ = ctx.trace(rays, Y.TRACE_CLOSEST | Y.TRACE_WIDE)
    ref, _ = ctx.trace(rays, Y.TRACE_CLOSEST | Y.TRACE_REFERENCE_ORDER)
    wh, rh = wide["didHit"] == 1, ref["didHit"] == 1
    # t within 1e-6 of the float64 t, or within the bound on testTriangle's own rounding where that is larger
    wide_miss = robust & ~(wh & (wide["prim"] == prim) & (np.abs(wide["t"] - t64) <= np.maximum(1e-6 * t64, dt64)))
    ref_miss = robust & ~(rh & (ref["prim"] == prim))
    print(f"{tag}: {robust.sum()} of {len(rays)} rays with a robust hit; robust hits missed: reference-order walk "
          f"{ref_miss.sum()}, wide walk {wide_miss.sum()}; rays where the wide walk loses a reference-order hit "
          f"{(rh & np.isfinite(ref['t']) & ~(wh & (wide['t'] <= ref['t']))).sum()}")
    assert not wide_miss.any(), f"{tag}: the wide walk misses {wide_miss.sum()} robust hits, e.g. rays {np.nonzero(wide_miss)[0][:5]}"
    # a NaN t is no hit to keep: testTriangle's products overflow on triangles of edge ~1e13 and more, and its
    # `t <= kTMin || hit.t <= t` test lets the NaN through, wherever the box test puts the ray
    lost = rh & np.isfinite(ref["t"]) & ~(wh & (wide["t"] <= ref["t"]))
    assert not lost.any(), f"{tag}: the wide walk loses {lost.sum()} hits of the reference-order walk, e.g. rays {np.nonzero(lost)[0][:5]}"
    differ = wh & ~(rh & (wide["prim"] == ref["prim"]) & (wide["t"].view(np.uint32) == ref["t"].view(np.uint32)))
    if differ.any():
        ok = float64_hit(o[differ], d[differ], v, wide["prim"][differ], wide["t"][differ], o_err[differ])
        assert ok.all(), f"{tag}: {(~ok).sum()} wide hits are no float64 hit of their triangle"
    # any hit at finite tMax around the hit distance
    base = np.where(robust, t64, np.where(rh, ref["t"], 1.0)).astype(np.float32)
    for name, tmax in (("0.5x", base * np.float32(0.5)), ("1x", base), ("2x", base * np.float32(2)),
                       ("ulp below", np.nextafter(base, np.float32(0))), ("ulp above", np.nextafter(base, np.float32(np.inf)))):
        r = rays.copy()
        r[:, 7] = tmax
        aw, _ = ctx.trace(r, Y.TRACE_ANY | Y.TRACE_WIDE)
        ar, _ = ctx.trace(r, Y.TRACE_ANY | Y.TRACE_REFERENCE_ORDER)
        occluded = robust & (t64 * (1 + 1e-6) < tmax)
        assert (aw["didHit"][occluded] == 1).all(), f"{tag} any-hit {name}: {(aw['didHit'][occluded] == 0).sum()} robust occlusions missed"
        assert (aw["didHit"] >= ar["didHit"]).all(), \
            f"{tag} any-hit {name}: the wide walk misses {(aw['didHit'] < ar['didHit']).sum()} occlusions of the reference-order walk"
    ctx.close()
    return int(robust.sum()), int(ref_miss.sum()), int(wide_miss.sum())


def far_cluster(seed, half, size, dist, m=3000, n=3000):
    rng = np.random.default_rng(seed)
    v = cluster(rng, m, (0, 0, 0), half, size).astype(np.float32)
    return v, aimed_rays(rng, v, n, dist)


def offset_mesh(seed, centre, half, size, dist, m=3000, n=3000):
    rng = np.random.default_rng(seed)
    v = cluster(rng, m, centre, half, size).astype(np.float32)
    return v, aimed_rays(rng, v, n, dist)


def flat_scene(kind, seed=5, n=3000):
    rng = np.random.default_rng(seed)
    z = np.float32(0.375)
    if kind == "random":
        v = cluster(rng, 3000, (0, 0, 0), 5.0, 0.2)
        v[:, :, 2] = z
    else:  # a 40 x 40 grid of quads with shared edges (ties on the diagonals and edges)
        g = np.linspace(-4, 4, 41)
        x0, y0 = np.meshgrid(g[:-1], g[:-1])
        x1, y1 = x0 + (g[1] - g[0]), y0 + (g[1] - g[0])
        a, b = np.stack([x0, y0], -1).reshape(-1, 2), np.stack([x1, y0], -1).reshape(-1, 2)
        c, dd = np.stack([x1, y1], -1).reshape(-1, 2), np.stack([x0, y1], -1).reshape(-1, 2)
        tri = np.concatenate([np.stack([a, b, c], 1), np.stack([a, c, dd], 1)])
        v = np.concatenate([tri, np.full(tri.shape[:2] + (1,), z)], -1)
    v = v.astype(np.float32)
    graz = ((0.0, 0.0, 1.0), 1e-3, 2e-2) if kind == "grazing" else None
    return v, aimed_rays(rng, v, n, 20.0, grazing=graz)


def huge_scene(seed=9, biggest=1e34, n=3000):
    """Unit triangles mixed with triangles of edge 1e20 .. `biggest` (the wide grid's largest quanta)."""
    rng = np.random.default_rng(seed)
    small = cluster(rng, 1500, (0, 0, 0), 10.0, 0.5)
    size = 10.0 ** rng.uniform(20, np.log10(biggest), 300)
    big = rng.normal(size=(300, 3, 3)) * size[:, None, None]
    v = np.concatenate([small, big]).astype(np.float32)
    r_small = aimed_rays(rng, v[:1500], n // 2, 30.0)
    r_big = np.concatenate([aimed_rays(rng, v[1500 + i:1501 + i], n // 600, float(size[i]) * 3) for i in range(300)])
    return v, np.concatenate([r_small, r_big])


def chain_scene(n):
    """n unit triangles in the planes x = 1.6^k: the SAH tree is a chain (one triangle split off per level)."""
    x = 1.6 ** np.arange(n)
    v = np.zeros((n, 3, 3))
    v[:, :, 0] = x[:, None]
    v[:, 1, 1], v[:, 2, 2] = 1.0, 1.0
    v[:, :, 1:] -= 0.25
    return v.astype(np.float32)


def chain_rays(v, seed=3, n=2000):
    rng = np.random.default_rng(seed)
    rays = aimed_rays(rng, v, n, 1.0)
    # half of them along the chain, through every plane, from before its first triangle: these walk the whole depth
    k = n // 2
    rays[:k, 0] = 0.5
    rays[:k, 1:3] = rng.uniform(-0.2, 0.2, (k, 2))
    rays[:k, 4:7] = (1.0, 0.0, 0.0)
    return rays


FAR_CLUSTERS = {  # (half-size, triangle size, origin distance)
    "control_10_0.05_30": (10.0, 0.05, 30.0),
    "tiny_1e-3_1e-5_at_1e3": (1e-3, 1e-5, 1e3),
    "tiny_1e-2_1e-4_at_1e4": (1e-2, 1e-4, 1e4),
    "tiny_1e-3_1e-5_at_1e5": (1e-3, 1e-5, 1e5),
    "tiny_1e-2_1e-4_at_1e3": (1e-2, 1e-4, 1e3),
}
OFFSETS = {  # (centre, half-size, triangle size, origin distance)
    "offset_1e4_1_0.01_5": ((1e4, 1e4, 0.0), 1.0, 0.01, 5.0),
    "offset_1e5_1_0.01_5": ((1e5, 1e5, 0.0), 1.0, 0.01, 5.0),
    "offset_1e5_10_0.1_50": ((1e5, 1e5, 0.0), 10.0, 0.1, 50.0),
}
TRANSFORMS = {  # the offset_1e5_10 mesh, its object space near the origin
    "translated": [scenes.translation(1e5, 1e5, 0.0)],
    "nested_scaled": [scenes.translation(5e4, 1e5, 0.0), scenes.scaling(4.0) @ scenes.rotation_y(30),
                      scenes.translation(12500.0, 0.0, 0.0) @ scenes.scaling(0.5)],
}


def build_case(case):
    """(scene, triangles in object space, rays in world space, node transforms) of one named case."""
    kind, name = case.split(":")
    if kind == "far":
        v, rays = far_cluster(11, *FAR_CLUSTERS[name])
        return mesh_scene(v), v, rays, ()
    if kind == "offset":
        v, rays = offset_mesh(12, *OFFSETS[name])
        return mesh_scene(v), v, rays, ()
    if kind == "xform":
        vw, rays = offset_mesh(12, *OFFSETS["offset_1e5_10_0.1_50"])
        full = np.eye(4)
        for xf in TRANSFORMS[name]:
            full = full @ np.asarray(xf, np.float64)
        inv = np.linalg.inv(full)
        v = (np.einsum("ij,tkj->tki", inv[:3, :3], vw.astype(np.float64)) + inv[:3, 3]).astype(np.float32)
        return mesh_scene(v, TRANSFORMS[name]), v, rays, TRANSFORMS[name]
    if kind == "flat":
        v, rays = flat_scene(name)
        return mesh_scene(v), v, rays, ()
    if kind == "huge":
        v, rays = huge_scene()
        return mesh_scene(v), v, rays, ()
    raise KeyError(case)


CASES = ([f"far:{k}" for k in FAR_CLUSTERS] + [f"offset:{k}" for k in OFFSETS] + [f"xform:{k}" for k in TRANSFORMS]
         + ["flat:random", "flat:grid", "flat:grazing", "huge:1e34"])


def run_case(case, tmp_path):
    sc, v, rays, xf = build_case(case)
    path = write(sc, tmp_path, case.replace(":", "_"))
    with _closing(open_ctx(path, Y.TRAVERSAL_AUTO)) as ctx:
        assert wide_active(ctx), f"{case}: the wide walk is not active"
    return check_scene(case, path, v, rays, xf)


class _closing:
    def __init__(self, ctx):
        self.ctx = ctx

    def __enter__(self):
        return self.ctx

    def __exit__(self, *exc):
        self.ctx.close()


def wide_depth_limit_cases(tmp_path):
    """(largest chain length that still runs the wide walk, a chain length that does not)."""
    n_ok, n_deep = None, None
    for n in range(40, 200, 4):
        path = write(mesh_scene(chain_scene(n)), tmp_path, f"chain{n}")
        with _closing(open_ctx(path, Y.TRAVERSAL_AUTO)) as ctx:
            if wide_active(ctx):
                n_ok = n
            else:
                n_deep = n
                break
    assert n_ok is not None and n_deep is not None, "no chain length reaches the wide walk's depth limit"
    return n_ok, n_deep


def check_deep(tmp_path):
    n_ok, n_deep = wide_depth_limit_cases(tmp_path)
    # too deep: AUTO is the reference-order walk bit for bit, WIDE is refused without the sampler hint
    v = chain_scene(n_deep)
    path = write(mesh_scene(v), tmp_path, f"chain{n_deep}")
    rays = chain_rays(v)
    with _closing(open_ctx(path, Y.TRAVERSAL_AUTO)) as ctx:
        auto, _ = ctx.trace(rays, Y.TRACE_CLOSEST)
        ref, _ = ctx.trace(rays, Y.TRACE_CLOSEST | Y.TRACE_REFERENCE_ORDER)
        assert auto.tobytes() == ref.tobytes()
        r = rays.copy()
        r[:, 7] = 50.0
        assert ctx.trace(r, Y.TRACE_ANY)[0].tobytes() == ctx.trace(r, Y.TRACE_ANY | Y.TRACE_REFERENCE_ORDER)[0].tobytes()
    with pytest.raises(Y.YartError, match="UNSUPPORTED.*exceeds the traversal stack") as e:
        open_ctx(path, Y.TRAVERSAL_WIDE)
    assert "SAMPLERS_LIB" not in str(e.value)
    # the deepest chain the wide walk takes
    v = chain_scene(n_ok)
    path = write(mesh_scene(v), tmp_path, f"chain{n_ok}")
    return check_scene(f"chain of {n_ok}", path, v, chain_rays(v))


def check_refused_extent(tmp_path):
    """A mesh wider than the quantised grid can hold: no wide layout (AUTO = reference-order walk), WIDE refused."""
    rng = np.random.default_rng(4)
    v = np.concatenate([cluster(rng, 200, (0, 0, 0), 5.0, 0.5), [[[-3e37, 0, 0], [3e37, 0, 0], [0, 1e37, 1.0]]]]).astype(np.float32)
    path = write(mesh_scene(v), tmp_path, "too_wide")
    rays = aimed_rays(rng, v[:200], 500, 20.0)
    with _closing(open_ctx(path, Y.TRAVERSAL_AUTO)) as ctx:
        assert not wide_active(ctx)
        assert ctx.trace(rays)[0].tobytes() == ctx.trace(rays, Y.TRACE_CLOSEST | Y.TRACE_REFERENCE_ORDER)[0].tobytes()
    with pytest.raises(Y.YartError, match="UNSUPPORTED.*quantised grid") as e:
        open_ctx(path, Y.TRAVERSAL_WIDE)
    assert "SAMPLERS_LIB" not in str(e.value)


# ------------------------------------------------------------------------------------------
# CPU build of the product sources
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES)
def test_wide_walk_robust_hits_cpu_build(case, tmp_path, hostsim_lib):
    run_case(case, tmp_path)


def test_wide_walk_depth_limit_cpu_build(tmp_path, hostsim_lib):
    check_deep(tmp_path)


def test_wide_layout_refused_for_extents_beyond_the_grid_cpu_build(tmp_path, hostsim_lib):
    check_refused_extent(tmp_path)


# ------------------------------------------------------------------------------------------
# CUDA library
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_wide_walk_robust_hits_gpu(case, tmp_path, cuda_lib):
    run_case(case, tmp_path)


@pytest.mark.gpu
def test_wide_walk_depth_limit_gpu(tmp_path, cuda_lib):
    check_deep(tmp_path)


@pytest.mark.gpu
def test_wide_layout_refused_for_extents_beyond_the_grid_gpu(tmp_path, cuda_lib):
    check_refused_extent(tmp_path)


def _records_and_render(path, rays, sh_entries, cam):
    """Closest-hit and any-hit records and a 4-bounce render with the wide walk and `sh_entries` shared stack entries."""
    ctx = Y.Context(max_depth=4, traversal=Y.TRAVERSAL_WIDE, sh_stack_entries=sh_entries)
    ctx.upload_scene(Y.Scene(path))
    closest, _ = ctx.trace(rays, Y.TRACE_CLOSEST)
    r = rays.copy()
    r[:, 7] = np.where(closest["didHit"] == 1, closest["t"] * np.float32(1.5), np.float32(1e30))
    anyh, _ = ctx.trace(r, Y.TRACE_ANY)
    ctx.set_camera(Y.make_camera(160, 120, cam["focal"], 0.0, cam["pos"], cam["target"]))
    ctx.begin_frame(160, 120, 4, 64, (0.2, 0.2, 0.2), Y.TONEMAP_AGX)
    ctx.render_wave(0, 4, 0)
    hdr, ldr, st = ctx.resolve()
    ctx.close()
    return closest.tobytes(), anyh.tobytes(), hdr.tobytes(), ldr.tobytes(), int(st.raysReference)


@pytest.mark.gpu
def test_wide_kernels_spill_path_gives_identical_records_and_frames(tmp_path, cuda_lib):
    """With 2 or 3 shared stack entries per lane the wide kernels spill to global memory at once: the same hit
    records and the same 4-bounce frame as with the default shared stack, on the deepest chain the wide walk takes
    and on the 100 K soup."""
    n_ok, _ = wide_depth_limit_cases(tmp_path)
    v = chain_scene(n_ok)
    chain = (write(mesh_scene(v), tmp_path, "chain_spill"), chain_rays(v), dict(pos=(-5.0, 0.1, 0.2), target=(1e3, 0.0, 0.0), focal=35.0))
    soup_cam = H.scene_camera("soup")
    rng = np.random.default_rng(8)
    o = rng.uniform(-12, 12, (20000, 3))
    d = rng.normal(size=(20000, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    soup_rays = np.zeros((20000, 8), np.float32)
    soup_rays[:, :3], soup_rays[:, 3], soup_rays[:, 4:7], soup_rays[:, 7] = o, KTMIN, d, np.inf
    soup = (H.scene_file("soup", n_tris=100_000), soup_rays, soup_cam)
    for tag, (path, rays, cam) in (("chain", chain), ("soup", soup)):
        want = _records_and_render(path, rays, 0, cam)
        for sh in (2, 3):
            got = _records_and_render(path, rays, sh, cam)
            for what, a, b in zip(("closest", "any", "hdr", "ldr", "rays"), got, want):
                assert a == b, f"{tag}, {sh} shared entries: {what} differs from the default shared stack's"


def fuzz_integrator(seed):
    """The integrator the reference's frame of random scene `seed` was recorded with (test_fuzz_parity)."""
    return "naive" if 100 <= seed < 114 else "mis"


def wide_fuzz_seeds():
    """Randomised scenes (with recorded reference frames of the default samplers) that run the wide walk under
    TRAVERSAL_AUTO; most random scenes have alpha-tested materials and keep the reference-order walk."""
    out = []
    for seed in (*range(40), *range(100, 114)):
        ctx = Y.Context(max_depth=1, traversal=Y.TRAVERSAL_AUTO)
        ctx.upload_scene(Y.Scene(H.scene_file("random_scene", seed=seed)))
        if wide_active(ctx):
            out.append(seed)
        ctx.close()
    return out


@pytest.mark.gpu
def test_random_scenes_default_walk_meets_the_wide_bars(cuda_lib):
    """Randomised scenes rendered with the library's default walk: the reference-order frame matches the recorded
    reference first, then the default walk's frame meets the wide walk's bars against it (test_gpu_parity)."""
    from test_fuzz_parity import render_case
    from test_gpu_parity import _check_wide_frame
    seeds = wide_fuzz_seeds()
    print(f"random scenes that run the wide walk: {seeds}")
    assert len(seeds) >= 4
    for seed in seeds:
        d, hdr, ldr = render_case(seed, fuzz_integrator(seed), traversal=Y.TRAVERSAL_REFERENCE_ORDER)
        rec = H.recorded(f"random_scene_{seed}")
        assert H.digest(hdr) == rec["hdr"] and H.digest(ldr) == rec["ldr"] and d["total_rays"] == rec["rays"], seed
        ref = dict(hdr=hdr, ldr=ldr, rays=d["total_rays"])
        d, hdr, ldr = render_case(seed, fuzz_integrator(seed), traversal=Y.TRAVERSAL_AUTO)
        _check_wide_frame(f"random scene {seed}", ref, hdr, ldr, types.SimpleNamespace(raysReference=d["total_rays"]))
