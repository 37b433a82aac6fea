"""Closest-hit on adversarial rays, bit for bit against the f32 mirror of the device arithmetic (oracle/gpu_f32.hpp: every
primitive in id order, no tree, no boxes): ids, t, p, n and front_face with zero tolerance.  Every case runs with both BVH
builders (fresh handles: the tree is built at upload), under the automatic slab-test choice and under B200RT_FAST_SLAB=0,
on small scenes staged in shared memory and on a 1e5-sphere scene read through L1.  Boxes only cull, so whatever the tree
and the slab form, the device must find what the mirror finds.

Ray families: power-of-two scaled directions (metamorphic), zero / subnormal / below-the-clamp direction components, short
directions, tangent and grazing rays at the points where primitives touch their boxes, origins on faces, inside primitives
and inside the box padding, t_min / t_max at the hit and one ulp either side, origins either side of the fast-slab
origin limit, and NaN / inf components inside ordinary batches.

Where f32 cannot follow the f64 reference the rays are compared with the mirror only: d.d overflows above |d| ~ 1.8e19 and
becomes subnormal below |d| ~ 1e-19, so the f64 oracle (`decidable` margins) checks only the unit-scale rays."""
import math

import numpy as np
import pytest

from common import decidable

pytestmark = pytest.mark.gpu
INF = float("inf")
F = np.float32
EPS = 1.1920929e-7


# ---- scenes ---------------------------------------------------------------------------------------------------------------
def _built(rt, geoms):
    b = rt.SceneBuilder()
    for g in geoms:
        b.add(g, rt.Lambertian(rt.TextureLoader.solid(0.5, 0.5, 0.5)))
    return b.finalize()


SCENES = {
    "two_spheres": lambda rt: _built(rt, [rt.Sphere((0, 5, 0), 1.0), rt.Sphere((0, -5, 0), 1.0)]),
    "rects": lambda rt: _built(rt, [rt.xy_rect(-1, 1, -1, 1, -2), rt.yz_rect(-1, 1, -1, 1, 3), rt.xz_rect(-1, 1, -1, 1, -3)]),
    # a unit box, slabs thinner than the box padding (4e-6 x 3 = 1.2e-5) in x and in z, a zero-thickness box
    "boxes": lambda rt: _built(rt, [rt.RectBox((0, 0, 0), (1, 1, 1)), rt.RectBox((2, 0, 0), (2 + 1e-6, 1, 1)),
                                    rt.RectBox((-3, -1, -1), (-1, 1, -1 + 1e-7)), rt.RectBox((0, 2, 0), (1, 2, 1))]),
    # the ground spans the scene: it is tested up front, outside the tree
    "ground": lambda rt: _built(rt, [rt.xz_rect(-1000, 1000, -1000, 1000, 0), rt.Sphere((0, 1, 0), 1.0), rt.Sphere((3, 0.5, 0), 0.5),
                                     rt.RectBox((-3, 0, -1), (-2, 1, 1))]),
    "weekend": lambda rt: rt.Scene.named("random", seed=0xDEADBEEF),
    "large": lambda rt: rt.Scene.named("scaled", seed=11, param=158),
}


class Prims:
    """The primitives of a scene description, as the host uploads them."""

    def __init__(self, rt, desc):
        d = desc.contents
        self.spheres, self.rects, self.boxes = [], [], []        # (id, centre, r) / (id, type, d1, d2, dn, bounds, offset) / (id, lo, hi)
        for i in range(d.n_prims):
            p = d.prims[i]
            if p.type == rt._ffi.PRIM_SPHERE:
                s = d.spheres[p.index]
                self.spheres.append((i, np.array([s.cx, s.cy, s.cz], F), F(s.radius)))
            elif p.type == rt._ffi.PRIM_BOX:
                b = d.boxes[p.index]
                self.boxes.append((i, np.array(b.min[:], F), np.array(b.max[:], F)))
            else:
                r = d.rects[p.index]
                d1 = 1 if p.type == rt._ffi.PRIM_RECT_YZ else 0
                d2 = 1 if p.type == rt._ffi.PRIM_RECT_XY else 2
                self.rects.append((i, p.type, d1, d2, 3 - d1 - d2, (F(r.d1_min), F(r.d1_max), F(r.d2_min), F(r.d2_max)), F(r.offset)))
        # scene_create: the largest |coordinate| of a primitive box (rects are 2e-4 thick), boxes grown by 4e-6 x that
        m = F(0)
        for _, c, r in self.spheres:
            m = max(m, np.abs(c - r).max(), np.abs(c + r).max())
        for _, _, d1, d2, dn, bd, off in self.rects:
            m = max(m, np.abs(np.array(bd, F)).max(), abs(off - F(0.0001)), abs(off + F(0.0001)))
        for _, lo, hi in self.boxes:
            m = max(m, np.abs(lo).max(), np.abs(hi).max())
        self.max_abs = F(m)
        self.pad = F(self.max_abs * F(4e-6))
        self.max_r = max([float(r) for _, _, r in self.spheres] + [0.0])

    def targets(self, rng, n):
        """n points inside primitives (sphere cores, rect interiors, box interiors)."""
        out = []
        for _ in range(n):
            k = rng.integers(0, 3)
            if k == 0 and self.spheres:
                _, c, r = self.spheres[rng.integers(0, len(self.spheres))]
                out.append(c + rng.uniform(-0.5, 0.5, 3) * r)
            elif k == 1 and self.rects:
                _, _, d1, d2, dn, (a0, a1, b0, b1), off = self.rects[rng.integers(0, len(self.rects))]
                p = np.zeros(3)
                p[d1], p[d2], p[dn] = rng.uniform(a0, a1), rng.uniform(b0, b1), off
                out.append(p)
            elif self.boxes:
                _, lo, hi = self.boxes[rng.integers(0, len(self.boxes))]
                out.append(rng.uniform(lo, hi))
            else:
                _, c, r = self.spheres[rng.integers(0, len(self.spheres))] if self.spheres else (0, np.zeros(3), 1.0)
                out.append(c + rng.uniform(-0.5, 0.5, 3) * r)
        return np.array(out)


@pytest.fixture(scope="module")
def scenes(rt, gpu_required):
    """name -> (mirror handle, Prims, [(builder, device handle)]), built on first use."""
    cache = {}

    def get(name):
        if name not in cache:
            handles = []
            for builder in ("sah", "lbvh"):
                with pytest.MonkeyPatch.context() as mp:
                    mp.setenv("B200RT_BUILDER", builder)
                    s = SCENES[name](rt)
                    info = s.info()                                  # uploads: the tree is built now
                assert info.bvh_builder == (builder == "lbvh"), (name, builder)
                if name == "large":
                    assert info.bvh_nodes_in_smem == 0 and info.n_prims > 90_000, "the large scene is read through L1"
                else:
                    assert info.bvh_nodes_in_smem == info.n_bvh_nodes, f"{name} is staged in shared memory"
                if name == "ground":
                    assert info.n_bvh_nodes == info.n_prims - 2, "the ground is tested up front, outside the tree"
                handles.append((builder, s))
            cache[name] = (handles[0][1], Prims(rt, handles[0][1].desc), handles)
        return cache[name]
    return get


# ---- comparison -----------------------------------------------------------------------------------------------------------
def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _diff(ids, hits, want):
    """Indices of rays whose id, or (on a hit) t / p / n / front_face bits, differ."""
    bad = ids != want["id"]
    hit = (want["id"] >= 0) & ~bad
    for f in ("t", "p", "n"):
        g, w = _bits(hits[f]).reshape(len(ids), -1), _bits(want[f]).reshape(len(ids), -1)
        # a NaN coordinate (a NaN origin component) carries no payload worth comparing: NaN matches NaN
        nan = np.isnan(np.asarray(hits[f], F).reshape(len(ids), -1)) & np.isnan(np.asarray(want[f], F).reshape(len(ids), -1))
        bad |= hit & ((g != w) & ~nan).any(axis=1)
    bad |= hit & (hits["front_face"] != want["front_face"])
    return np.nonzero(bad)[0]


def _run(rt, po, handles, desc, rays, t_min, t_max, label, errors, want=None):
    """The device under every builder and slab mode against the mirror; mismatches go to `errors`.  Returns the mirror's hits."""
    rays = np.ascontiguousarray(rays, dtype=F)
    if want is None:
        want = po.closest_hit_gpu32(desc, rays, t_min, t_max)
    for builder, h in handles:
        for slab in ("auto", "exact"):
            with pytest.MonkeyPatch.context() as mp:
                if slab == "exact":
                    mp.setenv("B200RT_FAST_SLAB", "0")
                ids, hits, _ = rt.closest_hit(h, rays, t_min, t_max)
            bad = _diff(ids, hits, want)
            if len(bad):
                i = int(bad[0])
                errors.append(f"{label} [{builder}, {slab}]: {len(bad)}/{len(rays)} rays differ; first: ray {rays[i].tolist()} "
                              f"t in [{t_min}, {t_max}]: id {ids[i]} t {hits['t'][i]!r} vs mirror id {want['id'][i]} t {want['t'][i]!r}")
    return want


def _rays(o, d):
    return np.concatenate([np.asarray(o, np.float64).reshape(-1, 3), np.asarray(d, np.float64).reshape(-1, 3)], axis=1).astype(F)


def _aimed(rng, P, n, spread):
    """Rays from random origins around the scene towards points inside primitives, unit directions."""
    tgt = P.targets(rng, n)
    o = tgt + rng.normal(size=(n, 3)) * spread
    d = tgt - o
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return o, d, tgt


def _spread(name):
    return {"weekend": 6.0, "large": 40.0, "ground": 4.0}.get(name, 3.0)


def _n(name, n):
    return max(n // 20, 16) if name == "large" else n       # the mirror costs rays x primitives


# ---- ray families ---------------------------------------------------------------------------------------------------------
def _family_degenerate(rng, P, name):
    """Zero (+-0.0), subnormal (1e-40, 1e-45) and below-the-clamp (1e-20) direction components, mixed with ordinary ones;
    short directions (|d| = 1e-15 .. 1e-25: t reaches 1e15 .. 1e25); the two-sphere ray that first showed the clamp culling."""
    n = _n(name, 512)
    o, d, tgt = _aimed(rng, P, n, _spread(name))
    out = []
    for label, vals in (("zero", [0.0, -0.0]), ("subnormal", [1e-40, -1e-40, 1e-45, -1e-45]), ("below-clamp", [1e-20, -1e-20])):
        for n_axes in (1, 2):
            oo, dd = o.copy(), d.copy()
            for i in range(n):
                for k in rng.choice(3, n_axes, replace=False):
                    oo[i, k] = tgt[i, k]                                  # the origin inside the target's slab on that axis
                    dd[i, k] = vals[rng.integers(0, len(vals))]
            out.append((f"{label} x{n_axes}", _rays(oo, dd), 0.001, INF))
    oo, dd = o.copy(), d.copy()
    for i in range(n):                                                     # axis-parallel through the target, others +-0
        k = rng.integers(0, 3)
        dd[i] = 0.0
        dd[i, k] = rng.choice([-1.0, 1.0])
        oo[i] = tgt[i] - dd[i] * rng.uniform(0.5, 3.0) * _spread(name)
        dd[i, (k + 1) % 3] = rng.choice([0.0, -0.0])
    out.append(("axis-parallel", _rays(oo, dd), 0.001, INF))
    for s in (1e-15, 1e-20, 1e-25):
        out.append((f"short |d|={s:g} axis-parallel", _rays(oo, dd * s), 0.001, INF))
        out.append((f"short |d|={s:g} oblique", _rays(o, d * s), 0.001, INF))
    if name == "two_spheres":
        out.append(("pinned short ray", _rays([[0.999, 0, 0], [0.999, 0, 0], [0.5, 0, 0.5]], [[0, 1e-15, 0], [0, -1e-20, 0], [0, 1e-13, 0]]),
                    0.001, INF))
    return out


def _touch_points(P, rng, n_max):
    """(point, outward normal axis k, sign, in-plane axes) where a primitive touches its box: sphere poles, rect corners and edge
    midpoints, RectBox corners and edge midpoints."""
    pts = []
    for _, c, r in P.spheres[:n_max]:
        for k in range(3):
            for s in (-1.0, 1.0):
                p = c.astype(np.float64).copy(); p[k] += s * float(r)
                pts.append((p, k, s))
    for _, _, d1, d2, dn, (a0, a1, b0, b1), off in P.rects[:n_max]:
        for u in (a0, 0.5 * (a0 + a1), a1):
            for v in (b0, 0.5 * (b0 + b1), b1):
                if u == 0.5 * (a0 + a1) and v == 0.5 * (b0 + b1):
                    continue
                p = np.zeros(3); p[d1], p[d2], p[dn] = u, v, off
                pts.append((p, dn, 1.0))
    for _, lo, hi in P.boxes[:n_max]:
        for mask in range(27):
            sel = [(mask // 3 ** k) % 3 for k in range(3)]
            if sel.count(1) > 1:                                        # corners (no 1) and edge midpoints (one 1)
                continue
            p = np.array([(lo[k], 0.5 * (float(lo[k]) + float(hi[k])), hi[k])[sel[k]] for k in range(3)], np.float64)
            k = [j for j in range(3) if sel[j] != 1][0]
            pts.append((p, k, 1.0 if sel[k] == 2 else -1.0))
    if len(pts) > 400:
        pts = [pts[i] for i in rng.choice(len(pts), 400, replace=False)]
    return pts


def _family_tangent(rng, P, name):
    """Rays at the points where each primitive touches its box, parallel to the face there and oblique; origins exactly on a
    face, inside a primitive and inside the padding band (between the primitive's face and the padded box face)."""
    pts = _touch_points(P, rng, 8 if name in ("weekend", "large") else 100)
    o_par, d_par, o_obl, d_obl, o_on, d_on, o_pad, d_pad = ([] for _ in range(8))
    L = 2.0 * _spread(name)
    for p, k, s in pts:
        e = np.eye(3)
        for j in range(3):
            if j == k:
                continue
            for sg in (-1.0, 1.0):
                o_par.append(p - sg * L * e[j]); d_par.append(sg * e[j])                 # along the face through the point
                dv = sg * e[j] - s * e[k]                                                  # oblique onto the point from outside
                dv /= np.linalg.norm(dv)
                o_obl.append(p - L * dv); d_obl.append(dv)
        q = p.copy()                                                                      # on the face / in the padding band
        for dv in (-s * e[k], s * e[k], e[(k + 1) % 3], (e[(k + 1) % 3] - s * e[k]) / math.sqrt(2)):
            o_on.append(q); d_on.append(dv)
            qp = q.copy(); qp[k] += s * 0.5 * float(P.pad)
            o_pad.append(qp); d_pad.append(dv)
    inside_o, inside_d = [], []
    for _, c, r in P.spheres[:50]:
        for dv in np.eye(3).tolist() + [[0.6, 0.0, -0.8]]:
            inside_o.append(c); inside_d.append(dv)
    for _, lo, hi in P.boxes[:50]:
        for dv in np.eye(3).tolist() + [[0.6, 0.0, -0.8]]:
            inside_o.append(0.5 * (lo.astype(np.float64) + hi)); inside_d.append(dv)
    out = [("parallel to the face", _rays(o_par, d_par), 0.001, INF), ("oblique onto the touch point", _rays(o_obl, d_obl), 0.001, INF),
           ("origin on the face", _rays(o_on, d_on), 0.001, INF), ("origin on the face, t_min 0", _rays(o_on, d_on), 0.0, INF),
           ("origin in the padding band", _rays(o_pad, d_pad), 0.001, INF)]
    if inside_o:
        out.append(("origin inside a primitive", _rays(inside_o, inside_d), 0.001, INF))
    return out


def _family_origin_switch(rng, P, name):
    """A batch whose largest |origin coordinate| sits one f32 step either side of where the fast slab test is switched off
    (box_pad >= 4 eps max(max_abs, max_origin)), so that both kernels run; one far origin inside a near batch; a batch
    whose shortest direction sits either side of the direction limit."""
    n = _n(name, 256)
    o, d, tgt = _aimed(rng, P, n, _spread(name))
    four_eps = F(4.0) * F(EPS)
    lim = F(P.pad / four_eps)
    while F(four_eps * lim) > P.pad:
        lim = np.nextafter(lim, F(0))
    while F(four_eps * np.nextafter(lim, F(INF))) <= P.pad:
        lim = np.nextafter(lim, F(INF))
    out = []
    for label, ox in (("below", lim), ("above", np.nextafter(lim, F(INF)))):
        if ox <= P.max_abs:
            continue
        oo, dd = o.copy(), d.copy()
        oo[0] = [float(ox), 0.3, -0.2]
        dv = tgt[0] - oo[0]; dd[0] = dv / np.linalg.norm(dv)
        out.append((f"max origin {label} the limit {float(lim)!r}", _rays(oo, dd), 0.001, INF))
    oo = o.copy(); oo[n // 2] += 3.0e5
    out.append(("one far origin", _rays(oo, d), 0.001, INF))
    M = max(float(P.max_abs), float(np.abs(_rays(o, d)[:, :3]).max()))
    dlim = 4.0 * (float(P.max_abs) + M) / (float(P.pad) * 1e18)
    for label, s in (("below", 0.5), ("at", 1.0 + 1e-6), ("above", 2.0)):
        dd = d.copy(); dd[0] = dd[0] / np.abs(dd[0]).max() * dlim * s
        out.append((f"shortest direction {label} the limit {dlim:.3g}", _rays(o, dd), 0.001, INF))
    return out


FAMILIES = {"degenerate": _family_degenerate, "tangent": _family_tangent, "origin_switch": _family_origin_switch}
SCENES_ORDER = {k: i for i, k in enumerate(SCENES)}
FAMILY_ORDER = {k: i for i, k in enumerate(FAMILIES)}


@pytest.mark.parametrize("family", list(FAMILIES))
@pytest.mark.parametrize("name", list(SCENES))
def test_adversarial_rays_match_the_mirror(rt, po, scenes, name, family):
    mirror, P, handles = scenes(name)
    rng = np.random.default_rng([SCENES_ORDER[name], FAMILY_ORDER[family]])
    errors = []
    for label, rays, t_min, t_max in FAMILIES[family](rng, P, name):
        _run(rt, po, handles, mirror.desc, rays, t_min, t_max, f"{name}/{family}/{label}", errors)
    assert not errors, "\n".join(errors)


# ---- power-of-two scale invariance ----------------------------------------------------------------------------------------
K_SCALES = (-60, -50, -40, -20, -1, 0, 1, 20, 40, 60)


def _scale_exact(P, rays, k):
    """Rays for which every f32 step of the sphere test scales exactly by 2^k: delta * a (the discriminant, 4^k times the
    unscaled one) is 0 or a normal float.  Rect and box tests scale exactly for the directions used here."""
    o, d = rays[:, :3].astype(np.float64), rays[:, 3:].astype(np.float64)
    ok = np.ones(len(rays), bool)
    for lo in range(0, len(P.spheres), 4096):
        sph = P.spheres[lo:lo + 4096]
        c = np.array([s[1] for s in sph], np.float64); r = np.array([s[2] for s in sph], np.float64)
        oc = o[:, None, :] - c[None]
        b = (oc * d[:, None, :]).sum(-1)
        l2 = (oc * oc).sum(-1) - b * b
        delta = r[None] ** 2 - l2
        disc = np.abs(delta) * 4.0 ** k
        ok &= ~(((disc < 2.0 ** -125) | (disc > 2.0 ** 126) | (np.abs(delta) < 1e-5 * r[None] ** 2)) & (delta > -1e-5 * r[None] ** 2)).any(axis=1)
    return ok


@pytest.mark.parametrize("name", list(SCENES))
def test_power_of_two_scaled_directions(rt, po, scenes, name):
    """d -> 2^k d with t_min, t_max -> 2^-k t_min, t_max: a = d.d scales by 4^k, q, t and 1/d by 2^-k, q * d and fma(t, d, o)
    not at all, so ids, p, n and front_face are bit-identical to k = 0 and t is exactly t0 2^-k — as long as every step
    stays a normal float: direction components are 0 or >= 1/8 (d_k^2 4^-60 >= 2^-126), and rays whose discriminant
    delta * a would leave the normal range (grazing rays at k < 0; radius^2 4^k > 2^120 at k > 0: Weekend's ground at k = 60)
    are left out of the comparison across k.  Every k is also compared with the mirror bit for bit, and at k = 0 the ids
    with the f64 oracle on decidable rays."""
    mirror, P, handles = scenes(name)
    rng = np.random.default_rng(100 + SCENES_ORDER[name])
    n = _n(name, 1024)
    o, d, tgt = _aimed(rng, P, n, _spread(name))
    d[: n // 4] = 0.0                                                      # axis-parallel: zero components, 1/d = inf
    ax = rng.integers(0, 3, n // 4)
    d[np.arange(n // 4), ax] = rng.choice([-1.0, 1.0], n // 4)
    o[: n // 4] = tgt[: n // 4] - d[: n // 4] * 2.0 * _spread(name)
    small = (np.abs(d) < 0.125) & (d != 0)
    d[small] = np.sign(d[small]) * 0.125
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d[(np.abs(d) < 0.125) & (d != 0)] = 0.0                                  # renormalising can push a component just below 1/8
    base = _rays(o, d)
    errors = []
    results = {}
    for k in K_SCALES:
        rays = base.copy()
        rays[:, 3:] *= F(2.0 ** k)
        t_min = float(F(0.001) * F(2.0 ** -k))
        _run(rt, po, handles, mirror.desc, rays, t_min, INF, f"{name}/scaled k={k}", errors)
        results[k] = (rays, rt.closest_hit(handles[0][1], rays, t_min, INF)[:2])
    assert not errors, "\n".join(errors)
    ids0, h0 = results[0][1]
    for k in K_SCALES:
        if P.max_r ** 2 * 4.0 ** k > 2.0 ** 120:
            continue                                                       # delta * a overflows for the largest sphere
        keep = _scale_exact(P, base, k) if P.spheres else np.ones(n, bool)
        assert keep.mean() > 0.5, (name, k, keep.mean())
        ids, h = results[k][1]
        assert np.array_equal(ids[keep], ids0[keep]), (name, k, int((ids[keep] != ids0[keep]).sum()))
        hit = keep & (ids0 >= 0)
        assert np.array_equal(h["t"][hit], h0["t"][hit] * F(2.0 ** -k)), (name, k)
        for f in ("p", "n"):
            assert np.array_equal(_bits(h[f][hit]), _bits(h0[f][hit])), (name, k, f)
        assert np.array_equal(h["front_face"][hit], h0["front_face"][hit]), (name, k)
    # unit scale: the ids agree with the f64 reference wherever f32 can decide the closest hit
    # (the oblique rays: an axis-parallel ray that starts in a rect's plane has t = 0 * inf = NaN, which the f64 reference's
    # rect test accepts and the device's rejects, and no margin flags that)
    o64 = po.OracleScene(mirror.desc, reference_topology=False)
    ids64, _, mg, _ = o64.closest_hit(base[n // 4:], 0.001, INF, margins=True)
    o64.close()
    # A zero-thickness RectBox is left out: the reference's unpadded box around it has zero width, where Aabb::hit2 never
    # passes, while the device tests the RectBox itself — a known difference from the reference, not checked here.
    flat = [i for i, lo, hi in P.boxes if (lo == hi).any()]
    keep = decidable(mg) & ~np.isin(ids0[n // 4:], flat) & ~np.isin(ids64, flat)
    assert keep.mean() > 0.8 and np.array_equal(ids0[n // 4:][keep], ids64[keep]), (name, keep.mean())


# ---- interval ends --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(SCENES))
def test_interval_ends(rt, po, scenes, name):
    """t_max and t_min equal to the mirror's hit t and one ulp to either side; t_min == t_max, t_min > t_max, t_min = 0,
    a negative t_min, t_max = 0."""
    mirror, P, handles = scenes(name)
    rng = np.random.default_rng(200 + SCENES_ORDER[name])
    o, d, _ = _aimed(rng, P, 256, _spread(name))
    rays = _rays(o, d)
    base = po.closest_hit_gpu32(mirror.desc, rays, 0.001, INF)
    errors = []
    sel = np.nonzero(base["id"] >= 0)[0][: (8 if name == "large" else 24)]
    assert len(sel) >= 8
    for i in sel:
        t = F(base["t"][i])
        for v in (np.nextafter(t, F(0)), t, np.nextafter(t, F(INF))):
            _run(rt, po, handles, mirror.desc, rays[i:i + 1], 0.001, float(v), f"{name}/t_max={float(v)!r}", errors)
            _run(rt, po, handles, mirror.desc, rays[i:i + 1], float(v), INF, f"{name}/t_min={float(v)!r}", errors)
    sub = rays[: _n(name, 256)]
    for t_min, t_max in ((1.0, 1.0), (2.0, 1.0), (0.0, INF), (-1.0, INF), (-INF, INF), (0.001, 0.0), (0.0, 0.0)):
        _run(rt, po, handles, mirror.desc, sub, t_min, t_max, f"{name}/[{t_min}, {t_max}]", errors)
    assert not errors, "\n".join(errors)


# ---- non-finite rays ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(SCENES))
def test_non_finite_rays_in_an_ordinary_batch(rt, po, scenes, name):
    """A few rays with NaN or inf components inside an ordinary batch: every comparison with NaN is false, so the traversal
    pops to its sentinel or leaves the axis unconstrained exactly as Aabb::hit2 does; the other rays' results do not change
    and the bad rays equal the mirror."""
    mirror, P, handles = scenes(name)
    rng = np.random.default_rng(300 + SCENES_ORDER[name])
    n = _n(name, 512)
    o, d, _ = _aimed(rng, P, n, _spread(name))
    good = _rays(o, d)
    nan, inf = float("nan"), float("inf")
    bad_rays = []
    for k in range(3):
        for v in (nan, inf, -inf):
            r = good[k].astype(np.float64).copy(); r[k] = v; bad_rays.append(r)               # origin component
            r = good[k + 3].astype(np.float64).copy(); r[3 + k] = v; bad_rays.append(r)       # direction component
    r = good[7].astype(np.float64).copy(); r[:] = nan; bad_rays.append(r)
    bad = np.array(bad_rays).astype(F)
    pos = np.sort(rng.choice(n + len(bad), len(bad), replace=False))
    mixed = np.empty((n + len(bad), 6), F)
    is_bad = np.zeros(n + len(bad), bool); is_bad[pos] = True
    mixed[is_bad], mixed[~is_bad] = bad, good
    errors = []
    want = _run(rt, po, handles, mirror.desc, mixed, 0.001, INF, f"{name}/non-finite", errors)
    _run(rt, po, handles, mirror.desc, good, 0.001, INF, f"{name}/finite part alone", errors, want=want[~is_bad])
    assert not errors, "\n".join(errors)


# ---- the Aabb::hit2 hook ---------------------------------------------------------------------------------------------------
def _aabb_hit2_f32(boxes, rays, t_min, t_max):
    """rt_device.cuh: aabb_hit2 in NumPy float32: (plane - o) * (1/d) rounded per step, the swap chosen by the sign of 1/d,
    fmaxf / fminf dropping a NaN operand (np.fmax / np.fmin), and `!(hi <= lo)`."""
    b, r = boxes.astype(F), rays.astype(F)
    with np.errstate(all="ignore"):
        inv = F(1) / r[:, 3:]
        a = (b[:, :3] - r[:, :3]) * inv
        c = (b[:, 3:] - r[:, :3]) * inv
    s = inv < 0
    t0, t1 = np.where(s, c, a), np.where(s, a, c)
    lo = np.fmax(np.fmax(t0[:, 0], t0[:, 1]), np.fmax(t0[:, 2], F(t_min)))
    hi = np.fmin(np.fmin(t1[:, 0], t1[:, 1]), np.fmin(t1[:, 2], F(t_max)))
    return ~(hi <= lo)


def test_aabb_hit_hook_bit_for_bit(rt, gpu_required):
    """The Aabb::hit2 hook (b200rt_aabb_hit) against a float32 restatement of its arithmetic on degenerate, tangent and
    interval-end rays, and on zero-thickness and inverted boxes."""
    rng = np.random.default_rng(400)
    n = 20_000
    lo = rng.uniform(-4, 4, (n, 3))
    ext = rng.choice([0.0, 1e-6, 0.5, 2.0], (n, 3))
    ext[: n // 10] *= -1                                                    # inverted boxes
    boxes = np.concatenate([lo, lo + ext], axis=1).astype(F)
    tgt = rng.uniform(boxes[:, :3], np.maximum(boxes[:, :3], boxes[:, 3:]))
    o = tgt + rng.normal(size=(n, 3)) * 3
    d = tgt - o
    fam = rng.integers(0, 6, n)
    k = rng.integers(0, 3, n)
    idx = np.arange(n)
    corner = np.where(rng.random((n, 3)) < 0.5, boxes[:, :3], boxes[:, 3:])
    # 0: ordinary  1: +-0 component, origin in the slab  2: subnormal / below-clamp component  3: origin on a face or a corner
    # 4: along a face (tangent)  5: short direction
    o[fam == 1, k[fam == 1]] = tgt[fam == 1, k[fam == 1]]
    d[fam == 1, k[fam == 1]] = rng.choice([0.0, -0.0], (fam == 1).sum())
    d[fam == 2, k[fam == 2]] = rng.choice([1e-40, -1e-45, 1e-20, -1e-20], (fam == 2).sum())
    o[fam == 3] = corner[fam == 3]
    o[fam == 4, k[fam == 4]] = corner[fam == 4, k[fam == 4]]
    d[fam == 4, k[fam == 4]] = 0.0
    d[fam == 5] *= 1e-15
    rays = _rays(o, d)
    for t_min, t_max in ((0.001, INF), (0.0, INF), (0.0, 0.0), (1.0, 1.0), (2.0, 1.0), (-INF, INF), (0.001, 3.4028235e38)):
        got = rt.aabb_hit(boxes, rays, t_min, t_max).astype(bool)
        want = _aabb_hit2_f32(boxes, rays, t_min, t_max)
        assert np.array_equal(got, want), (t_min, t_max, [(int(f), int((got != want)[fam == f].sum())) for f in range(6)])
    # interval ends: t_max / t_min at the entry and exit distances and one ulp either side
    with np.errstate(all="ignore"):
        inv = F(1) / rays[:, 3:]
        t_in = np.fmax(np.fmax(*[np.minimum((boxes[:, j] - rays[:, j]) * inv[:, j], (boxes[:, 3 + j] - rays[:, j]) * inv[:, j]) for j in (0, 1)]),
                       np.minimum((boxes[:, 2] - rays[:, 2]) * inv[:, 2], (boxes[:, 5] - rays[:, 2]) * inv[:, 2]))
    sel = np.nonzero(np.isfinite(t_in) & (t_in > 0) & (fam == 0))[0][:64]
    for i in sel:
        for v in (np.nextafter(t_in[i], F(0)), t_in[i], np.nextafter(t_in[i], F(INF))):
            for t_min, t_max in ((0.0, float(v)), (float(v), INF)):
                got = rt.aabb_hit(boxes[i:i + 1], rays[i:i + 1], t_min, t_max).astype(bool)
                assert got[0] == _aabb_hit2_f32(boxes[i:i + 1], rays[i:i + 1], t_min, t_max)[0], (i, t_min, t_max)
