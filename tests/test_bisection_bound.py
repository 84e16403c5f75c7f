"""The distance bound that lets pool_eval (csrc/cq_pool.cuh) apply refineTOI bisection steps without evaluating them,
restated in numpy and checked against the oracle's segment_triangle_distance (the function the reference and the kernels
evaluate, bit for bit: tests/test_device_math_on_host.py).  Each sweep runs sweepCapsuleTriangle's conservative advancement
(CollisionQuery.swift:1303-1356) to its first contact and then refineTOI's ten bisection steps (:1361-1394), EVERY midpoint
evaluated; alongside, the anchor of the kernel (the last evaluation it really makes: the contact that entered refineTOI,
then each midpoint the bound could not decide) predicts every step.  A prediction must never disagree with the
evaluation (DESIGN.md §5.1, "Decided bisection steps"), and the bound must decide a good share of the steps.  CPU only:
this pins the ARGUMENT; that the kernels implement it is what the GPU parity tests check (byte-equal to the oracle)."""
import numpy as np
import pytest

f32 = np.float32
MARGIN_REL = f32(1.9073486e-6)  # 16 * 2^-23, cq_pool.cuh bisect_margin


def bisect_margin(frm, L, hh, r):
    scale = np.abs(frm[:, 0]) + np.abs(frm[:, 1]) + np.abs(frm[:, 2]) + L + hh + r
    return np.where((r > f32(5e-3)) & (hh <= f32(16.0) * r), scale * MARGIN_REL, f32(np.inf)).astype(f32)


def decided(mid, tc, d, r, margin):
    """pool_eval's rule: |mid - tc| + margin < |d - r| (false for a NaN d)"""
    with np.errstate(invalid="ignore"):
        return np.abs(mid - tc) + margin < np.abs(d - r)


def refine_with_predictions(orc, frm, delta, r, hh, tris):
    """sweepCapsuleTriangle + refineTOI per row, every step evaluated.  Returns (bisection steps, decided, wrong, fin reuse)."""
    n = len(frm)
    L = np.sqrt(delta[:, 0] * delta[:, 0] + delta[:, 1] * delta[:, 1] + delta[:, 2] * delta[:, 2]).astype(f32)
    d_ = (delta / L[:, None]).astype(f32)
    minAdv = np.maximum(r * f32(0.02), f32(1e-4)).astype(f32)
    maxIter = np.minimum(256, np.ceil(L / minAdv).astype(np.int64) + 1)
    margin = bisect_margin(frm, L, hh, r)

    def dist_at(idx, t):
        c = (frm[idx] + d_[idx] * t[:, None]).astype(f32)
        return orc.segment_triangle_distance_batch(c, hh[idx], tris[idx])[0]

    t, last = np.zeros(n, f32), np.zeros(n, f32)
    live = L >= f32(1e-6)
    hit = np.zeros(n, bool)
    tc, dc = np.zeros(n, f32), np.zeros(n, f32)
    for it in range(256):
        live &= (it < maxIter) & ~(t > L)
        idx = np.nonzero(live)[0]
        if len(idx) == 0:
            break
        dist = dist_at(idx, t[idx])
        c = dist <= r[idx] + f32(1e-5)
        hi_, ad = idx[c], idx[~c]
        hit[hi_], tc[hi_], dc[hi_] = True, t[hi_], dist[c]
        live[hi_] = False
        last[ad] = t[ad]
        adv = np.maximum(dist[~c] - r[ad], minAdv[ad]).astype(f32)
        t[ad] = (t[ad] + np.where(adv <= 0, minAdv[ad], adv)).astype(f32)
    idx = np.nonzero(hit)[0]
    c0 = np.maximum(f32(0), np.minimum(last[idx], L[idx]))
    c1 = np.maximum(f32(0), np.minimum(t[idx], L[idx]))
    lo, hi = np.minimum(c0, c1), np.maximum(c0, c1)
    fin_reuse = int(((hi - lo < f32(1e-5)) & (hi.view(np.uint32) == tc[idx].view(np.uint32))).sum())
    bis = hi - lo >= f32(1e-5)
    idx, lo, hi = idx[bis], lo[bis], hi[bis]
    atc, ad = tc[idx].copy(), dc[idx].copy()  # the anchor: this trip's evaluation
    steps = decided_n = wrong = 0
    for k in range(10):
        mid = (f32(0.5) * (lo + hi)).astype(f32)
        dm = dist_at(idx, mid)
        pred = decided(mid, atc, ad, r[idx], margin[idx])
        contact = dm <= r[idx]
        wrong += int((pred & (contact != (ad <= r[idx]))).sum())
        steps += len(idx)
        decided_n += int(pred.sum())
        hi = np.where(contact, mid, hi)
        lo = np.where(contact, lo, mid)
        atc = np.where(pred, atc, mid)  # an undecided step is evaluated: it becomes the anchor
        ad = np.where(pred, ad, dm)
    fin_reuse += int((hi.view(np.uint32) == atc.view(np.uint32)).sum())
    return steps, decided_n, wrong, fin_reuse


def world_triangles(parts):
    out = []
    for p in parts:
        m = np.asarray(p["model"], np.float64).reshape(4, 4).T
        w = p["positions"].astype(np.float64) @ m[:3, :3].T + m[:3, 3]
        out.append(w[p["indices"].reshape(-1, 3)])
    return np.concatenate(out).astype(f32)


def sweeps_near(rng, tris, n, radius, hh, offset=0.0, grazing=0.3, start_at_r=0.1):
    """Sweeps aimed at points of the triangles (interior, edges and vertices: Voronoi-region boundaries), from random,
    grazing (nearly in the triangle's plane) and horizontal directions; some start in contact or at exactly r."""
    k = rng.integers(0, len(tris), n)
    T = tris[k].astype(np.float64)
    w = rng.dirichlet((1, 1, 1), n)
    on_edge = np.nonzero(rng.random(n) < 0.2)[0]
    w[on_edge, rng.integers(0, 3, len(on_edge))] = 0.0  # on an edge
    w[rng.random(n) < 0.1] = np.eye(3)[rng.integers(0, 3)]  # at a vertex
    w /= w.sum(1, keepdims=True)
    target = (T * w[:, :, None]).sum(1)
    nrm = np.cross(T[:, 1] - T[:, 0], T[:, 2] - T[:, 0])
    nrm /= np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-30)
    g = rng.standard_normal((n, 3))
    graze = rng.random(n) < grazing
    g[graze] -= (g[graze] * nrm[graze]).sum(1, keepdims=True) * nrm[graze] * (1 - rng.uniform(0, 1e-3, (graze.sum(), 1)))
    horiz = rng.random(n) < 0.3
    g[horiz, 1] = 0.0
    d = g / np.linalg.norm(g, axis=1, keepdims=True)
    r = np.broadcast_to(np.asarray(radius, np.float64), (n,)).copy()
    h = np.broadcast_to(np.asarray(hh, np.float64), (n,)).copy()
    L = rng.uniform(0.05, 6.0, n)
    back = rng.uniform(0.0, 1.0, n) * L
    standoff = (r + h) * rng.uniform(0.0, 1.5, n)
    frm = target + nrm * standoff[:, None] - d * back[:, None]
    at_r = rng.random(n) < start_at_r  # axis starting (about) r from the triangle's plane, or inside
    frm[at_r] = target[at_r] + nrm[at_r] * (r[at_r] * rng.choice([0.5, 1.0 - 1e-6, 1.0, 1.0 + 1e-6], at_r.sum()))[:, None]
    off = rng.uniform(-offset, offset, (n, 3))
    tr = (T + off[:, None, :]).astype(f32)
    return (frm + off).astype(f32), (d * L[:, None]).astype(f32), r.astype(f32), h.astype(f32), tr.reshape(n, 9)


def run(orc, frm, delta, r, hh, tris):
    return refine_with_predictions(orc, frm, delta, r, hh, np.ascontiguousarray(tris, f32).reshape(-1, 9))


@pytest.fixture(scope="module")
def scene_tris(scenes):
    hulls = world_triangles(scenes.mirror_scene(use_hulls=True))
    semla = world_triangles(scenes.semla_scene(use_hulls=False))
    parts, _ = scenes.terrain_scene(cells=64)
    terrain = world_triangles(parts)
    return {"hulls": hulls, "semla": semla, "terrain": terrain}


@pytest.mark.parametrize("scene,radius,hh,offset,seed,floor", [
    ("hulls", 1.5, 1.0, 0.0, 100, 0.15),      # C3 characters (measured: 21% of the steps decided)
    ("hulls", 0.4, 0.5, 0.0, 101, 0.10),      # (16%)
    ("semla", 1.5, 1.0, 0.0, 102, 0.15),      # C2 sweeps (21%)
    ("terrain", 0.4, 0.5, 0.0, 103, 0.07),    # C4 walkers (11%)
    ("terrain", 0.4, 0.5, 2236.0, 104, 0.002),  # the same cells anywhere on the 10 M-triangle terrain, +-2,236 m (0.4%)
])
def test_decided_bisection_steps_agree_with_the_evaluation(orc, scene_tris, scene, radius, hh, offset, seed, floor):
    rng = np.random.default_rng(seed)
    steps, dec, wrong, reuse = run(orc, *sweeps_near(rng, scene_tris[scene], 30000, radius, hh, offset))
    assert steps > 20000
    assert wrong == 0, (scene, wrong, steps)
    assert dec >= floor * steps, (scene, dec / steps)
    assert reuse > 0


def test_adversarial_sweeps(orc):
    """Random triangles at every scale (degenerate edges, nearly vertical triangles whose piercing test fails, nearly
    vertical edges), random radii and half heights (including the ones the rule refuses), offsets up to +-2,236 m."""
    rng = np.random.default_rng(77)
    n = 60000
    scale = 10.0 ** rng.uniform(-3, 1.5, (n, 1, 1))
    T = rng.standard_normal((n, 3, 3)) * scale
    deg = rng.random(n) < 0.1
    T[deg, 1] = T[deg, 0] + rng.standard_normal((deg.sum(), 3)) * 1e-5
    vert = rng.random(n) < 0.15  # (nearly) vertical triangles: the axis (nearly) in their plane
    T[vert, :, 2] = T[vert, 0:1, 2] + rng.standard_normal((vert.sum(), 3)) * 1e-7 * scale[vert, :, 0]
    edge = rng.random(n) < 0.15  # a (nearly) vertical edge
    tilt = 10.0 ** rng.uniform(-7, -3, edge.sum()) * np.abs(T[edge, 1, 1] - T[edge, 0, 1])
    for ax in (0, 2):
        T[edge, 1, ax] = T[edge, 0, ax] + rng.standard_normal(edge.sum()) * tilt
    tris = T.astype(f32)
    radius = (10.0 ** rng.uniform(-3, 0.5, n)).astype(f32)
    hh = np.where(rng.random(n) < 0.1, 0.0, 10.0 ** rng.uniform(-3, 0.5, n)).astype(f32)
    total = [0, 0, 0]
    for off in (0.0, 50.0, 2236.0):
        frm, delta, r, h, tr = sweeps_near(rng, tris, n, radius, hh, off, grazing=0.5, start_at_r=0.2)
        steps, dec, wrong, _ = run(orc, frm, delta, r, h, tr)
        assert wrong == 0, (off, wrong, steps)
        total = [total[0] + steps, total[1] + dec, total[2] + wrong]
    assert total[1] >= 0.02 * total[0], total  # (measured: 5.3%; many of these capsules are refused)


def test_nan_and_refused_capsules_never_decide():
    mid, tc = np.array([0.5, 0.5], f32), np.array([0.25, 0.25], f32)
    assert not decided(mid, tc, np.array([np.nan, np.nan], f32), f32(0.4), f32(0.0)).any()
    frm = np.zeros((3, 3), f32)
    m = bisect_margin(frm, np.ones(3, f32), np.array([0.5, 0.5, 1.0], f32), np.array([0.4, 0.004, 0.05], f32))
    assert np.isfinite(m[0]) and np.isinf(m[1]) and np.isinf(m[2])
