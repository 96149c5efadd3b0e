"""Seeded procedural occluder sets and adversarial shadow rays for the occluder any-hit tests (list, BVH, oracle).

Every set is float32 [n, 9] (three vertices per triangle) in or around the unit box of the synthetic scene."""
import numpy as np

import gvpm_b200 as g


def walls():
    """The 12 triangles of the synthetic box's walls."""
    return g.synth_occluders().reshape(-1, 9)


def blocker_sheets(cells=1, e=2e-4):
    """Sheets e inside every wall of the unit box (tests/functor_pin_cases.py _blocker), each split into
    cells x cells squares of two triangles."""
    tris = []
    s = np.linspace(0.0, 1.0, cells + 1)
    a0, b0 = np.meshgrid(s[:-1], s[:-1], indexing="ij")
    a1, b1 = a0 + 1.0 / cells, b0 + 1.0 / cells
    a1 = np.where(np.isclose(a1, 1.0), 1.0, a1)
    b1 = np.where(np.isclose(b1, 1.0), 1.0, b1)
    for axis in range(3):
        for side in (e, 1.0 - e):
            u, v = [k for k in range(3) if k != axis]

            def pt(a, b):
                q = np.zeros(a.shape + (3,))
                q[..., axis], q[..., u], q[..., v] = side, a, b
                return q
            p00, p10, p11, p01 = pt(a0, b0), pt(a1, b0), pt(a1, b1), pt(a0, b1)
            tris.append(np.concatenate([p00, p10, p11], axis=-1).reshape(-1, 9))
            tris.append(np.concatenate([p00, p11, p01], axis=-1).reshape(-1, 9))
    return np.concatenate(tris).astype(np.float32)


def uv_sphere(nu=128, nv=80, centre=(0.5, 0.5, 0.5), r=0.25):
    """A UV sphere of 2 * nu * (nv - 1) triangles (the pole rows are fans; their degenerate halves are kept)."""
    th = np.linspace(0.0, np.pi, nv + 1)
    ph = np.linspace(0.0, 2 * np.pi, nu + 1)
    T, P = np.meshgrid(th, ph, indexing="ij")
    V = np.stack([np.sin(T) * np.cos(P), np.sin(T) * np.sin(P), np.cos(T)], axis=-1) * r + np.asarray(centre)
    p00, p10, p11, p01 = V[:-1, :-1], V[1:, :-1], V[1:, 1:], V[:-1, 1:]
    t = np.concatenate([np.concatenate([p00, p10, p11], axis=-1).reshape(-1, 9),
                        np.concatenate([p00, p11, p01], axis=-1).reshape(-1, 9)])
    return t.astype(np.float32)


def soup(n=100000, seed=7, size=0.01, shift=0.0):
    """n small random triangles in the unit box; 2 % zero-area (a repeated vertex or a point), 2 % collinear, 2 %
    duplicates of other triangles."""
    rng = np.random.default_rng(seed)
    c = rng.uniform(0.0, 1.0, (n, 1, 3))
    t = c + rng.normal(0.0, size, (n, 3, 3))
    k = n // 50
    idx = rng.permutation(n)
    z, col, dup = idx[:k], idx[k:2 * k], idx[2 * k:3 * k]
    t[z[: k // 2], 2] = t[z[: k // 2], 0]                        # two equal vertices
    t[z[k // 2:], 1] = t[z[k // 2:], 0]; t[z[k // 2:], 2] = t[z[k // 2:], 0]   # a point
    w = rng.uniform(-1.0, 2.0, (k, 1))
    t[col, 2] = t[col, 0] + w * (t[col, 1] - t[col, 0])          # collinear
    t[dup] = t[rng.integers(0, n, k)]
    return (t.reshape(n, 9) + shift).astype(np.float32)


def height_field(m=708, seed=3):
    """A height field over [0, 1]^2 of 2 * (m - 1)^2 triangles (~1 M for m = 708)."""
    rng = np.random.default_rng(seed)
    s = np.linspace(0.0, 1.0, m)
    X, Y = np.meshgrid(s, s, indexing="ij")
    Z = 0.5 + 0.05 * np.sin(9 * X) * np.cos(7 * Y) + rng.normal(0.0, 1e-3, X.shape)
    V = np.stack([X, Y, Z], axis=-1)
    p00, p10, p11, p01 = V[:-1, :-1], V[1:, :-1], V[1:, 1:], V[:-1, 1:]
    t = np.concatenate([np.concatenate([p00, p10, p11], axis=-1).reshape(-1, 9),
                        np.concatenate([p00, p11, p01], axis=-1).reshape(-1, 9)])
    return t.astype(np.float32)


def _unit(v):
    v = np.asarray(v, dtype=np.float64)
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def adversarial_rays(tri, n=20000, seed=11, eps=1e-4):
    """Shadow rays (o, d, mint, maxt) that probe the rounding of the strict test: origins on triangles (reconnection
    parents on walls), rays aimed at shared vertices and at edges, grazing rays within 1e-7 rad of a triangle's plane,
    maxt at the double-precision distance of the aimed-at point and its float neighbours, maxt < mint, very short and
    full-length segments."""
    rng = np.random.default_rng(seed)
    T = np.asarray(tri, dtype=np.float64).reshape(-1, 3, 3)
    nt = T.shape[0]
    k = n // 8

    def on_tri(m):
        i = rng.integers(0, nt, m)
        a, b = rng.uniform(0, 1, (2, m, 1))
        flip = (a + b) > 1
        a, b = np.where(flip, 1 - a, a), np.where(flip, 1 - b, b)
        return T[i, 0] + a * (T[i, 1] - T[i, 0]) + b * (T[i, 2] - T[i, 0]), i

    O, D, MINT, MAXT = [], [], [], []

    def add(o, d, mint, maxt):
        O.append(o); D.append(_unit(d)); MINT.append(np.broadcast_to(mint, (len(o),))); MAXT.append(maxt)

    # 1. origins on triangles, random directions, full-length and very short segments
    o, _ = on_tri(k)
    add(o, rng.normal(size=(k, 3)), eps, rng.choice([10.0, 1.0, 1e-3, 1e-6], k))
    # 2. aimed at vertices (shared by neighbouring triangles) from points on other triangles
    o, _ = on_tri(k)
    tgt = T[rng.integers(0, nt, k), rng.integers(0, 3, k)]
    dist = np.linalg.norm(tgt - o, axis=1)
    ok = dist > 1e-6
    add(o[ok], tgt[ok] - o[ok], eps, dist[ok] * rng.choice([0.5, 1.0, 2.0], ok.sum()))
    # 3. aimed at edge points
    o, _ = on_tri(k)
    i = rng.integers(0, nt, k)
    s = rng.uniform(0, 1, (k, 1))
    tgt = T[i, 0] + s * (T[i, 1] - T[i, 0])
    dist = np.linalg.norm(tgt - o, axis=1)
    ok = dist > 1e-6
    add(o[ok], tgt[ok] - o[ok], eps, dist[ok] * rng.choice([0.999, 1.0, 1.001], ok.sum()))
    # 4. maxt at the double distance of an interior point and at its float neighbours
    o = rng.uniform(-0.2, 1.2, (k, 3))
    tgt, _ = on_tri(k)
    d = _unit(tgt - o)
    dist = np.linalg.norm(tgt - o, axis=1).astype(np.float32)
    which = rng.integers(0, 3, k)
    maxt = np.where(which == 0, dist, np.where(which == 1, np.nextafter(dist, np.float32(np.inf)),
                                                 np.nextafter(dist, np.float32(0))))
    add(o, d, 0.0, maxt.astype(np.float64))
    # 5. grazing: from a point on (or 1e-6 off) a triangle's plane, along the plane tilted by < 1e-7 rad
    o, i = on_tri(k)
    nrm = np.cross(T[i, 1] - T[i, 0], T[i, 2] - T[i, 0])
    good = np.linalg.norm(nrm, axis=1) > 0
    o, i, nrm = o[good], i[good], _unit(nrm[good])
    m = len(o)
    inplane = _unit(np.cross(nrm, rng.normal(size=(m, 3))))
    ang = rng.uniform(-1e-7, 1e-7, (m, 1))
    off = rng.choice([0.0, 1e-6, -1e-6], (m, 1))
    add(o + off * nrm - inplane * rng.uniform(0, 0.05, (m, 1)), inplane + ang * nrm, eps,
        rng.choice([1e-2, 0.1, 1.0], m))
    # 6. grazing rays started away from the set, through it
    o = rng.uniform(0, 1, (k, 3))
    tgt, i = on_tri(k)
    nrm = np.cross(T[i, 1] - T[i, 0], T[i, 2] - T[i, 0])
    good = np.linalg.norm(nrm, axis=1) > 0
    nrm = np.where(good[:, None], nrm, 1.0)
    nrm = _unit(nrm)
    inplane = _unit(np.cross(nrm, rng.normal(size=(k, 3))))
    add(tgt - 0.3 * inplane, inplane + rng.uniform(-1e-7, 1e-7, (k, 1)) * nrm, eps, rng.choice([0.3, 0.6], k))
    # 7. maxt < mint, and maxt == mint
    o, _ = on_tri(k)
    mx = rng.choice([0.5 * eps, eps], k)
    add(o, rng.normal(size=(k, 3)), eps, mx)
    # 8. reconnection-like: parent on a triangle, short segment of 0.1 % of a connection
    o, _ = on_tri(k)
    add(o, rng.normal(size=(k, 3)), eps, rng.uniform(0, 1, k) * 1e-3)
    o = np.concatenate(O).astype(np.float32)
    d = np.concatenate(D).astype(np.float32)
    return (o, d, np.concatenate(MINT).astype(np.float32), np.concatenate(MAXT).astype(np.float32))


def oracle_any_hit_by_triangle(tri, o, d, mint, maxt):
    """OR over the triangles of gvpm_oracle_pin_triangle (one triangle per query): the definition any-hit restates."""
    import ctypes as C
    from oracle import binding as ob
    lib = ob.load()
    fn = lib.gvpm_oracle_pin_triangle
    f32p = C.POINTER(C.c_float)
    fn.argtypes = [f32p, f32p, f32p, f32p, f32p, C.c_size_t, C.POINTER(C.c_uint8)]
    fn.restype = None
    tri = np.asarray(tri, dtype=np.float32).reshape(-1, 9)
    m = len(o)
    hit = np.zeros(m, dtype=bool)
    for t in tri:
        tt = np.ascontiguousarray(np.broadcast_to(t, (m, 9)))
        h = np.zeros(m, dtype=np.uint8)
        fn(tt.ctypes.data_as(f32p), np.ascontiguousarray(o).ctypes.data_as(f32p),
           np.ascontiguousarray(d).ctypes.data_as(f32p), np.ascontiguousarray(mint).ctypes.data_as(f32p),
           np.ascontiguousarray(maxt).ctypes.data_as(f32p), m, h.ctypes.data_as(C.POINTER(C.c_uint8)))
        hit |= h.astype(bool)
    return hit
