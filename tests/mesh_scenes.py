"""Mesh scenes of the mesh-generator tests (TEST INFRASTRUCTURE): the triangulated Cornell box, a tessellated sphere
over a height field, a random triangle soup.  Each -> mesh_trace_ref.Scene (the arrays of Context.set_trace_mesh)."""
import numpy as np

import gvpm_b200 as g
import mesh_trace_ref as MR


def cornell():
    return MR.Scene(**g.box_scene_as_mesh(g.box_scene_default()))


def _light(y=0.999, x0=0.35, x1=0.65, z0=0.35, z1=0.65):
    # two triangles whose winding normal points down
    return [((x0, y, z0), (x1, y, z0), (x1, y, z1)), ((x0, y, z0), (x1, y, z1), (x0, y, z1))]


def _walls():
    m = g.box_scene_as_mesh(g.box_scene_default())
    keep = m["emissive"] == 0
    return list(m["tri"][keep].reshape(-1, 3, 3)), list(m["albedo"][keep])


def height_field(res):
    """res x res quads of y = 0.08 + 0.05 sin(..) cos(..) over the floor, two triangles each"""
    xs = np.linspace(0.02, 0.98, res + 1)
    X, Z = np.meshgrid(xs, xs, indexing="ij")
    Y = 0.08 + 0.05 * np.sin(7.0 * X) * np.cos(5.0 * Z)
    P = np.stack([X, Y, Z], -1)
    a, b, c, d = P[:-1, :-1], P[1:, :-1], P[1:, 1:], P[:-1, 1:]
    tris = np.stack([np.stack([a, b, c], -2), np.stack([a, c, d], -2)], 2)   # [res, res, 2, 3, 3]
    return tris.reshape(-1, 3, 3).astype(np.float32)


def sphere(centre, r, nu, nv):
    tris = []
    for i in range(nu):
        for j in range(nv):
            t0, t1 = np.pi * i / nu, np.pi * (i + 1) / nu
            p0, p1 = 2 * np.pi * j / nv, 2 * np.pi * (j + 1) / nv

            def pt(t, p):
                return np.array(centre) + r * np.array([np.sin(t) * np.cos(p), np.cos(t), np.sin(t) * np.sin(p)])
            a, b, c, d = pt(t0, p0), pt(t1, p0), pt(t1, p1), pt(t0, p1)
            if i > 0:
                tris.append((a, b, d))
            if i < nu - 1:
                tris.append((b, c, d))
    return np.array(tris, dtype=np.float32)


def sphere_and_field(field_res=40, nu=24, nv=32):
    """Cornell walls + a height field over the floor + a sphere: a few thousand triangles"""
    walls, walb = _walls()
    hf = height_field(field_res)
    sp = sphere((0.45, 0.45, 0.55), 0.18, nu, nv)
    light = np.array(_light(), dtype=np.float32)
    tri = np.concatenate([np.array(walls, np.float32).reshape(-1, 3, 3), hf, sp, light])
    alb = np.concatenate([np.array(walb, np.float32), np.tile([[0.5, 0.6, 0.4]], (len(hf), 1)),
                          np.tile([[0.8, 0.3, 0.3]], (len(sp), 1)), np.tile([[0.7, 0.7, 0.7]], (len(light), 1))])
    em = np.zeros(len(tri), np.uint8)
    em[-len(light):] = 1
    return MR.Scene(tri, alb, em, 80.0, (0, 0, 0), (1, 1, 1))


def soup(n=3000, seed=7):
    """random triangles of random orientation inside the unit box, a few of them emissive: the normal cones bound
    nothing"""
    rng = np.random.default_rng(seed)
    c = rng.uniform(0.1, 0.9, (n, 1, 3))
    tri = np.clip(c + rng.normal(0, 0.04, (n, 3, 3)), 0.0, 1.0).astype(np.float32)
    alb = rng.uniform(0.2, 0.9, (n, 3)).astype(np.float32)
    em = np.zeros(n, np.uint8)
    em[rng.choice(n, 20, replace=False)] = 1
    return MR.Scene(tri, alb, em, 50.0, (0, 0, 0), (1, 1, 1))


def large_field(res):
    """a height field of 2 res^2 triangles plus the Cornell light: the ~1 M-triangle scene of tools/time_mesh_trace.py"""
    hf = height_field(res)
    light = np.array(_light(), dtype=np.float32)
    tri = np.concatenate([hf, light])
    alb = np.full((len(tri), 3), 0.6, np.float32)
    em = np.zeros(len(tri), np.uint8)
    em[-2:] = 1
    return MR.Scene(tri, alb, em, 100.0, (0, 0, 0), (1, 1, 1))
