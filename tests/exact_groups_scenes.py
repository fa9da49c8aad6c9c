"""Scenes where the reference's group bounding-box culls decide what a ray hits (RTC_OPT_EXACT_GROUPS), shared by the
host and GPU tests of the option.  Each builder takes the API to build with (product session or oracle)."""
import numpy as np

from ray_tracer_challenge_b200.scenes import CSG_DIFFERENCE, Material, PI, PointLight, _xorshift64star

RTC_OPT_EXACT_GROUPS = 9


def stale_box(rt, stale=True, width=96, height=64, n=400):
    """400 spheres in one group.  stale: divide(8) caches the group boxes, then set_transformation moves every sphere
    2 units along x — the reference keeps culling with the old boxes (group.rs:19) and clips whatever left them.
    Returns the camera, the world and the spheres' shape handles."""
    rnd = _xorshift64star(3)
    g = rt.GroupShape()
    handles = []
    for _ in range(n):
        cx, cy, cz = ((rnd() * 2 - 1) * 4 for _ in range(3))
        sphere = rt.Sphere.build(rt.translation(cx, cy, cz) * rt.scaling(0.3, 0.3, 0.3), Material(color=(0.8, 0.6, 0.3)))
        g.add_child(sphere)
        handles.append(sphere.handle)
    if stale:
        g.divide(8)
        g.set_transformation(rt.translation(2.0, 0.0, 0.0))
    else:
        g.set_transformation(rt.translation(2.0, 0.0, 0.0))
        g.divide(8)
    world = rt.World([g], PointLight((-10, 10, -10), (1, 1, 1)))
    cam = rt.Camera(width, height, PI / 3, rt.view_transform((0, 0, -14), (0, 0, 0), (0, 1, 0)))
    return cam, world, handles


def csg_in_group(rt, width=96, height=64, n_spheres=60, glass=False):
    """CSGs (sphere minus cylinder) and spheres in one group whose boxes go stale as in stale_box: the group culls the
    CSGs with the old box.  n_spheres = 60: a tree scene; a handful: a small scene.  glass: the CSGs are glass, so the
    n1 / n2 container walk meets them too."""
    rnd = _xorshift64star(11)
    g = rt.GroupShape()
    mat = (Material(color=(0.1, 0.1, 0.1), transparency=0.9, reflective=0.5, refractive_index=1.5) if glass
           else Material(color=(0.9, 0.8, 0.2)))
    for i in range(4):
        a = rt.Sphere.build(rt.identity_4x4(), mat)
        b = rt.Cylinder()
        b.minimum_y, b.maximum_y, b.closed = -2.0, 2.0, True
        b.set_transformation(rt.scaling(0.5, 1.0, 0.5))
        b.set_material(Material(color=(0.9, 0.2, 0.2)))
        csg = rt.CSG(CSG_DIFFERENCE, a, b)
        csg.set_transformation(rt.translation(-3.0 + 2.0 * i, 0.5 * (i % 2), 0.0) * rt.rotation_x(0.6 * i) * rt.scaling(0.8, 0.8, 0.8))
        g.add_child(csg)
    for _ in range(n_spheres):
        cx, cy, cz = ((rnd() * 2 - 1) * 4 for _ in range(3))
        g.add_child(rt.Sphere.build(rt.translation(cx, cy, cz + 3.0) * rt.scaling(0.25, 0.25, 0.25), Material(color=(0.3, 0.6, 0.8))))
    g.divide(2)
    g.set_transformation(rt.translation(1.5, 0.0, 0.0))
    floor = rt.Plane.build(rt.translation(0.0, -4.0, 0.0), Material(color=(0.8, 0.8, 0.8)))
    world = rt.World([g, floor], PointLight((-10, 10, -10), (1, 1, 1)))
    cam = rt.Camera(width, height, PI / 3, rt.view_transform((0, 1, -12), (0, 0, 0), (0, 1, 0)))
    return cam, world


def far_field(rt, grouped=True, n=400, dist=800.0, radius=0.004, spread=6.0, seed=5):
    """Tiny spheres far from the origin: the reference's f32 sphere test reports phantom hits many radii beyond their
    silhouettes, and with `grouped` the group boxes decide which of them survive.  Returns the camera, the world, the
    spheres' (centre, radius) and their shape handles.  (The tree's padding is far narrower
    than that phantom band, so ungrouped, the tree would miss phantom hits the reference reports: that is not a group
    cull, and these scenes keep every phantom hit the reference keeps inside the padding.)"""
    rnd = _xorshift64star(seed)
    spheres, centres = [], []
    for _ in range(n):
        c = ((rnd() * 2 - 1) * spread, (rnd() * 2 - 1) * spread, dist + (rnd() * 2 - 1) * spread)
        r = radius * (0.5 + rnd())
        spheres.append(rt.Sphere.build(rt.translation(*c) * rt.scaling(r, r, r), Material(color=(0.9, 0.9, 0.9))))
        centres.append((c, r))
    objects = spheres
    if grouped:  # every sphere in a group of its own: its box is the sphere's, inside the tree's padded box of the sphere
        outer = rt.GroupShape()
        for s in spheres:
            g = rt.GroupShape()
            g.add_child(s)
            outer.add_child(g)
        objects = [outer]
    world = rt.World(objects, PointLight((-10, 10, -10), (1, 1, 1)))
    cam = rt.Camera(32, 32, PI / 3, rt.view_transform((0, 0, 0), (0, 0, 1), (0, 1, 0)))
    return cam, world, centres, [sp.handle for sp in spheres]


def far_field_rays(centres, n_rays, seed=9, spread_radii=20.0):
    """Rays from the origin aimed within `spread_radii` radii of a random sphere's centre."""
    rng = np.random.default_rng(seed)
    o = np.zeros((n_rays, 3), np.float32)
    d = np.zeros((n_rays, 3), np.float32)
    for i in range(n_rays):
        c, r = centres[rng.integers(len(centres))]
        target = np.array(c, np.float64) + rng.normal(size=3) * r * spread_radii
        d[i] = target / np.linalg.norm(target)
    return o, d


def oracle_nearest(oracle, world, o, d, with_shapes=False):
    """World::intersect + Intersection::hit of the oracle: the hit distance, or -1 (and the hit shape's handle, or -1)."""
    out = np.full(len(o), -1.0, np.float32)
    shapes = np.full(len(o), -1, np.int64)
    for i in range(len(o)):
        ts, objs = oracle.probe.world_intersect(world, o[i], d[i], cap=4096)
        h = oracle.probe.hit_index(ts)
        if h >= 0:
            out[i], shapes[i] = np.float32(ts[h]), objs[h]
    return (out, shapes) if with_shapes else out


def same_spheres(host, world, emu_prims, host_handles, oracle_shapes, oracle_handles):
    """The device code's hit primitives (API primitive indices, -1: none) name the same spheres as the oracle's hit
    shapes, by position in the two builders' sphere lists."""
    prim_shape = host.flatten(world)[3]
    host_index = {h: i for i, h in enumerate(host_handles)}
    oracle_index = {h: i for i, h in enumerate(oracle_handles)}
    got = np.array([host_index[prim_shape[p]] if p >= 0 else -1 for p in emu_prims])
    want = np.array([oracle_index[int(h)] if h >= 0 else -1 for h in oracle_shapes])
    return got == want
