"""Scene builders for the BASELINE configs and the parity suite, written once against the reference-shaped
API (`rt` is an api.Api: the product session or, in tests, the oracle binding).

Parameters are transcribed from the reference's demos (SURVEY.md Appendix C):
  soft_shadows      demos/src/bin/soft_shadows.rs:33-169      (BASELINE configs 1 and 3)
  reflect_refract   demos/src/bin/reflect_refract.rs:35-178   (config 2)
  hexagons          demos/src/bin/hexagons.rs:33-103
  first_scene / first_plane / first_patterns / first_textures / skybox / here_be_dragons
                    the remaining camera demos of demos/src/bin/ (external image / mesh files replaced by synthetic ones)
  textured          first_textures.rs / skybox.rs in miniature (UVImage over every mapping, synthetic PPMs)
  filter_zoo        parity scene for the shadow filter (spheres / planes / axis-aligned cubes, area light)
  dragon_element    demos/src/bin/here_be_dragons.rs:242-338  (config 4, with a synthetic OBJ: lib/resources
                    holds no mesh besides test/triangles.obj)
  stress            SURVEY.md §8d config 5 (100 k spheres + cylinders/cones/cubes + CSG + checker plane)
Each builder returns (camera, world).
"""
from __future__ import annotations

import math

import numpy as np

from .api import REFRACTION_GLASS, Material, PointLight, RectangleLight, color_from_hex, glass, metal

PI = float(np.float32(math.pi))
CSG_UNION, CSG_INTERSECTION, CSG_DIFFERENCE = 0, 1, 2


def jitter_table(n: int, seed: int = 0xC0FFEE):
    """Deterministic table of n values in (0, 1] (the support of rand's OpenClosed01, rectangle_light.rs:46)."""
    out, state = [], seed & 0xFFFFFFFFFFFFFFFF
    for _ in range(n):
        state = (state * 6364136223846793005 + 1442695040888963407) & 0xFFFFFFFFFFFFFFFF
        out.append(float(np.float32(((state >> 40) + 1) * 2.0 ** -24)))
    return out


def default_world(rt, width=11, height=11):
    """camera.rs:155-167"""
    camera = rt.Camera(width, height, PI / 2.0, rt.view_transform((0, 0, -5), (0, 0, 0), (0, 1, 0)))
    return camera, rt.World.default()


def soft_shadows(rt, width=1000, height=400, u_steps=10, v_steps=10, jitter="table", seed=0):
    """jitter: "table" (2*cells entries from jitter_table), "constant" (0.5), a list, or None (counter RNG)."""
    if jitter == "table":
        jitter = jitter_table(2 * u_steps * v_steps)
    elif jitter == "constant":
        jitter = [0.5]
    light = RectangleLight((1.5, 1.5, 1.5), (-1, 2, 4), (2, 0, 0), u_steps, (0, 2, 0), v_steps, jitter, seed)
    lampshade = rt.Cube.build(rt.translation(0.0, 3.0, 4.0) * rt.scaling(1.0, 1.0, 0.01),
                              Material(color=(1.5, 1.5, 1.5), ambient=1.0, diffuse=0.0, specular=0.0))
    lampshade.set_casts_shadow(False)
    floor = rt.Plane.build(rt.identity_4x4(), Material(color=(1, 1, 1), ambient=0.025, diffuse=0.67, specular=0.0))
    sphere1 = rt.Sphere.build(rt.translation(0.5, 0.5, 0.0) * rt.scaling(0.5, 0.5, 0.5),
                              Material(color=(1, 0, 0), ambient=0.1, specular=0.0, diffuse=0.6, reflective=0.3))
    sphere2 = rt.Sphere.build(rt.translation(-0.25, 0.33, 0.0) * rt.scaling(0.33, 0.33, 0.33),
                              Material(color=(0.5, 0.5, 1), ambient=0.1, specular=0.0, diffuse=0.6, reflective=0.3))
    world = rt.World([lampshade, floor, sphere1, sphere2], light)
    camera = rt.Camera(width, height, PI / 4.0, rt.view_transform((-3, 1, 2.5), (0, 0.5, 0), (0, 1, 0)))
    return camera, world


def filter_zoo(rt, width=320, height=200, area_light=True, jitter=None, seed=11):
    """Parity scene for the shadow filter (rtc_device.cuh: shadow_filter): only spheres, planes and axis-aligned
    cubes, so every shadow ray goes through the filter — with rotated / sheared / squashed spheres, tilted planes,
    objects touching each other and the floor (tangent shadow rays), a non-casting sphere and cube between the light
    and the floor, and a light sample grid whose edge grazes a cube.  Not a reference demo."""
    if area_light:
        light = RectangleLight((1.2, 1.2, 1.2), (-2.0, 4.0, -3.0), (3.0, 0, 0), 3, (0, 0.5, 2.0), 2,
                               jitter_table(12) if jitter == "table" else jitter, seed)
    else:
        light = PointLight((-3.0, 5.0, -4.0), (1, 1, 1))
    floor = rt.Plane.build(rt.identity_4x4(), Material(color=(0.9, 0.9, 0.9), specular=0.0, reflective=0.1,
                                                       pattern=rt.Checkers((0.9, 0.9, 0.9), (0.3, 0.3, 0.35))))
    wall = rt.Plane.build(rt.translation(0.0, 0.0, 6.0) * rt.rotation_x(PI / 2.0 - 0.2) * rt.rotation_z(0.15),
                          Material(color=(0.7, 0.8, 1.0), specular=0.1))
    ball = rt.Sphere.build(rt.translation(0.0, 1.0, 0.0), Material(color=(1, 0.3, 0.2), reflective=0.2))
    egg = rt.Sphere.build(rt.translation(1.8, 0.6, -0.5) * rt.rotation_z(0.5) * rt.rotation_y(0.9) * rt.scaling(0.9, 0.45, 0.6),
                          Material(color=(0.2, 0.8, 0.3), shininess=50.0))
    sheared = rt.Sphere.build(rt.translation(-2.0, 0.7, 0.8) * rt.shearing(0.5, 0.0, 0.0, 0.3, 0.0, 0.0) * rt.scaling(0.7, 0.7, 0.7),
                              Material(color=(0.3, 0.4, 0.9)))
    disc = rt.Sphere.build(rt.translation(0.5, 0.05, -2.0) * rt.scaling(0.8, 0.05, 0.8), Material(color=(0.8, 0.8, 0.2)))
    touching = rt.Sphere.build(rt.translation(0.0, 0.4, -1.4) * rt.scaling(0.4, 0.4, 0.4),
                               Material(color=(0.9, 0.5, 0.9), reflective=0.3))
    box = rt.Cube.build(rt.translation(-0.9, 0.5, -2.2) * rt.scaling(0.4, 0.5, 0.3), Material(color=(0.6, 0.4, 0.2)))
    slab = rt.Cube.build(rt.translation(2.5, 1.5, 2.0) * rt.scaling(0.2, 1.5, 1.0), Material(color=(0.4, 0.7, 0.7), reflective=0.4))
    shade = rt.Cube.build(rt.translation(-0.5, 4.0, -2.0) * rt.scaling(1.5, 0.02, 1.0),
                          Material(color=(1.2, 1.2, 1.0), ambient=1.0, diffuse=0.0, specular=0.0))
    shade.set_casts_shadow(False)
    ghost = rt.Sphere.build(rt.translation(-1.0, 2.2, -1.0) * rt.scaling(0.5, 0.5, 0.5),
                            Material(color=(0.1, 0.1, 0.1), transparency=0.9, refractive_index=1.0, diffuse=0.1, ambient=0.0))
    ghost.set_casts_shadow(False)
    world = rt.World([floor, wall, ball, egg, sheared, disc, touching, box, slab, shade, ghost], light)
    camera = rt.Camera(width, height, PI / 3.0, rt.view_transform((0.5, 2.5, -7.0), (0, 1.0, 0), (0, 1, 0)))
    return camera, world


def _three_spheres(rt, pattern=None):
    """The left / middle / right spheres shared by first_scene.rs:54-87, first_plane.rs:34-67, first_patterns.rs:40-70."""
    def mat(color):
        return Material(color=color, diffuse=0.7, specular=0.3) if pattern is None else Material(pattern=pattern, diffuse=0.7, specular=0.3)
    middle = rt.Sphere.build(rt.translation(-0.5, 1.0, 0.5), mat((0.1, 1, 0.5)))
    right = rt.Sphere.build(rt.shearing(0.0, 1.0, 0.0, 0.0, 0.0, 1.0) * rt.translation(1.5, 0.5, -0.5) * rt.scaling(0.5, 0.5, 0.5),
                            mat((0.5, 1, 0.1)))
    left = rt.Sphere.build(rt.translation(-1.5, 0.33, -0.75) * rt.scaling(0.33, 0.33, 0.33), mat((1, 0.8, 0.1)))
    return left, middle, right


def _first_camera(rt, width, height):
    return rt.Camera(width, height, PI / 3.0, rt.view_transform((0, 1.5, -5), (0, 1, 0), (0, 1, 0)))


def first_scene(rt, width=1000, height=500):
    """demos/src/bin/first_scene.rs:25-107 — the room is made of extremely flattened spheres."""
    room = Material(color=(1, 0.9, 0.9), specular=0.0)
    floor = rt.Sphere.build(rt.scaling(10.0, 0.01, 10.0), room)
    left_wall = rt.Sphere.build(rt.translation(0.0, 0.0, 5.0) * rt.rotation_y(-PI / 4.0) * rt.rotation_x(PI / 2.0)
                                * rt.scaling(10.0, 0.01, 10.0), room)
    right_wall = rt.Sphere.build(rt.translation(0.0, 0.0, 5.0) * rt.rotation_y(PI / 4.0) * rt.rotation_x(PI / 2.0)
                                 * rt.scaling(10.0, 0.01, 10.0), room)
    left, middle, right = _three_spheres(rt)
    world = rt.World([floor, left_wall, right_wall, left, middle, right], PointLight((-10, 10, -10), (1, 1, 1)))
    return _first_camera(rt, width, height), world


def first_plane(rt, width=100, height=50):
    """demos/src/bin/first_plane.rs:24-86"""
    floor = rt.Plane.build(rt.scaling(10.0, 0.01, 10.0), Material(color=(1, 0.9, 0.9), specular=0.0))
    left, middle, right = _three_spheres(rt)
    world = rt.World([floor, left, middle, right], PointLight((-10, 10, -10), (1, 1, 1)))
    return _first_camera(rt, width, height), world


def first_patterns(rt, width=100, height=50):
    """demos/src/bin/first_patterns.rs:28-92"""
    stripes = rt.Stripes((1.0, 0.2, 0.4), (0.1, 0.1, 0.1))
    stripes.set_transformation(rt.scaling(0.3, 0.3, 0.3) * rt.rotation_z(3.0 * PI / 4.0))
    sine2d = rt.Sine2D((0.1, 1, 0.5), (0.9, 0.2, 0.6))
    sine2d.set_transformation(rt.scaling(0.005, 1.0, 0.005) * rt.translation(-5.0, 1.0, 0.5))
    floor = rt.Plane.build(rt.scaling(10.0, 0.01, 10.0), Material(pattern=sine2d, specular=0.0))
    left, middle, right = _three_spheres(rt, stripes)
    world = rt.World([floor, left, middle, right], PointLight((-10, 10, -10), (1, 1, 1)))
    return _first_camera(rt, width, height), world


# constants.rs:8-46 colours used by uv.rs:328-344
_YELLOW, _CYAN, _RED, _BLUE, _BROWN = (1, 1, 0), (0, 1, 1), (1, 0, 0), (0, 0, 1), (1, 0.5, 0)
_GREEN, _PURPLE, _WHITE = (0, 1, 0), (1, 0, 1), (1, 1, 1)


def align_check_cubic_map(rt):
    """get_align_check_cubic_map_pattern, uv.rs:328-344"""
    left = rt.AlignCheck(_YELLOW, _CYAN, _RED, _BLUE, _BROWN)
    front = rt.AlignCheck(_CYAN, _RED, _YELLOW, _BROWN, _GREEN)
    right = rt.AlignCheck(_RED, _YELLOW, _PURPLE, _GREEN, _WHITE)
    back = rt.AlignCheck(_GREEN, _PURPLE, _CYAN, _WHITE, _BLUE)
    up = rt.AlignCheck(_BROWN, _CYAN, _PURPLE, _RED, _YELLOW)
    down = rt.AlignCheck(_PURPLE, _BROWN, _GREEN, _BLUE, _WHITE)
    return rt.CubicMap(front, back, left, right, up, down)


def first_textures(rt, width=1000, height=500, earth_ppm=None, u_steps=10, v_steps=10, seed=3):
    """demos/src/bin/first_textures.rs:34-171.  The earth image is an external file there; here a synthetic PPM.  The
    light is the demo's 10x10 RectangleLight with jitter `None` (first_textures.rs:161-171): the counter-based
    generator stands in for thread_rng on both sides."""
    from .api import SG_MAP_CYLINDRICAL, SG_MAP_PLANAR, SG_MAP_SPHERICAL

    black, white = (0, 0, 0), (1, 1, 1)
    floor = rt.Plane.build(rt.scaling(10.0, 0.01, 10.0),
                           Material(specular=0.0, pattern=rt.TextureMap(rt.UVCheckers(16.0, 8.0, black, white), SG_MAP_PLANAR)))
    sphere = rt.Sphere.build(rt.translation(-2.5, 1.3, 3.0),
                             Material(pattern=rt.TextureMap(rt.UVCheckers(16.0, 8.0, black, white), SG_MAP_SPHERICAL),
                                      diffuse=0.7, specular=0.3))
    canvas = rt.canvas_from_ppm(earth_ppm if earth_ppm is not None else synthetic_ppm(128, 64, seed=7))
    earth = rt.Sphere.build(rt.translation(0.0, 1.0, 0.0) * rt.rotation_x(-0.5) * rt.rotation_y(-1.5),
                            Material(pattern=rt.TextureMap(rt.UVImage(canvas), SG_MAP_SPHERICAL), diffuse=0.9, specular=0.1,
                                     shininess=10.0, ambient=0.1))
    pedestal = rt.Cylinder()
    pedestal.maximum_y, pedestal.minimum_y, pedestal.closed = 0.0, -0.15, True
    pedestal.set_material(Material(color=(0.2, 0.2, 0.2), ambient=0.0, diffuse=0.8, specular=0.0, reflective=0.2))
    earth_display = rt.GroupShape()
    earth_display.add_child(earth)
    earth_display.add_child(pedestal)
    earth_display.set_transformation(rt.translation(-0.2, 0.15, 0.5))
    cylinder = rt.Cylinder()
    cylinder.set_transformation(rt.translation(2.0, 2.0, 2.0))
    cylinder.set_material(Material(ambient=0.1, specular=0.6, shininess=15.0, diffuse=0.8,
                                   pattern=rt.TextureMap(rt.UVCheckers(16.0, 16.0, (0, 0.5, 0), white), SG_MAP_CYLINDRICAL)))
    cylinder.maximum_y, cylinder.minimum_y = 3.0, -3.0
    cube = rt.Cube()
    cube.set_transformation(rt.translation(5.0, 2.0, 2.0) * rt.rotation_x(-PI / 4.0))
    cube.set_material(Material(pattern=align_check_cubic_map(rt)))
    light = RectangleLight((1.5, 1.5, 1.5), (-10, 10, -10), (2, 0, 0), u_steps, (0, 2, 0), v_steps, None, seed)
    world = rt.World([floor, sphere, cylinder, cube, earth_display], light)
    camera = rt.Camera(width, height, PI / 3.0, rt.view_transform((0, 1.5, -10), (2, 2.8, 0), (0, 1, 0)))
    return camera, world


def skybox(rt, width=800, height=400, face_size=64):
    """demos/src/bin/skybox.rs:26-129 with synthetic face images (the demo reads six external PPMs).  Note the demo's
    own assignment: left <- posx.ppm, right <- negx.ppm (skybox.rs:88-91)."""
    sphere = rt.Sphere.build(rt.scaling(0.75, 0.75, 0.75) * rt.translation(0.0, 0.0, 5.0),
                             Material(diffuse=0.4, specular=0.6, shininess=20.0, reflective=0.6, ambient=0.0))
    names = ["posz", "negz", "posx", "negx", "posy", "negy"]  # front, back, left, right, up, down
    faces = [rt.UVImage(rt.canvas_from_ppm(synthetic_ppm(face_size, face_size, seed=20 + i))) for i, _ in enumerate(names)]
    box = rt.Cube.build(rt.scaling(1000.0, 1000.0, 1000.0),
                        Material(diffuse=0.0, specular=0.0, ambient=1.0, pattern=rt.CubicMap(*faces)))
    world = rt.World([sphere, box], PointLight((0, 100, 0), (1, 1, 1)))
    camera = rt.Camera(width, height, 1.2, rt.view_transform((0, 0, 0), (0, 0, 5), (0, 1, 0)))
    return camera, world


def synthetic_ppm(width=48, height=32, seed=5, scale=255):
    """A deterministic P3 image (colour ramps + a checker overlay + a comment line and wrapped rows), as text."""
    rows, state = [f"P3\n# synthetic texture {width}x{height}\n{width} {height}\n{scale}"], seed
    for y in range(height):
        vals = []
        for x in range(width):
            state = (state * 1103515245 + 12345) & 0x7FFFFFFF
            check = ((x // 4) + (y // 4)) % 2
            r = (x * scale) // max(width - 1, 1)
            g = (y * scale) // max(height - 1, 1)
            b = (scale if check else scale // 4) - (state % (scale // 8 + 1))
            vals += [r, g, max(b, 0)]
        cut = len(vals) // 2 + 1  # not a multiple of 3: triplets span lines (canvas.rs ppm_parsing_allows_rgb_triplet_to_span_lines)
        rows.append(" ".join(str(v) for v in vals[:cut]) + "\n  " + " ".join(str(v) for v in vals[cut:]))
    return "\n".join(rows) + "\n"


def textured(rt, width=320, height=200):
    """first_textures.rs:34-171 / skybox.rs:26-129 in miniature, with synthetic PPMs instead of the external image
    files: UVImage (uv.rs:346-377) through the spherical, planar and cylindrical mappings and a six-image cube map."""
    from .api import SG_MAP_CYLINDRICAL, SG_MAP_PLANAR, SG_MAP_SPHERICAL

    earth = rt.UVImage(rt.canvas_from_ppm(synthetic_ppm(64, 32, seed=1)))
    tiles = rt.UVImage(rt.canvas_from_ppm(synthetic_ppm(16, 16, seed=2, scale=100)))
    label = rt.UVImage(rt.canvas_from_ppm(synthetic_ppm(40, 20, seed=3)))
    faces = [rt.UVImage(rt.canvas_from_ppm(synthetic_ppm(24, 24, seed=10 + i))) for i in range(6)]
    floor_map = rt.TextureMap(tiles, SG_MAP_PLANAR)
    floor = rt.Plane.build(rt.identity_4x4(), Material(pattern=floor_map, specular=0.0, reflective=0.2))
    globe_map = rt.TextureMap(earth, SG_MAP_SPHERICAL)
    globe_map.set_transformation(rt.rotation_y(1.9))
    globe = rt.Sphere.build(rt.translation(0.0, 1.1, 0.0) * rt.rotation_z(0.3), Material(pattern=globe_map, diffuse=0.9, specular=0.1, shininess=10.0))
    can_map = rt.TextureMap(label, SG_MAP_CYLINDRICAL)
    can_map.set_transformation(rt.scaling(1.0, 1.0 / PI, 1.0))
    can = rt.Cylinder()
    can.minimum_y, can.maximum_y, can.closed = 0.0, 1.0, True
    can.set_transformation(rt.translation(-2.4, 0.0, 0.5) * rt.scaling(0.6, 1.6, 0.6))
    can.set_material(Material(pattern=can_map, specular=0.6, shininess=15.0))
    box = rt.Cube.build(rt.translation(2.4, 0.8, 0.3) * rt.rotation_y(0.6) * rt.rotation_x(0.3) * rt.scaling(0.8, 0.8, 0.8),
                        Material(pattern=rt.CubicMap(*faces), specular=0.0))
    sky = rt.Cube.build(rt.scaling(50.0, 50.0, 50.0),
                        Material(pattern=rt.CubicMap(*faces), diffuse=0.0, specular=0.0, ambient=1.0))
    sky.set_casts_shadow(False)
    world = rt.World([floor, globe, can, box, sky], PointLight((-5.0, 8.0, -6.0), (1, 1, 1)))
    camera = rt.Camera(width, height, PI / 3.0, rt.view_transform((0.0, 2.2, -6.5), (0, 0.9, 0), (0, 1, 0)))
    return camera, world


def random_filter_scene(rt, seed, width=160, height=100, extreme=None):
    """A random filter-eligible scene (spheres with random rotations / shears / squashes, tilted planes, axis-aligned
    boxes, some touching or interpenetrating, some not casting shadows) under a random area or point light: fuzzing
    input for the shadow filter's on / off equality test.

    extreme: None, or one of the regimes the filter's RELATIVE error bounds must survive —
      "millimetre" / "kilometre"  every length of the scene (objects, light, camera) times 1e-3 / 1e3;
      "far light"                 the light 1e4 units away along its own direction from the scene;
      "tiny spheres"              radius-1e-3 spheres on the floor, seen (and shadow-tested) from units away;
      "stretched"                 ellipsoids near the eligibility limit (condition number ~60);
      "grazing"                   the light a hair above the floor plane: shadow segments almost parallel to it."""
    rnd = _xorshift64star(0x5EED0000 + seed)
    S = {"millimetre": 1e-3, "kilometre": 1e3}.get(extreme, 1.0)

    def u(a, b):
        return a + (b - a) * rnd()

    def mat():
        return Material(color=(u(0.2, 1), u(0.2, 1), u(0.2, 1)), reflective=u(0, 0.4) if rnd() < 0.3 else 0.0,
                        specular=u(0, 0.9), shininess=u(5, 200))

    objects = [rt.Plane.build(rt.identity_4x4(), Material(color=(0.9, 0.9, 0.9), specular=0.0))]
    if rnd() < 0.6:
        objects.append(rt.Plane.build(rt.translation(0.0, 0.0, u(4, 8)) * rt.rotation_x(PI / 2.0 + u(-0.3, 0.3)) * rt.rotation_z(u(-0.3, 0.3)), mat()))
    for _ in range(2 + int(rnd() * 5)):
        r = u(0.25, 1.1)
        t = rt.translation(u(-3, 3), r * u(0.6, 1.4), u(-2.5, 3))
        kind = rnd()
        if kind < 0.35:
            t = t * rt.scaling(r, r, r)
        elif kind < 0.7:
            t = t * rt.rotation_y(u(0, 6.28)) * rt.rotation_z(u(0, 6.28)) * rt.scaling(r, r * u(0.2, 1.0), r * u(0.4, 1.0))
        else:
            t = t * rt.shearing(u(-0.5, 0.5), 0.0, 0.0, u(-0.5, 0.5), 0.0, 0.0) * rt.scaling(r, r, r)
        sphere = rt.Sphere.build(t, mat())
        if rnd() < 0.15:
            sphere.set_casts_shadow(False)
        objects.append(sphere)
    for _ in range(int(rnd() * 3)):
        box = rt.Cube.build(rt.translation(u(-3, 3), u(0.2, 1.5), u(-2, 3)) * rt.scaling(u(0.2, 0.9), u(0.2, 1.2), u(0.2, 0.9)), mat())
        if rnd() < 0.25:
            box.set_casts_shadow(False)
        objects.append(box)
    if extreme == "tiny spheres":
        for _ in range(4):
            objects.append(rt.Sphere.build(rt.translation(u(-2, 2), 1e-3, u(-4, 1)) * rt.scaling(1e-3, 1e-3, 1e-3), mat()))
    if extreme == "stretched":
        for _ in range(3):
            r = u(0.4, 1.0)
            objects.append(rt.Sphere.build(rt.translation(u(-3, 3), u(0.5, 1.5), u(-2, 3)) * rt.rotation_y(u(0, 6.28)) *
                                           rt.rotation_z(u(0, 1.5)) * rt.scaling(r, r / u(20.0, 28.0), r * u(0.5, 1.0)), mat()))
    if rnd() < 0.7 or extreme == "grazing":
        us, vs = 1 + int(rnd() * 4), 1 + int(rnd() * 4)
        mode = rnd()
        jitter = jitter_table(2 * us * vs, seed + 11) if mode < 0.4 else ([0.5] if mode < 0.6 else None)
        corner, eu, ev = (u(-4, 0), u(2.5, 6), u(-5, -1)), (u(0.3, 1.0), 0, u(-0.2, 0.2)), (0, u(0.3, 1.0), u(-0.2, 0.2))
        if extreme == "grazing":  # a horizontal strip light just above the floor
            corner, eu, ev = (u(-6, -4), u(1e-4, 3e-3), u(-5, -1)), (u(0.3, 1.0), 0, u(-0.2, 0.2)), (0, u(1e-4, 1e-3), u(0.3, 1.0))
        if extreme == "far light":
            k = 1e4 / math.sqrt(sum(c * c for c in corner))
            corner = tuple(c * k for c in corner)
        light = RectangleLight((1.2, 1.2, 1.2), tuple(c * S for c in corner), tuple(c * S for c in eu), us,
                               tuple(c * S for c in ev), vs, jitter, seed)
    else:
        pos = (u(-6, 6), u(3, 9), u(-7, -2))
        if extreme == "far light":
            k = 1e4 / math.sqrt(sum(c * c for c in pos))
            pos = tuple(c * k for c in pos)
        light = PointLight(tuple(c * S for c in pos), (1, 1, 1))
    if S != 1.0:  # the whole scene in other units: every object's transform gains a uniform scaling on the left
        scaled = []
        for o in objects:
            o.set_transformation(rt.scaling(S, S, S) * o.transformation())
            scaled.append(o)
        objects = scaled
    world = rt.World(objects, light)
    frm = (u(-2, 2), u(1.5, 3.5), u(-8, -6))
    camera = rt.Camera(width, height, PI / 3.0, rt.view_transform(tuple(c * S for c in frm), (0, 1.0 * S, 0), (0, 1, 0)))
    return camera, world


def reflect_refract(rt, width=1000, height=500, with_csg=False):
    stripes = rt.Stripes((1.0, 0.2, 0.4), (0.1, 0.1, 0.1))
    stripes_t = rt.scaling(0.3, 0.3, 0.3) * rt.rotation_z(3.0 * PI / 4.0)
    stripes.set_transformation(stripes_t)
    sine2d = rt.Sine2D((0.1, 1, 0.5), (0.9, 0.2, 0.6))
    sine2d.set_transformation(rt.scaling(0.05, 1.0, 0.05) * rt.translation(-5.0, 1.0, 0.5))
    floor = rt.Plane.build(rt.scaling(10.0, 0.1, 10.0), Material(pattern=sine2d, specular=0.0, reflective=0.5))
    middle = _clear_sphere(rt)
    metal_rings = metal()
    rings = rt.Rings((0.5, 0.5, 0.0), (0.5, 0.5, 0.5))  # yellow() / 2., white() / 2.
    rings.set_transformation(rt.scaling(0.1, 0.1, 0.1))
    metal_rings.pattern = rings
    right = rt.Sphere.build(
        rt.shearing(0.0, 1.0, 0.0, 0.0, 0.0, 1.0) * rt.translation(1.5, 0.5, -0.5) * rt.scaling(0.5, 0.5, 0.5), metal_rings)
    stripes2 = rt.Stripes((0.25, 0.05, 0.1), (0.025, 0.025, 0.025))  # a / 4., b / 4.
    stripes2.set_transformation(stripes_t)
    left = rt.Sphere.build(rt.translation(-1.5, 0.33, -0.75) * rt.scaling(0.33, 0.33, 0.33),
                           Material(pattern=stripes2, diffuse=0.7, specular=1.0, reflective=0.8, shininess=300.0))
    cylinder = _rr_cylinder(rt)
    cone = rt.Cone()
    cone.maximum_y = 1.5
    cone.minimum_y = 0.0
    cone.set_material(Material(color=(0.6, 0.3, 0.1), reflective=0.5, shininess=10.0, specular=0.8))
    cone.set_transformation(rt.translation(-3.5, 0.0, 4.0) * rt.scaling(0.33, 1.8, 0.33))
    objects = [floor, left, middle, right, cylinder, cone]
    if with_csg:  # reflect_refract.rs:160-178 (commented out of the shipped world at :112)
        s1 = _clear_sphere(rt)
        s1.set_transformation(rt.translation(0.0, 1.0, 0.0))
        s2 = _rr_cylinder(rt)
        s2.set_transformation(rt.scaling(0.2, 2.0, 0.2))
        s2.set_material(Material(reflective=0.0, refractive_index=1.0, transparency=1.0))
        s2.set_casts_shadow(False)
        csg = rt.CSG(CSG_DIFFERENCE, s1, s2)
        csg.set_transformation(rt.translation(0.0, 0.0, 2.0))
        objects.append(csg)
    world = rt.World(objects, PointLight((-10, 10, -10), (1, 1, 1)))
    camera = rt.Camera(width, height, PI / 3.0, rt.view_transform((0, 1.5, -5), (0, 1, 0), (0, 1, 0)))
    return camera, world


def _clear_sphere(rt):
    s = rt.Sphere.build(rt.translation(-0.5, 1.0, 0.5),
                        Material(color=(0, 0, 0), specular=1.0, shininess=300.0, transparency=1.0,
                                 refractive_index=REFRACTION_GLASS, reflective=1.0))
    s.set_casts_shadow(False)
    return s


def _rr_cylinder(rt):
    c = rt.Cylinder()
    c.maximum_y = 1.5
    c.minimum_y = 0.0
    c.set_material(Material(reflective=1.0, color=(0.5, 0.5, 0.5), shininess=300.0, specular=0.8))
    c.set_transformation(rt.translation(3.7, 0.0, 4.0) * rt.scaling(0.33, 1.8, 0.33))
    return c


def hexagons(rt, width=1000, height=500):
    floor = rt.Plane()
    floor.set_transformation(rt.translation(0.0, 0.0, 5.0) * rt.rotation_x(PI / 2.0))
    floor.set_material(Material(pattern=rt.Checkers(color_from_hex("#C5D86D"), color_from_hex("#261C15"))))
    m = glass()

    def side():
        g = rt.GroupShape()
        g.add_child(rt.Sphere.build(rt.translation(0.0, 0.0, -1.0) * rt.scaling(0.25, 0.25, 0.25), m))
        edge = rt.Cylinder()
        edge.minimum_y = 0.0
        edge.maximum_y = 1.0
        edge.set_transformation(rt.translation(0.0, 0.0, -1.0) * rt.rotation_y(-PI / 6.0) * rt.rotation_z(-PI / 2.0)
                                * rt.scaling(0.25, 1.0, 0.25))
        edge.set_material(m)
        g.add_child(edge)
        return g

    hexagon = rt.GroupShape()
    for n in range(6):
        s = side()
        s.set_transformation(rt.rotation_y(n * PI / 3.0))
        hexagon.add_child(s)
    hexagon.set_transformation(rt.translation(0.0, 0.75, 0.0) * rt.rotation_x(PI / 2.0))
    world = rt.World([floor, hexagon], PointLight((-10, 10, -10), (1, 1, 1)))
    camera = rt.Camera(width, height, PI / 3.0, rt.view_transform((0, 1.5, -5), (0, 1, 0), (0, 1, 0)))
    return camera, world


def shapes_zoo(rt, width=320, height=200, area_light=False):
    """Every primitive kind, every pattern kind, closed cylinder / cone caps, a triangle fan, nested groups and a
    non-shadow-casting object in one frame (parity coverage, not a reference demo)."""
    floor_pat = rt.Checkers((0.9, 0.9, 0.9), (0.2, 0.25, 0.3))
    floor_pat.set_transformation(rt.scaling(0.75, 0.75, 0.75))
    floor = rt.Plane.build(rt.identity_4x4(), Material(pattern=floor_pat, specular=0.1, reflective=0.15))
    wall_pat = rt.Gradient((0.9, 0.3, 0.2), (0.2, 0.3, 0.9))
    wall_pat.set_transformation(rt.scaling(8.0, 1.0, 1.0) * rt.translation(-0.5, 0.0, 0.0))
    wall = rt.Plane.build(rt.translation(0.0, 0.0, 6.0) * rt.rotation_x(PI / 2.0), Material(pattern=wall_pat, specular=0.0))
    cube_pat = rt.CubicMap(*[rt.AlignCheck(*cols) for cols in _ALIGN_FACES])
    cube = rt.Cube.build(rt.translation(-2.2, 0.8, 1.0) * rt.rotation_y(0.6) * rt.rotation_x(0.3) * rt.scaling(0.7, 0.7, 0.7),
                         Material(pattern=cube_pat, ambient=0.2, diffuse=0.8, specular=0.3))
    globe_pat = rt.TextureMap(rt.UVCheckers(16.0, 8.0, (0.1, 0.5, 0.2), (0.95, 0.95, 0.8)), 0)
    globe = rt.Sphere.build(rt.translation(0.0, 1.0, 0.5) * rt.rotation_y(0.4), Material(pattern=globe_pat, shininess=50.0))
    can_pat = rt.TextureMap(rt.UVCheckers(8.0, 4.0, (0.8, 0.1, 0.1), (0.9, 0.9, 0.9)), 2)
    can = rt.Cylinder()
    can.minimum_y, can.maximum_y, can.closed = 0.0, 1.2, True
    can.set_transformation(rt.translation(2.0, 0.0, 0.3) * rt.scaling(0.5, 1.0, 0.5))
    can.set_material(Material(pattern=can_pat, reflective=0.1))
    hat = rt.Cone()
    hat.minimum_y, hat.maximum_y, hat.closed = -1.0, 0.0, True
    hat.set_transformation(rt.translation(2.0, 2.2, 0.3) * rt.scaling(0.6, 1.0, 0.6))
    ring_pat = rt.Rings((0.9, 0.8, 0.1), (0.3, 0.1, 0.5))
    ring_pat.set_transformation(rt.scaling(0.2, 0.2, 0.2))
    hat.set_material(Material(pattern=ring_pat, specular=0.6, shininess=30.0))
    marble = rt.Sphere.build(rt.translation(-0.9, 0.4, -1.2) * rt.scaling(0.4, 0.4, 0.4),
                             Material(color=(0.1, 0.1, 0.1), transparency=0.9, reflective=0.9, refractive_index=1.5,
                                      diffuse=0.1, ambient=0.05, shininess=300.0))
    bubble = rt.Sphere.build(rt.translation(-0.9, 0.4, -1.2) * rt.scaling(0.2, 0.2, 0.2),
                             Material(color=(1, 1, 1), transparency=1.0, reflective=0.5, refractive_index=1.00029,
                                      diffuse=0.0, ambient=0.0))
    ghost = rt.Sphere.build(rt.translation(0.8, 0.35, -1.6) * rt.scaling(0.35, 0.35, 0.35),
                            Material(color=(0.3, 0.6, 0.9), diffuse=0.7))
    ghost.set_casts_shadow(False)
    stripes = rt.Stripes((0.9, 0.9, 0.2), (0.1, 0.2, 0.7))
    stripes.set_transformation(rt.scaling(0.15, 1.0, 1.0) * rt.rotation_z(0.5))
    fan = rt.GroupShape()
    apex = (0.0, 1.0, 0.0)
    ring = [(math.cos(2 * math.pi * i / 6), 0.0, math.sin(2 * math.pi * i / 6)) for i in range(6)]
    for i in range(6):
        fan.add_child(rt.Triangle(apex, ring[i], ring[(i + 1) % 6]))
    fan.set_material(Material(pattern=stripes, specular=0.4))
    pyramid_holder = rt.GroupShape()
    pyramid_holder.add_child(fan)
    pyramid_holder.set_transformation(rt.translation(-3.0, 0.0, -1.0) * rt.scaling(0.6, 0.9, 0.6) * rt.rotation_y(0.3))
    sine = rt.Sine2D((0.9, 0.9, 0.9), (0.1, 0.4, 0.3))
    sine.set_transformation(rt.scaling(0.1, 1.0, 0.1))
    slab = rt.Cube.build(rt.translation(3.2, 0.15, -1.4) * rt.scaling(0.6, 0.15, 0.6), Material(pattern=sine, reflective=0.2))
    if area_light:
        light = RectangleLight((1.2, 1.2, 1.2), (-4, 6, -6), (2, 0, 0), 3, (0, 0, 2), 3, jitter_table(18))
    else:
        light = PointLight((-6, 8, -8), (1, 1, 1))
    world = rt.World([floor, wall, cube, globe, can, hat, marble, bubble, ghost, pyramid_holder, slab], light)
    camera = rt.Camera(width, height, PI / 3.0, rt.view_transform((0.5, 2.6, -6.5), (0, 0.9, 0), (0, 1, 0)))
    return camera, world


_R, _Y, _G, _C, _B, _P, _W, _BR = (1, 0, 0), (1, 1, 0), (0, 1, 0), (0, 1, 1), (0, 0, 1), (1, 0, 1), (1, 1, 1), (1, 0.5, 0)
# front, back, left, right, up, down (uv.rs:328-344)
_ALIGN_FACES = [(_C, _R, _Y, _BR, _G), (_G, _P, _C, _W, _B), (_Y, _C, _R, _B, _BR), (_R, _Y, _P, _G, _W),
                (_BR, _C, _P, _R, _Y), (_P, _BR, _G, _B, _W)]


def csg_gallery(rt, width=320, height=200):
    """Union / intersection / difference, a nested CSG, a CSG with a group operand and a transparent CSG child."""
    floor = rt.Plane.build(rt.identity_4x4(), Material(pattern=rt.Checkers((0.8, 0.8, 0.8), (0.3, 0.3, 0.3)), specular=0.0,
                                                       reflective=0.1))

    def lens():
        a = rt.Sphere.build(rt.translation(-0.35, 0, 0), Material(color=(0.9, 0.2, 0.2)))
        b = rt.Sphere.build(rt.translation(0.35, 0, 0), Material(color=(0.2, 0.2, 0.9)))
        return rt.CSG(CSG_INTERSECTION, a, b)

    c1 = lens()
    c1.set_transformation(rt.translation(-2.5, 1.0, 0.0) * rt.rotation_y(0.5))
    box = rt.Cube.build(rt.scaling(0.8, 0.8, 0.8), Material(color=(0.9, 0.7, 0.1), reflective=0.2))
    ball = rt.Sphere.build(rt.scaling(1.05, 1.05, 1.05), Material(color=(0.1, 0.7, 0.3)))
    c2 = rt.CSG(CSG_DIFFERENCE, box, ball)
    c2.set_transformation(rt.translation(0.0, 0.8, 0.0) * rt.rotation_y(0.7) * rt.rotation_x(0.2))
    # nested: (cube ∩ sphere) − three crossed cylinders (a group operand)
    rounded = rt.CSG(CSG_INTERSECTION, rt.Cube.build(rt.identity_4x4(), Material(color=(0.8, 0.3, 0.1))),
                     rt.Sphere.build(rt.scaling(1.35, 1.35, 1.35), Material(color=(0.2, 0.2, 0.2))))
    bars = rt.GroupShape()
    for rot in (rt.identity_4x4(), rt.rotation_x(PI / 2.0), rt.rotation_z(PI / 2.0)):
        cyl = rt.Cylinder()
        cyl.minimum_y, cyl.maximum_y, cyl.closed = -2.0, 2.0, True
        cyl.set_transformation(rot * rt.scaling(0.55, 1.0, 0.55))
        cyl.set_material(Material(color=(0.2, 0.7, 0.8)))
        bars.add_child(cyl)
    c3 = rt.CSG(CSG_DIFFERENCE, rounded, bars)
    c3.set_transformation(rt.translation(2.6, 1.0, 0.5) * rt.rotation_y(-0.5) * rt.rotation_x(0.4) * rt.scaling(0.8, 0.8, 0.8))
    # union with a glass operand (exercises n1/n2 through CSG-filtered hits)
    u1 = rt.Sphere.build(rt.translation(0, 0, 0), glass())
    u2 = rt.Cone()
    u2.minimum_y, u2.maximum_y, u2.closed = -1.0, 0.0, True
    u2.set_transformation(rt.translation(0.0, 1.6, 0.0))
    u2.set_material(Material(color=(0.8, 0.1, 0.6)))
    c4 = rt.CSG(CSG_UNION, u1, u2)
    c4.set_transformation(rt.translation(-0.6, 0.6, -2.2) * rt.scaling(0.6, 0.6, 0.6))
    holder = rt.GroupShape()
    holder.add_child(c4)
    world = rt.World([floor, c1, c2, c3, holder], PointLight((-5, 8, -8), (1, 1, 1)))
    camera = rt.Camera(width, height, PI / 3.0, rt.view_transform((0, 3.0, -7.0), (0, 0.8, 0), (0, 1, 0)))
    return camera, world


def _union_chain(rt, shapes):
    """CSG(union, CSG(union, ..., a), b): one more nesting level per shape after the second."""
    out = shapes[0]
    for s in shapes[1:]:
        out = rt.CSG(CSG_UNION, out, s)
    return out


def csg_die(rt, width=320, height=200, glassy=False, area_light=False, surrounded=False):
    """The book's chapter-16 die: a rounded cube (cube ∩ sphere) minus 21 pip spheres, a worst case of 46 hits per ray.
    Faces 1-3's pips are a union chain (the die nests 7 CSG levels deep), faces 4-6's pips sit in a group.
    `surrounded` adds 20 marbles, which puts the die in a tree scene rather than a small one."""
    if glassy:
        body = Material(color=(0.1, 0.1, 0.15), transparency=1.0, refractive_index=REFRACTION_GLASS, diffuse=0.1, ambient=0.05,
                        reflective=0.9, shininess=300.0)
    else:
        body = Material(color=(0.95, 0.93, 0.85), specular=0.4, shininess=80.0, reflective=0.05)
    pip_mat = Material(color=(0.1, 0.1, 0.12), specular=0.2) if not glassy else \
        Material(color=(0.6, 0.1, 0.1), transparency=0.6, refractive_index=1.2, diffuse=0.4, reflective=0.3)
    rounded = rt.CSG(CSG_INTERSECTION, rt.Cube.build(rt.identity_4x4(), body),
                     rt.Sphere.build(rt.scaling(1.45, 1.45, 1.45), body))
    grid = {1: [(0, 0)], 2: [(-1, -1), (1, 1)], 3: [(-1, -1), (0, 0), (1, 1)], 4: [(-1, -1), (-1, 1), (1, -1), (1, 1)],
            5: [(-1, -1), (-1, 1), (0, 0), (1, -1), (1, 1)], 6: [(-1, -1), (-1, 0), (-1, 1), (1, -1), (1, 0), (1, 1)]}
    # face -> (axis, sign); opposite faces add up to 7
    faces = {1: (2, -1.0), 6: (2, 1.0), 2: (0, 1.0), 5: (0, -1.0), 3: (1, 1.0), 4: (1, -1.0)}

    def pips(face):
        axis, sign = faces[face]
        out = []
        for a, b in grid[face]:
            c = [0.0, 0.0, 0.0]
            c[axis] = sign * 1.05
            c[(axis + 1) % 3], c[(axis + 2) % 3] = 0.5 * a, 0.5 * b
            out.append(rt.Sphere.build(rt.translation(*c) * rt.scaling(0.2, 0.2, 0.2), pip_mat))
        return out

    holes = rt.GroupShape()
    holes.add_child(_union_chain(rt, pips(1) + pips(2) + pips(3)))
    for face in (4, 5, 6):
        for p in pips(face):
            holes.add_child(p)
    die = rt.CSG(CSG_DIFFERENCE, rounded, holes)
    die.set_transformation(rt.translation(0.0, 1.0, 0.0) * rt.rotation_y(0.6) * rt.rotation_x(-0.25))
    floor = rt.Plane.build(rt.identity_4x4(), Material(pattern=rt.Checkers((0.8, 0.8, 0.8), (0.3, 0.35, 0.3)), specular=0.0,
                                                       reflective=0.1))
    objects = [floor, die]
    if surrounded:
        for i in range(20):
            a = 2 * math.pi * i / 20
            objects.append(rt.Sphere.build(rt.translation(3.0 * math.cos(a), 0.3, 3.0 * math.sin(a) + 1.0) * rt.scaling(0.3, 0.3, 0.3),
                                           Material(color=(0.2 + 0.04 * i, 0.5, 0.9 - 0.04 * i), reflective=0.2)))
    if area_light:
        light = RectangleLight((1.2, 1.2, 1.2), (-5.0, 7.0, -6.0), (2.0, 0, 0), 3, (0, 0, 2.0), 3, jitter_table(18))
    else:
        light = PointLight((-5.0, 8.0, -7.0), (1, 1, 1))
    camera = rt.Camera(width, height, PI / 3.0, rt.view_transform((1.0, 3.5, -5.5), (0, 0.9, 0), (0, 1, 0)))
    return camera, rt.World(objects, light)


def csg_carved_mesh(rt, width=320, height=200, n_u=24, n_v=12):
    """The divided synthetic_obj mesh minus a cylinder (one leaf per triangle: the worst case grows with the mesh), with a
    glass sphere in front of it."""
    mesh = rt.parse_obj(synthetic_obj(n_u, n_v))
    mesh.set_material(Material(color=(0.9, 0.5, 0.2), specular=0.3, shininess=20.0))
    mesh.divide(4)
    drill = rt.Cylinder()
    drill.minimum_y, drill.maximum_y, drill.closed = -3.0, 3.0, True
    drill.set_transformation(rt.translation(0.8, 0.0, 0.0) * rt.scaling(0.9, 1.0, 0.9))
    drill.set_material(Material(color=(0.2, 0.6, 0.9)))
    carved = rt.CSG(CSG_DIFFERENCE, mesh, drill)
    carved.set_transformation(rt.translation(0.0, 1.5, 0.0) * rt.rotation_x(0.4) * rt.scaling(0.8, 0.8, 0.8))
    marble = rt.Sphere.build(rt.translation(-0.8, 0.6, -2.2) * rt.scaling(0.6, 0.6, 0.6),
                             Material(color=(0.05, 0.05, 0.05), transparency=0.9, reflective=0.9, refractive_index=REFRACTION_GLASS,
                                      diffuse=0.1, ambient=0.05, shininess=300.0))
    floor = rt.Plane.build(rt.translation(0.0, -0.2, 0.0), Material(pattern=rt.Checkers((0.85, 0.85, 0.85), (0.25, 0.25, 0.3)),
                                                                    specular=0.0))
    camera = rt.Camera(width, height, PI / 3.0, rt.view_transform((0.0, 3.0, -6.5), (0, 1.2, 0), (0, 1, 0)))
    return camera, rt.World([floor, carved, marble], PointLight((-6.0, 9.0, -8.0), (1, 1, 1)))


def csg_chain(rt, width=320, height=200, n=40):
    """A glass union chain of n spheres along a helix (n - 1 nesting levels); every fifth sphere repeats the one before it,
    so equal distances from different leaves are common."""
    balls = []
    for i in range(n):
        k = i - 1 if i % 5 == 4 else i
        a = 0.45 * k
        balls.append(rt.Sphere.build(rt.translation(1.6 * math.cos(a), 0.5 + 0.06 * k, 1.6 * math.sin(a)) * rt.scaling(0.45, 0.45, 0.45),
                                     Material(color=(0.1, 0.15, 0.2), transparency=0.8, reflective=0.5,
                                              refractive_index=1.3 + 0.005 * i, diffuse=0.3, shininess=200.0)))
    chain = _union_chain(rt, balls)
    floor = rt.Plane.build(rt.identity_4x4(), Material(pattern=rt.Checkers((0.9, 0.9, 0.9), (0.2, 0.3, 0.2)), specular=0.0))
    camera = rt.Camera(width, height, PI / 3.0, rt.view_transform((0.0, 4.0, -6.0), (0, 1.2, 0), (0, 1, 0)))
    return camera, rt.World([floor, chain], PointLight((-5.0, 9.0, -6.0), (1, 1, 1)))


def synthetic_obj(n_u=48, n_v=24, smooth=False) -> str:
    """A deterministic 'teapot-class' mesh as OBJ text: a torus knot-ish bumpy tube, n_u * n_v quads written as
    4-vertex faces (fan-triangulated by the loader into 2 * n_u * n_v triangles)."""
    lines = []
    for i in range(n_u):
        t = 2 * math.pi * i / n_u
        # (2,3) torus knot centre line
        cx, cy, cz = (2 + math.cos(3 * t)) * math.cos(2 * t), math.sin(3 * t), (2 + math.cos(3 * t)) * math.sin(2 * t)
        dt = 1e-3
        t2 = t + dt
        nx = (2 + math.cos(3 * t2)) * math.cos(2 * t2) - cx
        ny = math.sin(3 * t2) - cy
        nz = (2 + math.cos(3 * t2)) * math.sin(2 * t2) - cz
        ln = math.sqrt(nx * nx + ny * ny + nz * nz)
        tx, ty, tz = nx / ln, ny / ln, nz / ln
        # frame: b1 = tangent x up, b2 = tangent x b1
        ux, uy, uz = 0.0, 1.0, 0.0
        b1 = (ty * uz - tz * uy, tz * ux - tx * uz, tx * uy - ty * ux)
        l1 = math.sqrt(sum(c * c for c in b1)) or 1.0
        b1 = tuple(c / l1 for c in b1)
        b2 = (ty * b1[2] - tz * b1[1], tz * b1[0] - tx * b1[2], tx * b1[1] - ty * b1[0])
        for j in range(n_v):
            a = 2 * math.pi * j / n_v
            r = 0.45 + 0.08 * math.sin(5 * a + 3 * t)
            x = cx + r * (math.cos(a) * b1[0] + math.sin(a) * b2[0])
            y = cy + r * (math.cos(a) * b1[1] + math.sin(a) * b2[1])
            z = cz + r * (math.cos(a) * b1[2] + math.sin(a) * b2[2])
            lines.append(f"v {x:.6f} {y:.6f} {z:.6f}")
    if smooth:
        for i in range(n_u * n_v):
            lines.append("vn 0 1 0")
    lines.append("g knot")
    for i in range(n_u):
        for j in range(n_v):
            a = i * n_v + j + 1
            b = ((i + 1) % n_u) * n_v + j + 1
            c = ((i + 1) % n_u) * n_v + (j + 1) % n_v + 1
            d = i * n_v + (j + 1) % n_v + 1
            if smooth:
                lines.append(f"f {a}//{a} {b}//{b} {c}//{c} {d}//{d}")
            else:
                lines.append(f"f {a} {b} {c} {d}")
    return "\n".join(lines) + "\n"


def dragon_element(rt, width=480, height=270, n_u=48, n_v=24, divide=4, case=True, smooth=False):
    """One display element of here_be_dragons.rs (get_scene_element :298-338) around a synthetic mesh."""
    mesh = rt.parse_obj(synthetic_obj(n_u, n_v, smooth))
    mesh.set_transformation(rt.translation(0.0, 0.69, 0.0))
    element = rt.GroupShape()
    element.set_transformation(rt.translation(0.0, 0.5, -4.0) * rt.rotation_y(PI))
    mesh.set_material(Material(color=(1, 0.5, 0.1), ambient=0.1, diffuse=0.6, specular=0.3, shininess=15.0))
    if case:
        display_case = rt.Cube()
        display_case.set_casts_shadow(False)
        display_case.set_transformation(rt.scaling(1.1, 0.77, 0.49) * rt.translation(0.0, 1.001, 0.0))
        display_case.set_material(Material(ambient=0.0, diffuse=0.2, specular=0.0, transparency=0.8))
        box = rt.GroupShape()
        box.add_child(mesh)
        box.add_child(display_case)
    else:
        box = mesh
    element.add_child(box)
    pedestal = rt.Cylinder()
    pedestal.maximum_y, pedestal.minimum_y, pedestal.closed = 0.0, -0.15, True
    pedestal.set_material(Material(color=(0.2, 0.2, 0.2), ambient=0.0, diffuse=0.8, specular=0.0, reflective=0.2))
    element.add_child(pedestal)
    if divide:
        element.divide(divide)
    floor = rt.Plane.build(rt.translation(0.0, 0.35, 0.0), Material(color=(0.6, 0.6, 0.65), specular=0.0, reflective=0.1))
    world = rt.World([element, floor], PointLight((-10, 100, -100), (1, 1, 1)))
    camera = rt.Camera(width, height, 1.2, rt.view_transform((0, 2.5, -10), (0, 1, 0), (0, 1, 0)))
    return camera, world


def here_be_dragons(rt, width=500, height=200, n_u=32, n_v=16):
    """demos/src/bin/here_be_dragons.rs:36-218: six display elements (transforms / materials :42-138, element builder
    :298-338 with divide(4), display case :242-250, pedestal :264-281, mesh lift :291) around clones of one mesh — a
    synthetic OBJ here, the demo reads an external dragon.obj."""
    def dragon_mat(color):
        return Material(color=color, ambient=0.1, diffuse=0.6, specular=0.3, shininess=15.0)

    def case_mat(diffuse, transparency):
        return Material(ambient=0.0, diffuse=diffuse, specular=0.0, transparency=transparency)

    elements = [  # (transform, dragon material, case material), in the demo's order :143-180
        (rt.translation(0.0, 0.5, -4.0) * rt.rotation_y(PI), dragon_mat((1, 1, 1)), None),
        (rt.translation(0.0, 2.0, 2.0), dragon_mat((1, 0, 0.1)), case_mat(0.4, 0.6)),
        (rt.translation(-2.0, 0.75, -1.0) * rt.rotation_y(-PI / 8.0) * rt.scaling(0.75, 0.75, 0.75), dragon_mat((0.9, 0.5, 0.1)),
         case_mat(0.2, 0.8)),
        (rt.translation(-4.0, 0.0, -2.0) * rt.rotation_y(-PI / 16.0) * rt.scaling(0.5, 0.5, 0.5), dragon_mat((1, 0.9, 0.1)),
         case_mat(0.1, 0.9)),
        (rt.translation(2.0, 1.0, -1.0) * rt.rotation_y(5.0 * PI / 4.0) * rt.scaling(0.75, 0.75, 0.75), dragon_mat((1, 0.5, 0.1)),
         case_mat(0.2, 0.8)),
        (rt.translation(4.0, 0.0, -2.0) * rt.rotation_y(21.0 * PI / 20.0) * rt.scaling(0.5, 0.5, 0.5), dragon_mat((0.9, 1, 0.1)),
         case_mat(0.1, 0.9)),
    ]
    dragon = rt.parse_obj(synthetic_obj(n_u, n_v))
    dragon.set_transformation(rt.translation(0.0, 0.69, 0.0))
    objects = []
    for i, (transform, d_mat, c_mat) in enumerate(elements):
        mesh = dragon.clone() if i + 1 < len(elements) else dragon
        element = rt.GroupShape()
        element.set_transformation(transform)
        mesh.set_material(d_mat)
        if c_mat is not None:
            case = rt.Cube()
            case.set_casts_shadow(False)
            case.set_transformation(rt.scaling(1.1, 0.77, 0.49) * rt.translation(0.0, 1.001, 0.0))
            case.set_material(c_mat)
            box = rt.GroupShape()
            box.add_child(mesh)
            box.add_child(case)
        else:
            box = mesh
        element.add_child(box)
        pedestal = rt.Cylinder()
        pedestal.maximum_y, pedestal.minimum_y, pedestal.closed = 0.0, -0.15, True
        pedestal.set_material(Material(color=(0.2, 0.2, 0.2), ambient=0.0, diffuse=0.8, specular=0.0, reflective=0.2))
        element.add_child(pedestal)
        element.divide(4)
        objects.append(element)
    world = rt.World(objects, PointLight((-10, 100, -100), (1, 1, 1)))
    camera = rt.Camera(width, height, 1.2, rt.view_transform((0, 2.5, -10), (0, 1, 0), (0, 1, 0)))
    return camera, world


def _xorshift64star(seed):
    state = seed & 0xFFFFFFFFFFFFFFFF

    def nxt():
        nonlocal state
        state ^= state >> 12
        state ^= (state << 25) & 0xFFFFFFFFFFFFFFFF
        state ^= state >> 27
        return ((state * 2685821657736338717) & 0xFFFFFFFFFFFFFFFF) / 2.0 ** 64

    return nxt


def stress(rt, width=3840, height=2160, n_spheres=100_000, n_each=64, n_csg=16, extent=50.0, divide=8, seed=1):
    """SURVEY.md §8d config 5: random sphere field + cylinders / cones / cubes + CSG + checker plane."""
    rnd = _xorshift64star(seed)
    plain = Material(color=(0.8, 0.6, 0.3), diffuse=0.8, specular=0.4, shininess=60.0)
    mirror = Material(color=(0.7, 0.7, 0.8), diffuse=0.5, reflective=0.5, shininess=100.0)
    glassy = Material(color=(0.05, 0.05, 0.05), diffuse=0.1, ambient=0.05, transparency=0.9, reflective=0.9,
                      refractive_index=REFRACTION_GLASS, shininess=300.0)
    field = rt.GroupShape()
    for i in range(n_spheres):
        cx, cy, cz = ((rnd() * 2 - 1) * extent for _ in range(3))
        r = 0.2 + 0.4 * rnd()
        m = glassy if i % 16 == 0 else (mirror if i % 8 == 1 else plain)
        field.add_child(rt.Sphere.build(rt.translation(cx, cy, cz) * rt.scaling(r, r, r), m))
    if divide:
        field.divide(divide)
    objects = [field]

    def placed():
        return (rt.translation((rnd() * 2 - 1) * extent * 0.5, (rnd() * 2 - 1) * extent * 0.5, (rnd() * 2 - 1) * extent * 0.5)
                * rt.rotation_y(rnd() * 2 * PI) * rt.rotation_x(rnd() * 2 * PI) * rt.scaling(1.5, 1.5, 1.5))

    for i in range(n_each):
        cyl = rt.Cylinder()
        cyl.minimum_y, cyl.maximum_y, cyl.closed = -1.0, 1.0, True
        cyl.set_transformation(placed())
        cyl.set_material(Material(color=(0.2, 0.7, 0.4), reflective=0.2))
        cone = rt.Cone()
        cone.minimum_y, cone.maximum_y, cone.closed = -1.0, 0.0, True
        cone.set_transformation(placed())
        cone.set_material(Material(color=(0.8, 0.3, 0.3)))
        cube = rt.Cube.build(placed(), Material(color=(0.3, 0.4, 0.9), reflective=0.3))
        objects += [cyl, cone, cube]
    for i in range(n_csg):
        kind = i % 3
        if kind == 0:
            a = rt.Sphere.build(rt.identity_4x4(), Material(color=(0.9, 0.8, 0.2)))
            b = rt.Cylinder()
            b.minimum_y, b.maximum_y, b.closed = -2.0, 2.0, True
            b.set_transformation(rt.scaling(0.5, 1.0, 0.5))
            b.set_material(Material(color=(0.9, 0.2, 0.2)))
            csg = rt.CSG(CSG_DIFFERENCE, a, b)
        elif kind == 1:
            csg = rt.CSG(CSG_INTERSECTION, rt.Cube.build(rt.identity_4x4(), Material(color=(0.2, 0.9, 0.9))),
                         rt.Sphere.build(rt.scaling(1.3, 1.3, 1.3), Material(color=(0.9, 0.2, 0.9))))
        else:
            csg = rt.CSG(CSG_UNION, rt.Sphere.build(rt.identity_4x4(), Material(color=(0.4, 0.9, 0.3))),
                         rt.Cube.build(rt.translation(0.8, 0.8, 0.0) * rt.scaling(0.6, 0.6, 0.6), Material(color=(0.9, 0.5, 0.1))))
        csg.set_transformation(placed())
        objects.append(csg)
    ground = rt.Plane.build(rt.translation(0.0, -extent - 1.0, 0.0),
                            Material(pattern=rt.Checkers((0.85, 0.85, 0.85), (0.25, 0.25, 0.25)), specular=0.0, reflective=0.1))
    objects.append(ground)
    world = rt.World(objects, PointLight((-extent * 2, extent * 3, -extent * 3), (1, 1, 1)))
    camera = rt.Camera(width, height, PI / 3.0,
                       rt.view_transform((0, extent * 0.4, -extent * 2.2), (0, 0, 0), (0, 1, 0)))
    return camera, world


def orbit_cameras(rt, camera, n, degrees=360.0, field_of_view=None):
    """`n` cameras of `camera`'s canvas size (a host session's camera) whose eyes turn about the vertical axis through the
    look-at point: the point of the camera's forward ray nearest that axis — the turntable of rtc_render_views.  View i is
    at i * degrees / n (view 0 is the camera's own eye); field_of_view defaults to the camera's."""
    inv = np.asarray(rt.camera_view(camera).transform_inverse, np.float64).reshape(4, 4)
    eye, fwd = inv[:3, 3], -inv[:3, 2]
    h2 = fwd[0] ** 2 + fwd[2] ** 2
    t = -(eye[0] * fwd[0] + eye[2] * fwd[2]) / h2 if h2 > 1e-12 else 1.0
    pivot = eye + t * fwd
    fov = camera.field_of_view if field_of_view is None else field_of_view
    out = []
    for i in range(n):
        a = math.radians(degrees * i / n)
        dx, dz = eye[0] - pivot[0], eye[2] - pivot[2]
        e = (pivot[0] + dx * math.cos(a) + dz * math.sin(a), eye[1], pivot[2] - dx * math.sin(a) + dz * math.cos(a))
        out.append(rt.Camera(camera.width_pixels, camera.height_pixels, fov,
                             rt.view_transform(tuple(float(c) for c in e), tuple(float(c) for c in pivot), (0, 1, 0))))
    return out
