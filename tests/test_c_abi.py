"""The drop-in boundary: every entry point declared in include/*.h is exported by the library that implements it
(loaded with ctypes — no compute calls, no GPU needed), and the product fails loudly without a device."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared(header, prefix):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(" + prefix + r"\w+)\s*\(", text)))


def test_device_library_exports_the_whole_c_abi():
    import ray_tracer_challenge_b200 as rt

    names = declared("rtc_b200.h", "rtc_")
    assert len(names) >= 20 and "rtc_render" in names and "rtc_scene_commit" in names
    lib = C.CDLL(rt.LIB_DEVICE)
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, f"librtc_b200.so lacks {missing}"


def test_host_library_exports_the_scene_api():
    import ray_tracer_challenge_b200 as rt

    names = declared("rtc_scene.h", "sg_")
    assert "sg_camera_render" in names and "sg_group_add_child" in names
    lib = C.CDLL(rt.LIB_HOST)
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, f"librtc_host.so lacks {missing}"


def test_oracle_exports_the_same_scene_api(oracle):
    names = declared("rtc_scene.h", "sg_")
    missing = [n for n in names if not hasattr(oracle.lib, n)]
    assert not missing, f"the oracle lacks {missing}"


def test_libraries_do_not_link_the_oracle():
    """The product must never route through the CPU oracle: neither library may depend on it."""
    import subprocess

    import ray_tracer_challenge_b200 as rt

    for lib in (rt.LIB_DEVICE, rt.LIB_HOST):
        out = subprocess.run(["ldd", lib], capture_output=True, text=True).stdout
        assert "oracle" not in out, out
        syms = subprocess.run(["nm", "-D", "--defined-only", lib], capture_output=True, text=True).stdout
        assert "orc_" not in syms


def test_shard_band_rule_matches_python_mirror():
    import ray_tracer_challenge_b200 as rt
    from ray_tracer_challenge_b200.sharding import BAND_ROWS, bands_of, rows_of

    lib = C.CDLL(rt.LIB_DEVICE)
    lib.rtc_shard_bands.argtypes = [C.c_uint32, C.c_int32, C.c_int32, C.POINTER(C.c_uint32)]
    for height in (1, 7, 8, 9, 77, 400, 2160):
        for n in (1, 2, 3, 8):
            seen = []
            for shard in range(n):
                buf = (C.c_uint32 * 512)()
                cnt = lib.rtc_shard_bands(height, shard, n, buf)
                assert cnt == len(bands_of(height, shard, n))
                assert [buf[i] for i in range(cnt)] == [b * BAND_ROWS for b in bands_of(height, shard, n)]
                for r in rows_of(height, shard, n):
                    seen.extend(r)
            assert sorted(seen) == list(range(height)), (height, n)  # every row exactly once
    assert lib.rtc_shard_bands(100, 2, 2, None) < 0  # bad shard index is an error, not a silent no-op


def test_no_device_is_a_loud_error():
    """Without a GPU the product refuses to render: there is no CPU fallback."""
    import ray_tracer_challenge_b200 as rt

    lib = C.CDLL(rt.LIB_DEVICE)
    if lib.rtc_device_count() > 0:
        pytest.skip("a CUDA device is present")
    session = rt.new_session()
    cam = session.Camera(8, 8, 1.0, session.identity_4x4())
    world = session.World.default()
    with pytest.raises(rt.RtcError):
        cam.render_b200(world, 1)
    with pytest.raises(rt.RtcError):
        cam.prepare(world)


def test_raw_c_abi_validates_scenes_without_a_device():
    """The C ABI driven the way a foreign host (the Rust -sys crate) drives it: plain structs in, error codes out.
    rtc_scene_inspect runs the host half of the commit, so bad references are reported without a GPU."""
    import ray_tracer_challenge_b200 as rt

    lib = C.CDLL(rt.LIB_DEVICE)
    lib.rtc_last_error.restype = C.c_char_p
    scene = C.c_void_p()
    assert lib.rtc_scene_create(C.byref(scene)) == 0
    ident = (C.c_float * 16)(1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1)
    lib.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
    assert lib.rtc_set_camera(scene, 64, 32, 1.0, 0.5, 2.0 / 64, ident) == 0
    info = rt.RtcCommitInfo()
    # no light yet: the reference's own failure (world.rs:66), as an error code
    assert lib.rtc_scene_inspect(scene, C.byref(info)) < 0 and b"World light should be set" in lib.rtc_last_error()
    pos, rgb = (C.c_float * 3)(-10, 10, -10), (C.c_float * 3)(1, 1, 1)
    assert lib.rtc_set_point_light(scene, pos, rgb) == 0

    class RtcMaterial(C.Structure):
        _fields_ = [("color", C.c_float * 3), ("v", C.c_float * 7), ("pattern", C.c_int32)]

    class RtcPattern(C.Structure):
        _fields_ = [("kind", C.c_int32), ("mapping", C.c_int32), ("uv", C.c_int32 * 6), ("inv", C.c_float * 16),
                    ("a", C.c_float * 3), ("b", C.c_float * 3)]

    class RtcUvPattern(C.Structure):
        _fields_ = [("kind", C.c_int32), ("params", C.c_float * 15)]

    class RtcTexture(C.Structure):
        _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("rgb", C.POINTER(C.c_float))]

    prim = rt.RtcPrim()
    prim.type, prim.material, prim.casts_shadow, prim.parent = 0, 0, 1, -1
    prim.inv[:] = list(ident)
    prim.bbox_min[:], prim.bbox_max[:] = [-1, -1, -1], [1, 1, 1]
    assert lib.rtc_set_primitives(scene, 1, C.byref(prim)) == 0
    mat = RtcMaterial()
    mat.color[:], mat.v[:], mat.pattern = [1, 1, 1], [0.1, 0.9, 0.9, 200.0, 0.0, 0.0, 1.0], 0
    assert lib.rtc_set_materials(scene, 1, C.byref(mat)) == 0
    pat = RtcPattern()
    pat.kind, pat.mapping = 6, 0  # RTC_PAT_TEXTURE_MAP, spherical
    pat.uv[:] = [0, -1, -1, -1, -1, -1]
    pat.inv[:] = list(ident)
    uv = RtcUvPattern()
    uv.kind = 2  # RTC_UV_IMAGE
    uv.params[0] = 3.0  # texture 3 of none
    assert lib.rtc_set_patterns(scene, 1, C.byref(pat), 1, C.byref(uv)) == 0
    assert lib.rtc_scene_inspect(scene, C.byref(info)) < 0 and b"texture" in lib.rtc_last_error()
    pixels = (C.c_float * 12)(*([0.5] * 12))
    tex = RtcTexture(2, 2, pixels)
    uv.params[0] = 0.0
    assert lib.rtc_set_patterns(scene, 1, C.byref(pat), 1, C.byref(uv)) == 0
    assert lib.rtc_set_textures(scene, 1, C.byref(tex)) == 0
    assert lib.rtc_scene_inspect(scene, C.byref(info)) == 0
    assert (info.small_n, info.n_positions, info.filter_ok, info.n_bvh_nodes) == (1, 1, 1, 0)
    mat.pattern = 5  # a pattern that does not exist
    assert lib.rtc_set_materials(scene, 1, C.byref(mat)) == 0
    assert lib.rtc_scene_inspect(scene, C.byref(info)) < 0
    if lib.rtc_device_count() == 0:
        assert lib.rtc_scene_commit(scene, 1, None) < 0 and b"no CPU fallback" in lib.rtc_last_error()
    lib.rtc_scene_destroy(scene)


def test_ctypes_mirrors_have_the_layout_of_the_header(tmp_path):
    """Every ctypes structure that crosses the C ABI has the size and the field offsets gcc gives the header's struct
    (the Rust `#[repr(C)]` mirrors in rust/rtc-b200-sys follow the same field lists)."""
    import shutil
    import subprocess

    import ray_tracer_challenge_b200 as rt

    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    mirrors = [getattr(rt, n) for n in ("RtcStats", "RtcCommitInfo", "RtcPrim", "RtcNode", "RtcMaterial", "RtcPattern",
                                        "RtcUvPattern", "RtcTexture") if hasattr(rt, n)]
    assert len(mirrors) >= 4
    from ray_tracer_challenge_b200.api import SgStats

    c_names = {m: m.__name__ for m in mirrors}
    mirrors.append(SgStats)  # include/rtc_scene.h
    c_names[SgStats] = "sg_stats"
    lines = []
    for m in mirrors:
        lines.append(f'printf("{m.__name__} %zu", sizeof({c_names[m]}));')
        for field, _ in m._fields_:
            c_field = "type" if field == "type_" else field
            lines.append(f'printf(" %zu", offsetof({c_names[m]}, {c_field}));')
        lines.append('printf("\\n");')
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "rtc_b200.h"\n#include "rtc_scene.h"\nint main(void) {\n'
                   + "\n".join(lines) + "\nreturn 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    for m, line in zip(mirrors, out):
        name, size, *offsets = line.split()
        assert name == m.__name__
        assert int(size) == C.sizeof(m), (name, size, C.sizeof(m))
        assert [int(o) for o in offsets] == [getattr(m, f).offset for f, _ in m._fields_], name


def _raw_scene(lib, rt):
    """A scene handle with a camera, a point light and one default material — through the raw C ABI."""
    ident = (C.c_float * 16)(1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1)
    lib.rtc_last_error.restype = C.c_char_p
    lib.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
    scene = C.c_void_p()
    assert lib.rtc_scene_create(C.byref(scene)) == 0
    assert lib.rtc_set_camera(scene, 64, 32, 1.0, 0.5, 2.0 / 64, ident) == 0
    pos, rgb = (C.c_float * 3)(-10, 10, -10), (C.c_float * 3)(1, 1, 1)
    assert lib.rtc_set_point_light(scene, pos, rgb) == 0

    class RtcMaterial(C.Structure):
        _fields_ = [("color", C.c_float * 3), ("v", C.c_float * 7), ("pattern", C.c_int32)]

    mat = RtcMaterial()
    mat.color[:], mat.v[:], mat.pattern = [1, 1, 1], [0.1, 0.9, 0.9, 200.0, 0.0, 0.0, 1.0], -1
    assert lib.rtc_set_materials(scene, 1, C.byref(mat)) == 0
    return scene, ident


def _sphere(rt, ident, centre=(0.0, 0.0, 0.0), parent=-1):
    p = rt.RtcPrim()
    p.type, p.material, p.casts_shadow, p.parent = 0, 0, 1, parent
    p.inv[:] = list(ident)
    p.inv[3], p.inv[7], p.inv[11] = -centre[0], -centre[1], -centre[2]
    p.bbox_min[:] = [c - 1 for c in centre]
    p.bbox_max[:] = [c + 1 for c in centre]
    return p


def test_node_graph_must_be_a_forest():
    """ADVICE r1: parent cycles (A -> B -> A) would spin the device's cull-chain walk, reference cycles would recurse
    the CSG emitter; links that disagree are rejected too.  All without a device (rtc_scene_inspect)."""
    import ray_tracer_challenge_b200 as rt

    lib = C.CDLL(rt.LIB_DEVICE)
    scene, ident = _raw_scene(lib, rt)
    info = rt.RtcCommitInfo()
    lib.rtc_set_nodes.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(rt.RtcNode), C.c_uint32, C.POINTER(C.c_int32)]

    def group(parent, begin, count):
        n = rt.RtcNode()
        n.kind, n.parent, n.op, n.child_begin, n.child_count = 0, parent, 0, begin, count
        n.inv[:] = list(ident)
        n.bbox_min[:], n.bbox_max[:] = [-1, -1, -1], [1, 1, 1]
        n.world_bbox_min[:], n.world_bbox_max[:] = [-1, -1, -1], [1, 1, 1]
        return n

    def inspect(prims, nodes, refs):
        pa = (rt.RtcPrim * len(prims))(*prims)
        na = (rt.RtcNode * len(nodes))(*nodes)
        ra = (C.c_int32 * max(len(refs), 1))(*refs)
        assert lib.rtc_set_primitives(scene, len(prims), pa) == 0
        assert lib.rtc_set_nodes(scene, len(nodes), na, len(refs), ra) == 0
        rc = lib.rtc_scene_inspect(scene, C.byref(info))
        return rc, lib.rtc_last_error()

    # a well-formed group of one sphere
    rc, _ = inspect([_sphere(rt, ident, parent=0)], [group(-1, 0, 1)], [0])
    assert rc == 0
    # A's parent is B and B's parent is A; each lists the other as its child
    rc, msg = inspect([_sphere(rt, ident)], [group(1, 0, 1), group(0, 1, 1)], [~1, ~0])
    assert rc == -1 and b"cycle" in msg
    # the sphere says its parent is node 0, but node 0 does not list it
    rc, msg = inspect([_sphere(rt, ident, parent=0)], [group(-1, 0, 0)], [])
    assert rc == -1 and b"child list" in msg
    # node 0 lists the sphere, but the sphere claims no parent
    rc, msg = inspect([_sphere(rt, ident, parent=-1)], [group(-1, 0, 1)], [0])
    assert rc == -1 and b"point back" in msg
    # the same child twice
    rc, msg = inspect([_sphere(rt, ident, parent=0)], [group(-1, 0, 2)], [0, 0])
    assert rc == -1 and b"twice" in msg
    lib.rtc_scene_destroy(scene)


def test_jitter_table_that_does_not_divide_the_draws_is_rejected():
    """ADVICE r1: the reference's table closure carries its cursor across intensity_at calls (test/utils.rs); restarting
    it per call is the same thing only when the table length divides 2 * u_steps * v_steps."""
    import ray_tracer_challenge_b200 as rt

    lib = C.CDLL(rt.LIB_DEVICE)
    scene, _ = _raw_scene(lib, rt)
    v3 = lambda *a: (C.c_float * 3)(*a)
    lib.rtc_set_rect_light.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int32,
                                       C.POINTER(C.c_float), C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_uint32,
                                       C.c_uint64]
    table5 = (C.c_float * 5)(0.7, 0.3, 0.9, 0.1, 0.5)
    args = (v3(1, 1, 1), v3(0, 0, 0), v3(1, 0, 0))
    # 2 * 4 * 4 = 32 draws: 5 does not divide them, 4 and 32 do; 10 x 10 cells = 200 draws: 5 does
    assert lib.rtc_set_rect_light(scene, *args, 4, v3(0, 1, 0), 4, v3(0.5, 0.5, 0), table5, 5, 0) == -1
    assert b"does not divide" in lib.rtc_last_error()
    assert lib.rtc_set_rect_light(scene, *args, 4, v3(0, 1, 0), 4, v3(0.5, 0.5, 0), table5, 4, 0) == 0
    assert lib.rtc_set_rect_light(scene, *args, 10, v3(0, 1, 0), 10, v3(0.5, 0.5, 0), table5, 5, 0) == 0
    assert lib.rtc_set_rect_light(scene, *args, 4, v3(0, 1, 0), 4, v3(0.5, 0.5, 0), None, 0, 7) == 0  # counter mode
    lib.rtc_scene_destroy(scene)


@pytest.mark.parametrize("layout", ["coincident", "geometric", "line"])
def test_bvh_depth_is_bounded_for_degenerate_scenes(layout):
    """VERDICT r1 weak #2: the traversal stack (48 entries) must never be asked to hold more than the builder allows.
    10^5 spheres with one centroid, with geometrically shrinking spacing (SAH peels one sphere per level) and on a line:
    the tree stays below the cap, without a device."""
    import numpy as np

    import ray_tracer_challenge_b200 as rt

    lib = C.CDLL(rt.LIB_DEVICE)
    scene, ident = _raw_scene(lib, rt)
    n = 100_000
    prims = (rt.RtcPrim * n)()
    base = _sphere(rt, ident)
    for i in range(n):
        C.memmove(C.byref(prims[i]), C.byref(base), C.sizeof(rt.RtcPrim))
    if layout != "coincident":
        xs = np.cumsum(2.0 ** -np.arange(n, dtype=np.float64).clip(max=100)) * 1e3 if layout == "geometric" else np.arange(n) * 2.5
        arr = np.ctypeslib.as_array(C.cast(prims, C.POINTER(C.c_float)), shape=(n, C.sizeof(rt.RtcPrim) // 4))
        inv_off, lo_off, hi_off = rt.RtcPrim.inv.offset // 4, rt.RtcPrim.bbox_min.offset // 4, rt.RtcPrim.bbox_max.offset // 4
        arr[:, inv_off + 3] = -xs
        arr[:, lo_off] = xs - 1
        arr[:, hi_off] = xs + 1
    assert lib.rtc_set_primitives(scene, n, prims) == 0
    info = rt.RtcCommitInfo()
    assert lib.rtc_scene_inspect(scene, C.byref(info)) == 0, lib.rtc_last_error()
    assert info.n_bvh_nodes >= n // 16 and 17 <= info.bvh_depth <= 47, info.bvh_depth
    lib.rtc_scene_destroy(scene)


def test_rust_sys_crate_mirrors_the_header(tmp_path):
    """The `#[repr(C)]` structs of rust/rtc-b200-sys/src/lib.rs (not compilable here: no Rust toolchain) declare the same
    fields, in the same order, with the same element types and array lengths, as include/rtc_b200.h — and every
    `rtc_*` function of the header is declared in the crate's `extern "C"` block."""
    header = open(os.path.join(ROOT, "include", "rtc_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    rust = open(os.path.join(ROOT, "rust", "rtc-b200-sys", "src", "lib.rs")).read()
    rust = re.sub(r"//[^\n]*", "", rust)
    c_to_rust = {"int32_t": "i32", "uint32_t": "u32", "uint64_t": "u64", "int64_t": "i64", "float": "f32", "double": "f64",
                 "const float*": "*const f32"}

    def c_fields(body):
        out = []
        for decl in body.split(";"):
            decl = " ".join(decl.split())
            if not decl:
                continue
            m = re.match(r"(const float\s*\*|\w+)\s*(.*)", decl)
            ctype = "const float*" if m.group(1).startswith("const") else m.group(1)
            for name in m.group(2).split(","):
                name = name.strip()
                arr = re.match(r"(\w+)\[(\d+)\]", name)
                out.append((arr.group(1), f"[{c_to_rust[ctype]}; {arr.group(2)}]") if arr else (name, c_to_rust[ctype]))
        return out

    def rust_fields(body):
        out = []
        for name, ty in re.findall(r"pub\s+(\w+)\s*:\s*([^,\n]+)", body):
            out.append((name[2:] if name.startswith("r#") else name, ty.strip()))
        return out

    structs = re.findall(r"typedef struct (\w+) \{(.*?)\} \1;", header, flags=re.S)
    assert {n for n, _ in structs} >= {"RtcPrim", "RtcNode", "RtcMaterial", "RtcPattern", "RtcUvPattern", "RtcTexture", "RtcStats",
                                      "RtcCommitInfo"}
    for name, body in structs:
        m = re.search(r"#\[repr\(C\)\][^{]*pub struct " + name + r"\s*\{(.*?)\n\}", rust, flags=re.S)
        assert m, f"rtc-b200-sys lacks #[repr(C)] struct {name}"
        want, got = c_fields(body), rust_fields(m.group(1))
        want = [("type_" if f == "type" else f, t) for f, t in want]
        got = [("type_" if f in ("type", "type_", "kind_") and False else f, t) for f, t in got]
        assert [t for _, t in got] == [t for _, t in want], (name, got, want)
        assert [f.rstrip("_") for f, _ in got] == [f.rstrip("_") for f, _ in want], (name, got, want)
    for fn in declared("rtc_b200.h", "rtc_"):
        assert re.search(r"pub fn " + fn + r"\s*\(", rust), f"rtc-b200-sys lacks `{fn}`"
    for const in re.findall(r"\b(RTC_[A-Z0-9_]+)\s*=\s*(-?\d+)", header):
        m = re.search(r"pub const " + const[0] + r"\s*:\s*\w+\s*=\s*(-?\d+)", rust)
        assert m and m.group(1) == const[1], f"rtc-b200-sys: constant {const[0]} missing or different"


def test_rust_glue_covers_every_implementer_and_only_uses_what_the_sys_crate_declares():
    """rust/lib_patch/render_b200.rs (not compilable here) lowers EVERY Shape / Pattern / UVPattern / UVMapping / Light
    implementer of the reference, and every `sys::` item it names is declared by rust/rtc-b200-sys.  The lists below are
    held to the reference's own census of its implementers, stored in tests/golden/reference_implementers.json."""
    import json

    glue = open(os.path.join(ROOT, "rust", "lib_patch", "render_b200.rs")).read()
    sys_crate = open(os.path.join(ROOT, "rust", "rtc-b200-sys", "src", "lib.rs")).read()
    expected = {
        "flatten": {"Sphere", "Plane", "Cube", "Cylinder", "Cone", "Triangle", "SmoothTriangle", "GroupShape", "CSG", "TestShape", "BaseShape"},
        "lower": {"Stripes", "Gradient", "Rings", "Checkers", "Sine2D", "TestPattern", "TextureMap", "CubicMap", "BasePattern",
                  "PointLight", "RectangleLight"},
        "lower_uv": {"UVCheckers", "AlignCheck", "UVImage"},
        "mapping_id": {"SphericalMap", "PlanarMap", "CylindricalMap"},
    }
    with open(os.path.join(ROOT, "tests", "golden", "reference_implementers.json")) as fh:
        found = {trait: set(names) for trait, names in json.load(fh)["implementers"].items()}
    assert found["Shape"] == expected["flatten"], found["Shape"] ^ expected["flatten"]
    assert found["Pattern"] | found["Light"] == expected["lower"], (found["Pattern"] | found["Light"]) ^ expected["lower"]
    assert found["UVPattern"] == expected["lower_uv"] and found["UVMapping"] == expected["mapping_id"]
    for method, types in expected.items():
        for t in types:
            body = re.search(r"impl " + t + r"(?:<'_>)? \{(.*?)\n\}", glue, flags=re.S)
            assert body and re.search(r"fn " + method + r"\(", body.group(1)), f"render_b200.rs: `{t}` lacks `{method}`"
    declared_names = set(re.findall(r"pub (?:const|fn|struct) (\w+)", sys_crate))
    used = set(re.findall(r"\bsys::(\w+)", glue))
    assert used and used <= declared_names, used - declared_names
    # field names used in struct literals exist in the sys crate's structs
    for struct, body in re.findall(r"sys::(Rtc\w+) \{(.*?)\}", glue, flags=re.S):
        decl = re.search(r"pub struct " + struct + r"\s*\{(.*?)\n\}", sys_crate, flags=re.S).group(1)
        fields = set(re.findall(r"pub (\w+)\s*:", decl))
        for name in re.findall(r"(?:^|,|\{)\s*(\w+)\s*(?::|,|$)", body):
            if name in ("if", "else", "sys", "self", "unsafe"):
                continue
            assert name in fields or not name.islower() or name in ("w", "h", "px"), (struct, name, fields)


def test_mapped_arrays_commit_like_copied_ones():
    """rtc_map_primitives / rtc_map_nodes hand out the scene's own storage: records written in place give the commit
    plan (digest included) that rtc_set_primitives / rtc_set_nodes give for the same records."""
    import ray_tracer_challenge_b200 as rt

    lib = C.CDLL(rt.LIB_DEVICE)
    lib.rtc_set_primitives.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(rt.RtcPrim)]
    lib.rtc_set_nodes.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(rt.RtcNode), C.c_uint32, C.POINTER(C.c_int32)]
    lib.rtc_map_primitives.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.POINTER(rt.RtcPrim))]
    lib.rtc_map_nodes.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.POINTER(rt.RtcNode)), C.POINTER(C.POINTER(C.c_int32))]

    def records(ident):
        prims = [_sphere(rt, ident, centre=(3.0 * i, 0.0, 5.0), parent=0 if i < 3 else -1) for i in range(40)]
        node = rt.RtcNode()
        node.kind, node.parent, node.op, node.child_begin, node.child_count = 0, -1, 0, 0, 3
        node.inv[:] = list(ident)
        node.bbox_min[:], node.bbox_max[:] = [-1, -1, 4], [7, 1, 6]
        node.world_bbox_min[:], node.world_bbox_max[:] = [-1, -1, 4], [7, 1, 6]
        return prims, [node], [0, 1, 2]

    digests = []
    for mapped in (False, True):
        scene, ident = _raw_scene(lib, rt)
        prims, nodes, refs = records(ident)
        if mapped:
            pp, pn, pr = C.POINTER(rt.RtcPrim)(), C.POINTER(rt.RtcNode)(), C.POINTER(C.c_int32)()
            assert lib.rtc_map_primitives(scene, len(prims), C.byref(pp)) == 0
            assert lib.rtc_map_nodes(scene, len(nodes), len(refs), C.byref(pn), C.byref(pr)) == 0
            for i, p in enumerate(prims):
                pp[i] = p
            for i, n in enumerate(nodes):
                pn[i] = n
            for i, r in enumerate(refs):
                pr[i] = r
        else:
            assert lib.rtc_set_primitives(scene, len(prims), (rt.RtcPrim * len(prims))(*prims)) == 0
            assert lib.rtc_set_nodes(scene, len(nodes), (rt.RtcNode * len(nodes))(*nodes), len(refs), (C.c_int32 * len(refs))(*refs)) == 0
        info = rt.RtcCommitInfo()
        assert lib.rtc_scene_inspect(scene, C.byref(info)) == 0, lib.rtc_last_error()
        digests.append((info.digest, info.n_positions, info.n_bvh_nodes))
        lib.rtc_scene_destroy(scene)
    assert digests[0] == digests[1] and digests[0][1] == 40
    assert lib.rtc_map_primitives(None, 1, None) != 0
