"""CPU tests of the C-ABI library: loads, exports every declared symbol, generates and compiles the
sm_100a program of every config scene (NVRTC needs no GPU), attributes compile errors to the owning
scene element, and refuses -- loudly -- to render without a CUDA device (no CPU fallback exists)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, SCENES, load_ir
from portal_b200 import capi
from portal_b200.capi import PeTarget, PortalB200Error
from portal_b200.renderer import SceneRenderer, camera_scale, orbit_camera_matrix


def _declared():
    text = open(os.path.join(ROOT, "include", "portal_b200.h")).read() + open(os.path.join(ROOT, "include", "portal_b200_host.h")).read()
    return sorted(set(re.findall(r"PE_API\s+[\w\s\*]+?\b(p[eh]_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = capi.lib()
    declared = _declared()
    assert len(declared) >= 55
    out = subprocess.run(["nm", "-D", "--defined-only", capi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (p[eh]_[a-z0-9_]+)", out))
    assert set(declared) <= exported, sorted(set(declared) - exported)
    assert exported <= set(declared), f"exported but undeclared: {sorted(exported - set(declared))}"
    for name in declared:
        assert getattr(lib, name)
    assert lib.pe_abi_version() == 102      # 1.02: + pe_frames_differ, pe_autotune's bit guard (1.01: pe_sharder_*, anaglyph uniforms, tile_w)


def test_library_is_built_for_sm_100a():
    out = subprocess.run(["cuobjdump", "-lelf", capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


@pytest.mark.parametrize("scene", SCENES)
@pytest.mark.parametrize("persistent", [False, True])
def test_scene_program_compiles_for_sm_100a(scene, persistent, tmp_path):
    r = SceneRenderer(load_ir(scene), device=-1, persistent=persistent)
    src = r.source()
    assert "pe_render_kernel" in src and "__constant__" in src
    assert "!FOR_NUMBER!" not in src
    cubin = r.cubin()
    assert cubin[:4] == b"\x7fELF" and len(cubin) > 10000
    path = str(tmp_path / f"{scene}_{int(persistent)}.cubin")
    open(path, "wb").write(cubin)
    res = subprocess.run(["cuobjdump", "-res-usage", path], capture_output=True, text=True).stdout
    assert "pe_render_kernel" in res
    m = re.search(r"REG:(\d+) STACK:(\d+)", res)
    assert m and int(m.group(1)) <= 255
    r.close()


def test_int_uniforms_are_specialisation_constants():
    ir = load_ir("portal_in_portal")
    r = SceneRenderer(ir, device=-1)
    s1 = r.source()
    assert "#define show_teleported_u (10)" in s1 and "#define _ray_tracing_depth (PE_C.i[" in s1
    r.set_uniform("show_teleported_u", 3)
    r.compile()
    assert "#define show_teleported_u (3)" in r.source()
    r2 = SceneRenderer(ir, device=-1, specialize_ints=False)
    assert "#define show_teleported_u (PE_C.i[" in r2.source()


def test_compile_error_is_attributed_to_the_scene_element():
    ir = load_ir("monoportal")
    ir["objects"][6]["code"] = "float q = 1.0;\nreturn undefined_function_zzz(x);\n"
    with pytest.raises(PortalB200Error) as e:
        SceneRenderer(ir, device=-1)
    msg = str(e.value)
    assert "object `monoportal` is_inside(2)" in msg and "undefined_function_zzz" in msg


def test_unknown_uniform_and_frozen_scene_are_errors():
    r = SceneRenderer(load_ir("monoportal"), device=-1)
    with pytest.raises(PortalB200Error, match="unknown float uniform"):
        r.set_uniform("no_such_u", 1.0)
    lib = capi.lib()
    assert lib.pe_scene_add_library(r._ctx, b"x", b"float f() { return 1.; }") != 0
    assert b"frozen" in lib.pe_last_error(r._ctx)


def test_render_without_gpu_fails_loudly():
    """There is no CPU rendering path: every entry point that would touch the device says so on a compile-only context."""
    import ctypes as C
    r = SceneRenderer(load_ir("monoportal"), device=-1)
    with pytest.raises(PortalB200Error, match="no CUDA device"):
        r.render_host(16, 16)
    lib, ctx, t = r._lib, r._ctx, r.full_target(16, 16)
    buf = (C.c_uint8 * (16 * 16 * 16))()
    tk, vp = C.c_uint64(), C.c_void_p()
    calls = {
        "pe_render": lambda: lib.pe_render(ctx, C.byref(t), C.addressof(buf), None, None),
        "pe_render_rgba8": lambda: lib.pe_render_rgba8(ctx, C.byref(t), C.addressof(buf), None),
        "pe_render_host_rgba8": lambda: lib.pe_render_host_rgba8(ctx, C.byref(t), C.addressof(buf)),
        "pe_submit_host_rgba8": lambda: lib.pe_submit_host_rgba8(ctx, C.byref(t), C.addressof(buf), C.byref(tk)),
        "pe_submit_host_strips_rgba8": lambda: lib.pe_submit_host_strips_rgba8(ctx, C.byref(t), C.addressof(buf), C.byref(tk)),
        "pe_host_malloc": lambda: lib.pe_host_malloc(ctx, 64, C.byref(vp)),
        "pe_host_register": lambda: lib.pe_host_register(ctx, C.addressof(buf), 4096),
        "pe_device_malloc": lambda: lib.pe_device_malloc(ctx, 64, C.byref(vp)),
        "pe_sync": lambda: lib.pe_sync(ctx),
    }
    for name, call in calls.items():
        assert call() != 0, name
        assert b"no CPU rendering path" in lib.pe_last_error(ctx), name
    assert lib.pe_wait_host(ctx, 1) != 0 and b"unknown ticket" in lib.pe_last_error(ctx)
    a = (C.c_float * 3)(0, 0, 0)
    o, h1, h2, h3 = (C.c_float * 3)(), C.c_int32(), C.c_int32(), C.c_int32()
    assert lib.pe_probe_ray(ctx, a, a, o, C.byref(h1), C.byref(h2), C.byref(h3)) != 0


def test_strip_targets_partition_the_frame():
    for h, s, world in [(2160, 16, 8), (1080, 16, 8), (90, 16, 4), (4320, 16, 8), (17, 16, 8), (256, 8, 3)]:
        rows = []
        for rank in range(world):
            t = SceneRenderer.strip_target(64, h, s, rank, world)
            for k in range(t.n_strips):
                g = t.strip_first + k * t.strip_step
                rows += [y for y in range(g * s, (g + 1) * s) if y < h]
        assert sorted(rows) == list(range(h))


def test_orbit_camera_matches_oracle_frontend():
    from oracle import frontend
    ir = load_ir("portal_in_portal")
    cam = ir["cam"]
    m = orbit_camera_matrix(cam["look_at"], cam["alpha"], cam["beta"], cam["r"])
    assert np.allclose(m, np.array(ir["camera_matrix"]), rtol=0, atol=1e-15)
    assert camera_scale(m) == pytest.approx(ir["camera_scale"], abs=1e-15)
    cols = frontend.orbit_camera_matrix(cam["look_at"], cam["alpha"] + 0.3, cam["beta"], cam["r"])
    m2 = orbit_camera_matrix(cam["look_at"], cam["alpha"] + 0.3, cam["beta"], cam["r"])
    assert np.allclose(m2, np.array([x for c in cols for x in c]), rtol=0, atol=1e-15)


def _build_c_example(tmp_path):
    exe = str(tmp_path / "render_frame_c")
    libdir = os.path.dirname(capi.LIB_PATH)
    cc = subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                         os.path.join(ROOT, "examples", "render_frame.c"), "-L", libdir, "-lportal_b200", f"-Wl,-rpath,{libdir}", "-o", exe],
                        capture_output=True, text=True)
    assert cc.returncode == 0, cc.stderr
    return exe


def test_headers_are_c11_and_a_plain_c_caller_links(tmp_path):
    """The boundary is a C ABI: both headers are valid ISO C11, and examples/render_frame.c (no C++, no Python) links
    against the library, compiles a scene for sm_100a and -- without a GPU -- is refused loudly at the render call."""
    for h in ("portal_b200.h", "portal_b200_host.h"):
        src = tmp_path / f"inc_{h}.c"
        src.write_text(f'#include "{h}"\nint main(void) {{ return 0; }}\n')
        cc = subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)],
                            capture_output=True, text=True)
        assert cc.returncode == 0, cc.stderr
    exe = _build_c_example(tmp_path)
    run = subprocess.run([exe, os.path.join(ROOT, "tests", "fixtures", "two_spheres.ron"), str(tmp_path / "o.ppm"), "64", "36", "8", "-1"],
                         capture_output=True, text=True, timeout=300)
    assert run.returncode == 3 and "no CPU rendering path" in run.stderr
    assert "bytes of sm_100a code for 10 objects" in run.stdout


def test_adaptive_despecialisation_bounds_recompiles():
    """An int uniform that keeps changing between renders (an animation driving it) is a specialisation constant for the
    first four changes and a constant-block read from then on; "adaptive" 0 keeps the old behaviour; a rebuilt scene starts
    afresh."""
    ir = load_ir("portal_in_portal")
    r = SceneRenderer(ir, device=-1)
    seen = []
    for v in range(1, 9):
        r.set_uniform("show_teleported_u", v)
        r.uniform_block(64, 36)                       # selects the variant exactly as a render would
        seen.append(re.search(r"#define show_teleported_u (.*)", r.source()).group(1))
    assert seen[:4] == ["(1)", "(2)", "(3)", "(4)"] and all(s.startswith("(PE_C.i[") for s in seen[4:])
    assert "#define teleport_light_u (1)" in r.source()          # the others stay baked in
    r2 = SceneRenderer(ir, device=-1, options={"adaptive": 0})
    for v in range(1, 9):
        r2.set_uniform("show_teleported_u", v)
        r2.uniform_block(64, 36)
    assert "#define show_teleported_u (8)" in r2.source()


def test_bulk_matrix_upload_equals_individual_uploads():
    """pe_set_uniforms_mat4 (n names, 16n floats) == n x pe_set_uniform_mat4, observed through pe_scene_uniform_block;
    an unknown name is reported with code 2 and leaves the others applied, like the single call."""
    ir = load_ir("monoportal")
    names = [k for k, u in ir["uniforms"].items() if u["type"] == "mat4"][:4]
    rng = np.random.default_rng(3)
    vals = rng.standard_normal((len(names), 16)).astype(np.float32)
    a = SceneRenderer(ir, device=-1)
    for n, v in zip(names, vals):
        a._check(a._lib.pe_set_uniform_mat4(a._ctx, n.encode(), v.ctypes.data_as(C.POINTER(C.c_float))))
    b = SceneRenderer(ir, device=-1)
    arr = (C.c_char_p * len(names))(*[n.encode() for n in names])
    flat = np.ascontiguousarray(vals.reshape(-1))
    b._check(b._lib.pe_set_uniforms_mat4(b._ctx, len(names), arr, flat.ctypes.data_as(C.POINTER(C.c_float))))

    def block(r):
        p, n = C.c_void_p(), C.c_size_t()
        r._check(r._lib.pe_scene_uniform_block(r._ctx, 64, 36, C.byref(p), C.byref(n)))
        return C.string_at(p, n.value)
    assert block(a) == block(b) and flat.tobytes()[:64] in block(b)
    arr2 = (C.c_char_p * 2)(names[0].encode(), b"no_such_mat")
    assert b._lib.pe_set_uniforms_mat4(b._ctx, 2, arr2, flat.ctypes.data_as(C.POINTER(C.c_float))) == 2
    assert b"no_such_mat" in b._lib.pe_last_error(b._ctx)


def test_uniform_block_symbol_and_smem_variant(tmp_path):
    """The host finds the uniform block by symbol name after loading the cubin: the name it looks up must be a constant-space
    symbol of exactly the block's size in the cubin -- in the default program (`PE_C`) and in the shared-memory-staging
    variant (`PE_C_UPLOAD`, with `PE_C` a shared image)."""
    ir = load_ir("portal_in_portal")
    for opts, symbol in (({}, "PE_C"), ({"uniforms_in_smem": 1}, "PE_C_UPLOAD")):
        r = SceneRenderer(ir, device=-1, options=opts)
        size = int(re.search(r"sizeof\(PeConstBlock\) == (\d+)", r.source()).group(1))
        assert len(r.uniform_block(64, 36)) == size
        path = str(tmp_path / f"symbol_{symbol}.cubin")
        open(path, "wb").write(r.cubin())
        ptx_like = subprocess.run(["cuobjdump", "-elf", path], capture_output=True, text=True).stdout
        rows = [ln for ln in ptx_like.splitlines() if re.search(rf"\b{symbol}$", ln.strip())]
        assert rows, symbol
        assert any(f"0x{size:x}" in ln for ln in rows), (symbol, rows)
        res = subprocess.run(["cuobjdump", "-res-usage", path], capture_output=True, text=True).stdout
        shared = int(re.search(r"SHARED:(\d+)", res).group(1))
        assert (shared >= size) == bool(opts)


def test_target_validation():
    """pe_target fields are validated before anything is launched or allocated: garbage never reaches the device, and every
    target the repo's own code builds (full frames, cyclic strips of any rank / world, ragged and tiny frames) is accepted
    (on this compile-only context "accepted" shows as the no-GPU error instead of the invalid-target one)."""
    import random
    r = SceneRenderer(load_ir("basics"), device=-1)
    buf = (C.c_uint8 * 64)()

    def verdict(t):
        assert r._lib.pe_render_rgba8(r._ctx, C.byref(t), C.addressof(buf), None) != 0
        return "invalid" if b"invalid pe_target" in r._lib.pe_last_error(r._ctx) else "valid"
    rng = random.Random(5)
    vals = [0, 1, -1, 2, 16, 17, 255, 4096, 65536, 65537, 2 ** 31 - 1, -2 ** 31, 7680, 4320]
    seen = set()
    for _ in range(5000):
        t = PeTarget(*[rng.choice(vals) for _ in range(7)])
        v = verdict(t)
        seen.add(v)
        if v == "valid":
            assert 0 < t.width <= 65536 and 0 < t.height <= 65536 and t.n_strips * t.strip_rows <= 2 ** 24
    assert seen == {"invalid", "valid"}
    for w, h in [(1, 1), (1, 37), (37, 1), (5, 3), (256, 256), (3840, 2160), (7680, 4320), (65536, 8)]:
        assert verdict(SceneRenderer.full_target(w, h)) == "valid"
        for world in (1, 2, 3, 8):
            for rank in range(world):
                t = SceneRenderer.strip_target(w, h, 16, rank, world)
                assert verdict(t) == "valid", (w, h, rank, world)      # a rank that owns no strip (n_strips == 0) renders nothing
    assert verdict(PeTarget(64, 64, 16, 0, 1, -1, 0)) == "invalid"
    assert verdict(PeTarget(2 ** 31 - 1, 2 ** 31 - 1, 1, 0, 1, 1, 1)) == "invalid"
    assert verdict(PeTarget(64, 64, 65536, 65535, 65536, 65536, 0)) == "invalid"


def test_option_validation():
    """pe_set_option rejects unknown keys and launch geometries the kernel cannot index (a block is a column of 64-thread warp
    pairs), with a message; accepted values survive a compile."""
    r = SceneRenderer(load_ir("basics"), device=-1, compile_now=False)
    for bad in (0, 32, 96, 1088, -64):
        assert r._lib.pe_set_option(r._ctx, b"block_threads", bad) != 0
        assert b"block_threads" in r._lib.pe_last_error(r._ctx)
    assert r._lib.pe_set_option(r._ctx, b"no_such_option", 1) != 0
    assert b"no_such_option" in r._lib.pe_last_error(r._ctx)
    for good in (64, 128, 512, 1024):
        assert r._lib.pe_set_option(r._ctx, b"block_threads", good) == 0
    assert r._lib.pe_set_option(r._ctx, b"block_threads", 128) == 0 and r._lib.pe_set_option(r._ctx, b"min_blocks", 4) == 0
    assert r._lib.pe_scene_compile(r._ctx) == 0, r._lib.pe_last_error(r._ctx)
