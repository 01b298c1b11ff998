"""The C++ host front-end (RON reader, fasteval-style formulas, glam-style matrix DAG, orbit camera --
portal_b200/csrc/host, C API include/portal_b200_host.h) against the oracle's independent Python
restatement (oracle/frontend.py), and -- on the GPU -- the whole path .ron -> pixels."""
import glob
import math
import os

import numpy as np
import pytest

from conftest import ROOT, SCENES, load_ir
from portal_b200 import capi
from portal_b200.capi import PortalB200Error
from portal_b200.host import HostRenderer, HostScene

FIXTURE = os.path.join(ROOT, "tests", "fixtures", "two_spheres.ron")


def _oracle_ir(path, name, time=0.0):
    from oracle import frontend
    return frontend.scene_ir(frontend.load_scene(path), name, time=time)


def _assert_same_table(table, ir):
    assert list(table) == list(ir["uniforms"])           # same names, same upload order
    for k, (typ, v) in table.items():
        u = ir["uniforms"][k]
        assert typ == u["type"], k
        assert np.array_equal(np.asarray(v, dtype=np.float64), np.asarray(u["value"], dtype=np.float64), equal_nan=True), k


def test_fixture_scene_table_matches_oracle_frontend():
    hs = HostScene.from_file(FIXTURE)
    ir = _oracle_ir(FIXTURE, "two_spheres")
    _assert_same_table(hs.uniform_table(), ir)
    assert hs.camera() == ir["cam"]
    assert hs.counts() == {"objects": 10, "materials": 7, "intersection_materials": 1, "library": 2, "textures": 0, "videos": 0}
    t = hs.uniform_table()
    assert t["steps_u"] == ("int", 7) and t["open_u"] == ("int", 1)
    assert t["lift_u"][1] == 0.5 + 0.25 * 2 + -(math.sin(0.6) * (1 / 4))
    # If(open) picks portal_a; Inv is the inverse; Teleport = second * first^-1 * what
    assert t["chosen_mat"] == t["portal_a_mat"] and t["ball_inv_mat"] == t["ball_mat_inv"]
    assert "portal_a_to_portal_b_mat_teleport" in t and "portal_b_to_portal_a_mat_teleport" in t
    assert "between_mat" in t and "between_q_mat" in t             # Lerp matrices
    # TrefoilSpecial: 18 packed ints value + 10000 * enabled + 1000 * colour (scene.rs:488-492, 644-650); -1 inside formulas
    assert "knot_u" not in t and [t[f"ts_{i}_knot_u"][1] for i in (0, 1, 2, 17)] == [0, 10005 + 1000, 10010 + 2000, 10013 + 2000]
    assert t["knot_as_number_u"] == ("float", -2.0)


def test_set_value_and_time_reevaluate():
    hs = HostScene.from_file(FIXTURE)
    hs.set_value("open", 0)
    hs.set_value("p", 0.75)
    t = hs.uniform_table()
    assert t["open_u"] == ("int", 0) and t["chosen_mat"] == t["portal_b_mat"]
    assert t["lift_u"][1] == 0.5 + 0.75 * 2 + -(math.sin(0.6) * (1 / 4))
    with pytest.raises(PortalB200Error):
        hs.set_value("lift", 1.0)          # formulas are not settable
    with pytest.raises(PortalB200Error):
        hs.set_value("nope", 1.0)


def test_animation_stages():
    """Scene::init_stage for animation stages (scene.rs:1180-1200): C++ host vs the oracle front-end."""
    from oracle import frontend
    assert HostScene.from_file(FIXTURE).stage_names() == ["closed", "reset"]
    for stage in ("closed", "reset"):
        hs = HostScene.from_file(FIXTURE)
        hs.init_stage(stage)
        sc = frontend.load_scene(FIXTURE)
        ir = frontend.scene_ir(sc, "two_spheres", stage=stage)
        _assert_same_table(hs.uniform_table(), ir)
    hs = HostScene.from_file(FIXTURE)
    base = hs.uniform_table()
    hs.init_stage("closed")
    t = hs.uniform_table()
    assert t["open_u"] == ("int", 0) and t["p_u"] == ("float", 0.75) and t["count_u"] == ("int", 5) and t["spin_u"] == ("float", 0.2)
    assert t["portal_a_mat"] != base["portal_a_mat"] and t["chosen_mat"] == t["portal_b_mat"]     # If(open) now picks portal_b
    assert t["ball_mat"] != base["ball_mat"]                                                      # FromDev -> dev-stage matrix
    hs.init_stage("reset")
    assert hs.uniform_table()["p_u"] == ("float", 0.4)
    with pytest.raises(PortalB200Error, match="no stage named"):
        hs.init_stage("nope")


def test_every_stage_of_the_config_scenes_matches_oracle_frontend(reference):
    from oracle import frontend
    n = 0
    for scene in SCENES:
        path = f"{reference}/scenes/{scene}.ron"
        for stage in HostScene.from_file(path).stage_names():
            hs = HostScene.from_file(path)
            hs.init_stage(stage)
            ir = frontend.scene_ir(frontend.load_scene(path), scene, stage=stage)
            _assert_same_table(hs.uniform_table(), ir)
            n += 1
    assert n == 44


LERP_SCENES = ("half_spheres", "portal_in_portal_cone", "teleportation_degrees", "portal_in_portal_plus_ultra")


def test_lerp_matrix_stages_match_oracle_frontend(reference):
    """Matrix::Lerp (matrix.rs:614-628) only appears in animation stages of four reference scenes;
    every stage at three times: C++ host == oracle front-end, value for value."""
    from oracle import frontend
    n = 0
    for scene in LERP_SCENES:
        path = f"{reference}/scenes/{scene}.ron"
        sc = frontend.load_scene(path)
        hs = HostScene.from_file(path)
        hs.set_formula_camera()
        for stage in hs.stage_names():
            hs.init_stage(stage)
            for tm in (0.0, 0.3, 1.0):
                hs.set_time(tm)
                _assert_same_table(hs.uniform_table(), frontend.scene_ir(sc, scene, time=tm, stage=stage))
                n += 1
    assert n == 22 * 3


def test_lerp_matrix_properties():
    """t=0 / t=1 reproduce the endpoints (to ~1 ulp through the quaternion round trip), mirrored input
    (negative determinant) keeps its handedness, and the nlerp takes the short arc."""
    from oracle import frontend as F
    a = F.srt_matrix([2.0, 2.0, 2.0], [0.3, -0.2, 1.0], [1.0, 2.0, 3.0])
    b = F.srt_matrix([-1.0, 1.0, 1.0], [0.0, 2.5, 0.1], [0.0, 0.0, -1.0])
    for m, t in ((a, 0.0), (b, 1.0)):
        got = F.mat_lerp(a, b, t)
        assert np.allclose(np.asarray(got), np.asarray(m), atol=1e-14)
    assert F.mat_determinant(b) < 0 and F.mat_to_scale_rotation_translation(b)[0][0] < 0
    mid = F.mat_lerp(a, a, 0.5)
    assert np.allclose(np.asarray(mid), np.asarray(a), atol=1e-14)
    q = F.quat_lerp((0.0, 0.0, 0.0, 1.0), (0.0, 0.0, 0.0, -1.0), 0.5)     # antipodal -> same rotation
    assert q == (0.0, 0.0, 0.0, 1.0)


def test_bad_scene_files_are_errors():
    with pytest.raises(PortalB200Error, match="RON parse error"):
        HostScene("(cam: (")
    with pytest.raises(PortalB200Error, match="uniforms"):
        HostScene("(cam: (look_at: (0,0,0), alpha: 0, beta: 1, r: 1, offset_after_material: 0.1))")


def test_camera_functions():
    import ctypes as C
    lib = capi.lib()
    ir = load_ir("mobius_monoportal")
    cam = ir["cam"]
    out = (C.c_double * 16)()
    lib.ph_orbit_camera_matrix((C.c_double * 3)(*cam["look_at"]), cam["alpha"], cam["beta"], cam["r"], out)
    assert list(out) == ir["camera_matrix"]
    assert lib.ph_camera_scale(out) == ir["camera_scale"]


def test_program_from_host_scene_compiles():
    r = HostRenderer(HostScene.from_file(FIXTURE), device=-1)
    src = r.source()
    assert "sphere_hit" in src and "#define steps_u (7)" in src and "float& t" in src
    assert "intersection material `floating_disk`" in src


@pytest.mark.parametrize("scene", SCENES)
def test_config_scene_tables_match_oracle_and_golden(scene, reference):
    hs = HostScene.from_file(f"{reference}/scenes/{scene}.ron")
    _assert_same_table(hs.uniform_table(), load_ir(scene))          # committed golden (oracle front-end output)
    if scene in ("triple_portal", "portal_in_portal"):             # use_time scenes: `time` reaches the formulas
        hs.set_time(0.37)
        _assert_same_table(hs.uniform_table(), _oracle_ir(f"{reference}/scenes/{scene}.ron", scene, time=0.37))


def test_every_reference_scene_loads_and_evaluates(reference):
    from oracle import frontend
    n_ok = 0
    for path in sorted(glob.glob(f"{reference}/scenes/*.ron")):
        name = os.path.basename(path)[:-4]
        if name == "empty":
            continue
        hs = HostScene.from_file(path)
        hs.set_formula_camera()                                    # the `Camera` matrix kind = the renderer's camera
        ir = frontend.scene_ir(frontend.load_scene(path), name)
        table = hs.uniform_table()
        common = [k for k in table if k in ir["uniforms"]]
        assert len(common) >= 0.9 * len(ir["uniforms"]), name
        for k in common:
            assert np.array_equal(np.asarray(table[k][1], dtype=np.float64),
                                  np.asarray(ir["uniforms"][k]["value"], dtype=np.float64), equal_nan=True), (name, k)
        n_ok += 1
    assert n_ok >= 80


@pytest.mark.gpu
def test_ron_to_pixels_matches_oracle():
    from oracle import runner
    ir = _oracle_ir(FIXTURE, "two_spheres")
    ref = runner.Oracle(ir, "fast").render(480, 270, 12)
    for persistent in (False, True):
        r = HostRenderer(HostScene.from_file(FIXTURE), device=0, persistent=persistent)
        img = r.render_frame(480, 270, 12)
        assert np.array_equal(img.view(np.uint32), ref.view(np.uint32))
        q = r.render_frame(480, 270, 12, rgba8=True)
        assert np.array_equal(q, np.rint(np.clip(img, 0, 1) * 255).astype(np.uint8))
    cam = dict(ir["cam"], alpha=ir["cam"]["alpha"] + 1.0)
    from portal_b200.renderer import camera_scale, orbit_camera_matrix
    m = orbit_camera_matrix(cam["look_at"], cam["alpha"], cam["beta"], cam["r"])
    ref2 = runner.Oracle(ir, "fast").render(320, 180, 12, camera=m, camera_scale=camera_scale(m), aa_count=2)
    img2 = HostRenderer(HostScene.from_file(FIXTURE), device=0).render_frame(320, 180, 12, aa_count=2, camera=cam)
    assert np.array_equal(img2.view(np.uint32), ref2.view(np.uint32))


@pytest.mark.gpu
def test_motion_blur_frame_matches_reference_pipeline():
    """render_animation's inner loop (main.rs:1789-1817): sub-frame times, aa_start = j, RGBA8 readback,
    average_images -- the oracle side composes it from oracle frames + a numpy restatement of the average."""
    from oracle import frontend, runner
    w, h, depth, count, mb, dur, i = 192, 108, 12, 24, 4, 6.0, 5
    hs = HostScene.from_file(FIXTURE)
    got = HostRenderer(hs, device=0).render_motion_blur_frame(w, h, depth, i, count, mb, dur)
    subs = []
    for j in range(mb):
        t = (i / count + j / mb / count * 0.5) * dur
        ir = frontend.scene_ir(frontend.load_scene(FIXTURE), "two_spheres", time=t)
        f = runner.Oracle(ir, "fast").render(w, h, depth, aa_start=j)
        subs.append(np.rint(np.clip(f, 0, 1) * 255.0).astype(np.uint8))
    acc = (np.stack(subs)[..., :3].astype(np.uint32) ** 2).sum(axis=0) // mb
    want = np.concatenate([(np.sqrt(acc.astype(np.float32)) + np.float32(0.5)).astype(np.uint8), np.full((h, w, 1), 255, np.uint8)], axis=-1)
    assert np.array_equal(got, want)
    assert not np.array_equal(subs[0], subs[-1])        # time really moves the scene between sub-frames


@pytest.mark.gpu
def test_stage_to_pixels():
    from oracle import frontend, runner
    hs = HostScene.from_file(FIXTURE)
    hs.init_stage("closed")
    img = HostRenderer(hs, device=0).render_frame(320, 180, 12)
    ir = frontend.scene_ir(frontend.load_scene(FIXTURE), "two_spheres", stage="closed")
    ref = runner.Oracle(ir, "fast").render(320, 180, 12)
    assert np.array_equal(img.view(np.uint32), ref.view(np.uint32))
    base = HostRenderer(HostScene.from_file(FIXTURE), device=0).render_frame(320, 180, 12)
    assert not np.array_equal(img, base)


@pytest.mark.gpu
def test_render_frame_cli(tmp_path):
    """The C++ command-line mirror of `portal render-frame` (no Python in the loop)."""
    import subprocess
    out = tmp_path / "f.rgba"
    exe = os.path.join(ROOT, "portal_b200", "portal_b200_render")
    p = subprocess.run([exe, "render-frame", FIXTURE, "--width", "160", "--height", "90", "--render-depth", "12", "--output", str(out)],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr
    got = np.frombuffer(out.read_bytes(), dtype=np.uint8).reshape(90, 160, 4)
    want = HostRenderer(HostScene.from_file(FIXTURE), device=0).render_frame(160, 90, 12, rgba8=True)
    assert np.array_equal(got, want)


def _random_formulas(n, seed):
    """Expressions over the grammar both formula evaluators implement (fasteval 0.2.4 as the reference uses it,
    uniform.rs:602-635, 1009-1140): numbers in several spellings, + - * / % ^, comparisons, and / or (both spellings), unary
    minus and !, parentheses, one- and many-argument built-ins, the application's own functions, other uniforms, `time`."""
    import random
    rng = random.Random(seed)
    nums = ["0", "1", "2", "3.5", ".25", "1e-3", "2.5E2", "10", "0.1", "7", "1e10", "0.333"]
    names = ["time", "p", "spin", "count", "room_size", "pi()", "e()"]
    f1 = ["sin", "cos", "tan", "abs", "floor", "ceil", "int", "sign", "asin", "acos", "atan", "sinh", "cosh", "tanh", "deg2rad", "rad2deg",
          "easing_in", "easing_out", "easing_in_out", "easing_in_out_fast", "easing_plus_minus", "easing_elastic_out", "not", "round", "log"]
    fn = ["min", "max"]
    ops = ["+", "-", "*", "/", "%", "^", "<", "<=", ">", ">=", "==", "!=", "&&", "||", " and ", " or "]

    def expr(d):
        k = rng.random()
        if d <= 0 or k < 0.25:
            return rng.choice(nums) if rng.random() < 0.6 else rng.choice(names)
        if k < 0.60:
            return f"{expr(d - 1)}{rng.choice(ops)}{expr(d - 1)}"
        if k < 0.70:
            return f"({expr(d - 1)})"
        if k < 0.76:
            return f"-{expr(d - 1)}"
        if k < 0.79:
            return f"!{expr(d - 1)}"
        if k < 0.90:
            return f"{rng.choice(f1)}({expr(d - 1)})"
        if k < 0.94:
            return f"{rng.choice(fn)}({', '.join(expr(d - 1) for _ in range(rng.randint(1, 4)))})"
        if k < 0.97:
            return f"if({expr(d - 1)}, {expr(d - 1)}, {expr(d - 1)})"
        return f"lerp({expr(d - 1)}, {expr(d - 1)}, {expr(d - 1)})" if rng.random() < 0.5 else f"log({expr(d - 1)}, {expr(d - 1)})"
    return [expr(4) for _ in range(n)]


def test_formula_evaluators_agree_on_random_expressions(tmp_path):
    """Differential fuzz of the two fasteval restatements (C++ ph_formula.cpp vs oracle/formula.py), through both RON readers:
    1500 random expressions as Formula uniforms of the fixture scene; same set of evaluable uniforms, same float64 bits."""
    from oracle import frontend
    exprs = _random_formulas(1500, seed=20260923)
    text = open(FIXTURE, encoding="utf-8").read()
    marker = '        (name: "wobble", data: Formula(('
    assert marker in text
    extra = "".join(f'        (name: "fz{i}", data: Formula(("{e}"))),\n' for i, e in enumerate(exprs))
    text = text.replace(marker, extra + marker, 1)
    path = tmp_path / "fuzz.ron"
    path.write_text(text, encoding="utf-8")
    s = frontend.load_scene(str(path))
    hs = HostScene.from_file(str(path))
    n_val = n_nan = 0
    for tm in (0.0, 0.37):
        s.time = s.total_time = tm
        hs.set_time(tm)
        want, got = s.uniform_table(), hs.uniform_table()
        assert list(want) == list(got)                              # the same expressions are (un)evaluable on both sides
        for i, e in enumerate(exprs):
            k = f"fz{i}_u"
            if k in want:
                a, b = float(want[k][1]), float(got[k][1])
                assert np.array_equal(np.float64(a).view(np.uint64), np.float64(b).view(np.uint64)) or (math.isnan(a) and math.isnan(b)), (e, a, b)
                n_val += 1
                n_nan += math.isnan(a)
    assert n_val >= 2000 and n_nan < n_val // 2


def _random_matrix_scene(n, seed):
    """RON text of the fixture scene with n extra named matrices of every kind, built on each other at random."""
    import random
    rng = random.Random(seed)

    def num():
        k = rng.random()
        if k < 0.12:
            return rng.choice(["0.0", "1.0", "-1.0", "0.5", "2.0", "-0.0"])
        if k < 0.17:
            return rng.choice(["1e-9", "1e9", "3.0e-5"])
        return repr(round(rng.uniform(-3.0, 3.0), rng.choice([1, 3, 6])))

    names = ["origin", "portal_a", "portal_b", "ball"]

    def ref():
        return f'Some(Named("{rng.choice(names)}"))'

    def val():
        return f"Value({num()})" if rng.random() < 0.8 else rng.choice(['Uniform(Some(Named("p")))', 'Uniform(Some(Named("spin")))',
                                                                       'Uniform(Some(Inline(Formula(("lift * 0.5 - time")))))'])

    def vec3(keys="xyz"):
        return "(" + ", ".join(f"{c}: {val()}" for c in keys) + ")"

    out = []
    for i in range(n):
        kind = rng.choice(["Simple", "Parametrized", "Mul", "Teleport", "Inv", "Lerp", "If", "Exact", "ExactFull", "Sqrt"])
        if kind == "Simple":
            d = (f"Simple(offset: ({num()}, {num()}, {num()}), scale: {num()}, rotate: ({num()}, {num()}, {num()}), "
                 f"mirror: ({rng.choice(['true', 'false'])}, {rng.choice(['true', 'false'])}, {rng.choice(['true', 'false'])}))")
        elif kind == "Parametrized":
            d = f"Parametrized(offset: {vec3()}, rotate: {vec3()}, mirror: {vec3()}, scale: {val()})"
        elif kind == "Mul":
            d = f"Mul(to: {ref()}, what: {ref()})"
        elif kind == "Teleport":
            d = f"Teleport(first_portal: {ref()}, second_portal: {ref()}, what: {ref()})"
        elif kind == "Inv":
            d = f"Inv({ref()})"
        elif kind == "Sqrt":
            d = f"Sqrt({ref()})"
        elif kind == "Lerp":
            d = f"Lerp(t: {val()}, first: {ref()}, second: {ref()})"
        elif kind == "If":
            d = f"If(condition: {val()}, then: {ref()}, otherwise: {ref()})"
        elif kind == "Exact":
            d = f"Exact(i: {vec3()}, j: {vec3()}, k: {vec3()}, pos: {vec3()})"
        else:
            d = "ExactFull(" + ", ".join(f"c{c}: {vec3('xyzw')}" for c in range(4)) + ")"
        out.append(f'        (name: "mz{i}", data: {d}),\n')
        names.append(f"mz{i}")
    text = open(FIXTURE, encoding="utf-8").read()
    marker = '        (name: "ball_inv", data: Inv(Some(Named("ball")))),\n'
    assert marker in text
    return text.replace(marker, marker + "".join(out), 1)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_matrix_evaluators_agree_on_random_matrix_dags(seed, tmp_path):
    """Differential fuzz of the two glam restatements (C++ ph_scene.cpp vs oracle/frontend.py): 300 random matrices of every
    kind stacked on each other -- scale 0, mirrors, singular inverses, Lerp between mirrored frames, Teleport chains, Sqrt (the
    BFGS minimisation: found on both sides or on neither) -- must give identical float64 tables (M and M^-1 of every matrix),
    NaN / Inf patterns included."""
    from oracle import frontend
    path = tmp_path / "mat.ron"
    path.write_text(_random_matrix_scene(300, seed), encoding="utf-8")
    s = frontend.load_scene(str(path))
    hs = HostScene.from_file(str(path))
    for tm in (0.0, 0.6):
        s.time = s.total_time = tm
        hs.set_time(tm)
        want, got = s.uniform_table(), hs.uniform_table()
        assert list(want) == list(got)
        n = nonfinite = 0
        for k in want:
            a, b = np.asarray(want[k][1], dtype=np.float64), np.asarray(got[k][1], dtype=np.float64)
            same = (a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))
            assert same.all(), (k, a, b)
            if k.startswith("mz"):
                n += 1
                nonfinite += int(not np.isfinite(a).all())
        assert n >= 400 and 0 < nonfinite < n


def test_matrix_kinds_known_answers(tmp_path):
    """Conventions of the matrix kinds, by hand (matrix.rs:510-631): rotation order Rx*Ry*Rz in radians, scale before rotation
    before offset; Mul{to, what} = what * to; Teleport = second * first^-1 * what; Inv; If on > 0.5; Lerp endpoints.  Both
    front-ends, checked on what they do to a point."""
    from oracle import frontend
    hp = "1.5707963267948966"
    text = open(FIXTURE, encoding="utf-8").read()
    marker = '        (name: "ball_inv", data: Inv(Some(Named("ball")))),\n'

    def simple(off, scale="1.0", rot="0.0, 0.0, 0.0"):
        return f"Simple(offset: ({off}), scale: {scale}, rotate: ({rot}), mirror: (false, false, false))"
    extra = [
        ("k_srt", simple("1.0, 2.0, 3.0", "2.0", f"0.0, 0.0, {hp}")),
        ("k_xz", simple("0.0, 0.0, 0.0", "1.0", f"{hp}, 0.0, {hp}")),
        ("k_x", simple("0.0, 0.0, 0.0", "1.0", f"{hp}, 0.0, 0.0")), ("k_y", simple("0.0, 0.0, 0.0", "1.0", f"0.0, {hp}, 0.0")),
        ("k_t1", simple("1.0, 0.0, 0.0")), ("k_s2", simple("0.0, 0.0, 0.0", "2.0")),
        ("k_mul", 'Mul(to: Some(Named("k_t1")), what: Some(Named("k_s2")))'),
        ("k_first", simple("0.0, 0.0, 1.0")), ("k_second", simple("0.0, 5.0, 0.0", "1.0", f"0.0, 0.0, {hp}")), ("k_what", simple("1.0, 0.0, 1.0")),
        ("k_tp", 'Teleport(first_portal: Some(Named("k_first")), second_portal: Some(Named("k_second")), what: Some(Named("k_what")))'),
        ("k_inv", 'Inv(Some(Named("k_srt")))'),
        ("k_if1", 'If(condition: Value(0.51), then: Some(Named("k_t1")), otherwise: Some(Named("k_s2")))'),
        ("k_if0", 'If(condition: Value(0.5), then: Some(Named("k_t1")), otherwise: Some(Named("k_s2")))'),
        ("k_l0", 'Lerp(t: Value(0.0), first: Some(Named("k_srt")), second: Some(Named("k_second")))'),
        ("k_l1", 'Lerp(t: Value(1.0), first: Some(Named("k_srt")), second: Some(Named("k_second")))'),
        ("k_lh", 'Lerp(t: Value(0.5), first: Some(Named("k_t1")), second: Some(Named("k_what")))'),
    ]
    path = tmp_path / "kinds.ron"
    path.write_text(text.replace(marker, marker + "".join(f'        (name: "{n}", data: {d}),\n' for n, d in extra), 1), encoding="utf-8")
    for table in (frontend.load_scene(str(path)).uniform_table(), HostScene.from_file(str(path)).uniform_table()):
        def at(name, p):
            m = np.asarray(table[f"{name}_mat"][1], dtype=np.float64).reshape(4, 4).T
            return (m @ np.array([*p, 1.0]))[:3]
        near = lambda got, want: np.testing.assert_allclose(got, want, atol=1e-12)       # noqa: E731
        near(at("k_srt", (1, 0, 0)), (1, 4, 3))            # scale 2, quarter turn about z: (1,0,0) -> (0,2,0), + offset
        near(at("k_srt", (0, 0, 1)), (1, 2, 5))
        near(at("k_xz", (1, 0, 0)), (0, 0, 1))             # Rx*Ry*Rz: z-turn first (x -> y), then x-turn (y -> z)
        near(at("k_x", (0, 1, 0)), (0, 0, 1))              # right-handed quarter turns: about x, y -> z
        near(at("k_y", (0, 0, 1)), (1, 0, 0))              # about y, z -> x
        near(at("k_mul", (0, 0, 0)), (2, 0, 0))            # what * to = S(2) T(1,0,0)
        near(at("k_tp", (0, 0, 0)), (0, 6, 0))             # (1,0,1) -> first^-1 -> (1,0,0) -> quarter turn (0,1,0) + (0,5,0)
        near(at("k_inv", (1, 4, 3)), (1, 0, 0))
        near(at("k_if1", (0, 0, 0)), (1, 0, 0))            # condition > 0.5 -> then
        near(at("k_if0", (1, 1, 1)), (2, 2, 2))            # 0.5 is not > 0.5 -> otherwise
        near(at("k_l0", (1, 1, 1)), at("k_srt", (1, 1, 1)))
        near(at("k_l1", (1, 1, 1)), at("k_second", (1, 1, 1)))
        near(at("k_lh", (0, 0, 0)), (1, 0, 0.5))           # translations interpolate linearly
        inv = np.asarray(table["k_srt_mat_inv"][1], dtype=np.float64).reshape(4, 4).T
        near((inv @ np.array([1, 4, 3, 1.0]))[:3], (1, 0, 0))


def test_sqrt_matrices(tmp_path):
    """Matrix kind `Sqrt` (matrix.rs:606-613, 909-985; oracle/mat_sqrt.py, ph_matsqrt.cpp): known answers -- the case the one
    reference scene that uses the kind evaluates (portal_in_portal_plus_ultra.ron:961: b0 = scale 0.81 + offset -0.95 along z ->
    scale 0.9, offset -0.5), a quarter turn -> an eighth turn, the identity -> itself; X*X reproduces M; a mirror has no real
    root: the matrix and everything built on it is missing on both sides, as in the reference; C++ and oracle agree bit for bit."""
    from oracle import frontend
    text = open(FIXTURE, encoding="utf-8").read()
    marker = '        (name: "ball_inv", data: Inv(Some(Named("ball")))),\n'
    assert marker in text
    extra = [
        ('sq_b0', 'Simple(offset: (0.0, 0.0, -0.95), scale: 0.81, rotate: (0.0, 0.0, 0.0), mirror: (false, false, false))'),
        ('sq_turn', 'Simple(offset: (0.0, 0.0, 0.0), scale: 1.0, rotate: (0.0, 0.0, 0.25), mirror: (false, false, false))'),
        ('sq_id', 'Simple(offset: (0.0, 0.0, 0.0), scale: 1.0, rotate: (0.0, 0.0, 0.0), mirror: (false, false, false))'),
        ('sq_mirror', 'Simple(offset: (0.0, 0.0, 0.0), scale: 1.0, rotate: (0.0, 0.0, 0.0), mirror: (true, false, false))'),
        ('sq_eighth', 'Simple(offset: (0.0, 0.0, 0.0), scale: 1.0, rotate: (0.0, 0.0, 0.125), mirror: (false, false, false))'),
        ('r_b0', 'Sqrt(Some(Named("sq_b0")))'), ('r_turn', 'Sqrt(Some(Named("sq_turn")))'), ('r_id', 'Sqrt(Some(Named("sq_id")))'),
        ('r_mirror', 'Sqrt(Some(Named("sq_mirror")))'), ('on_mirror', 'Mul(to: Some(Named("r_mirror")), what: Some(Named("sq_id")))'),
        ('r_b0_squared', 'Mul(to: Some(Named("r_b0")), what: Some(Named("r_b0")))'),
    ]
    path = tmp_path / "sqrt.ron"
    path.write_text(text.replace(marker, marker + "".join(f'        (name: "{n}", data: {d}),\n' for n, d in extra), 1), encoding="utf-8")
    want = frontend.load_scene(str(path)).uniform_table()
    got = HostScene.from_file(str(path)).uniform_table()
    assert list(want) == list(got)
    for k in want:
        a, b = np.asarray(want[k][1], dtype=np.float64), np.asarray(got[k][1], dtype=np.float64)
        assert ((a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))).all(), k

    def m(name):
        return np.asarray(got[f"{name}_mat"][1], dtype=np.float64).reshape(4, 4).T          # column-major -> [row][col]
    assert "r_mirror_mat" not in got and "on_mirror_mat" not in got and "r_mirror_mat_inv" not in got
    np.testing.assert_allclose(m("r_b0"), np.array([[.9, 0, 0, 0], [0, .9, 0, 0], [0, 0, .9, -.5], [0, 0, 0, 1]]), atol=1e-8)
    np.testing.assert_allclose(m("r_id"), np.eye(4), atol=0)
    np.testing.assert_allclose(m("r_turn"), m("sq_eighth"), atol=1e-7)
    np.testing.assert_allclose(m("r_b0_squared"), m("sq_b0"), atol=1e-8)
    np.testing.assert_allclose(m("r_turn") @ m("r_turn"), m("sq_turn"), atol=1e-7)


def test_garbage_formulas_and_mutated_scene_files_are_handled(tmp_path):
    """Robustness of the host front-end on hostile input: (1) 2000 random character strings as formulas -- the C++ evaluator and
    the oracle's accept exactly the same ones, with the same values; (2) 400 random mutations of the fixture scene file --
    every one is either rejected with a message or loads and evaluates; nothing crashes."""
    import random
    from oracle import frontend
    rng = random.Random(7)
    alphabet = "0123456789.+-*/%^()<>=!&|, eEpixyzsincotafbrmlgud_[]"
    exprs = ["".join(rng.choice(alphabet) for _ in range(rng.randint(1, 24))) for _ in range(2000)]
    text = open(FIXTURE, encoding="utf-8").read()
    marker = '        (name: "wobble", data: Formula(('
    path = tmp_path / "garbage.ron"
    path.write_text(text.replace(marker, "".join(f'        (name: "gz{i}", data: Formula(("{e}"))),\n' for i, e in enumerate(exprs)) + marker, 1),
                    encoding="utf-8")
    want = frontend.load_scene(str(path)).uniform_table()
    got = HostScene.from_file(str(path)).uniform_table()
    assert list(want) == list(got)
    evaluable = [k for k in want if k.startswith("gz")]
    assert 5 < len(evaluable) < 200
    for k in evaluable:
        a, b = float(want[k][1]), float(got[k][1])
        assert np.float64(a).view(np.uint64) == np.float64(b).view(np.uint64) or (math.isnan(a) and math.isnan(b)), (k, a, b)
    loaded = rejected = 0
    for _ in range(400):
        t = list(text)
        for _ in range(rng.randint(1, 6)):
            k, pos = rng.random(), rng.randrange(len(t))
            if k < 0.3:
                del t[pos:pos + rng.randint(1, 40)]
            elif k < 0.6:
                t[pos:pos] = rng.choice(["(", ")", "[", "]", "{", "}", ",", ":", '"', "Some(", "None", "-", "1e999", chr(92), "'", "/*", "//", "nan", "(((("])
            elif k < 0.8:
                t[pos] = rng.choice("()[]{},:' 0123456789abcxyz._-" + chr(34) + chr(10))
            else:
                t = t[:pos] or ["("]
        try:
            hs = HostScene("".join(t))
            hs.uniform_table()
            loaded += 1
        except PortalB200Error as e:
            assert str(e)
            rejected += 1
    assert loaded + rejected == 400 and rejected > 300


def test_vendored_config_scenes_are_the_references_files(reference):
    """tests/golden/ron/*.ron -- the scene files bench.py and the GPU tests feed to the product's own front-end -- are byte
    copies of the reference's."""
    files = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "ron", "*.ron")))
    assert len(files) == 5
    for f in files:
        with open(f, "rb") as a, open(os.path.join(reference, "scenes", os.path.basename(f)), "rb") as b:
            assert a.read() == b.read(), f
