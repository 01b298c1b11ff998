"""CPU tests of the oracle itself: it must reproduce its own committed pins and the hand-derived
known answers of SURVEY.md Appendix A.  (The reference has no tests, golden images or known-answer
vectors for this path -- SURVEY.md §4 -- so these pins are this repo's: "parity unpinned" upstream.)"""
import hashlib
import math
import os

import numpy as np
import pytest

from conftest import DEPTH, GOLDEN, SCENES, load_ir, load_tex
from oracle import formula, frontend, gen_oracle, ron, runner


def test_ron_subset():
    v = ron.loads('(a: 1, b: [1.5, -2e3], c: Some("x\\ny"), d: None, e: Foo(x: true), f: Bar, g: r#"q"uote"#, h: {"k": (1, 2)})')
    assert v["a"] == 1 and v["b"] == [1.5, -2000.0] and v["c"] == "x\ny" and v["d"] is None
    assert v["e"].tag == "Foo" and v["e"].value == {"x": True}
    assert v["f"].tag == "Bar" and v["f"].value is None
    assert v["g"] == 'q"uote' and v["h"] == {"k": [1, 2]}
    with pytest.raises(ron.RonError):
        ron.loads("(a: 1")


def _ev(text, **vars_):
    def ns(name, args):
        if name == "deg2rad":
            return args[0] / 180.0 * math.pi
        if name == "sqrt":
            return math.sqrt(args[0])
        return vars_.get(name)
    return formula.Evaluator(ns).eval_text(text)


def test_formula_semantics():
    assert _ev("1 - progress * 1.73", progress=0.5) == 1 - 0.5 * 1.73
    assert _ev("2^3^2") == 2.0 ** 9            # right-associative
    assert _ev("7 % 4 * 2") == 6.0             # % binds tighter than *
    assert _ev("8 / 2 / 2") == 8 * (1 / 2) * (1 / 2)
    assert _ev("-(3.0^0.5)/4*0.5") == -(3.0 ** 0.5) * (1 / 4) * 0.5
    assert _ev("min(progress, 0.3) / 0.3", progress=0.1) == 0.1 * (1 / 0.3)
    assert _ev("pi()+acos(1/3)-0.0001") == pytest.approx(math.pi + math.acos(1 / 3) - 0.0001, abs=1e-15)
    assert _ev("((time*speed)*180)%360", time=3.0, speed=0.9) == math.fmod(3.0 * 0.9 * 180, 360)
    assert _ev("1 < 2 and 2 < 1") == 0.0 and _ev("1 < 2 or 2 < 1") == 1.0
    assert _ev("deg2rad(-90) * min(p, 0.5) / 0.5", p=0.25) == pytest.approx(-math.pi / 4)
    with pytest.raises(formula.FormulaError):
        _ev("nope + 1")


def test_glam_restatement():
    m = frontend.srt_matrix([2.0, 2.0, 2.0], [0.3, -0.7, 1.1], [1.0, 2.0, 3.0])
    inv = frontend.mat_inverse(m)
    prod = frontend.mat_mul(m, inv)
    for c in range(4):
        for r in range(4):
            assert prod[c][r] == pytest.approx(1.0 if c == r else 0.0, abs=1e-14)
    # rotation order Rx*Ry*Rz (matrix.rs:537-547): a pure z-rotation maps x to (cos, sin, 0)
    rz = frontend.srt_matrix([1, 1, 1], [0.0, 0.0, math.pi / 2], [0, 0, 0])
    assert rz[0][0] == pytest.approx(0.0, abs=1e-15) and rz[0][1] == pytest.approx(1.0)
    # singular input -> non-finite inverse, no exception (SURVEY.md Appendix A trap 1)
    sing = frontend.mat_inverse(frontend.srt_matrix([0.0, 0.0, 0.0], [0, 0, 0], [1, 2, 3]))
    assert any(not math.isfinite(x) for col in sing for x in col)


def test_known_answers_portal_in_portal():
    ir = load_ir("portal_in_portal")
    u = ir["uniforms"]

    def tz(name):
        m = u[name]["value"]
        assert m[:12] == [1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0]
        return m[12:]
    assert tz("a_mat") == [0.0, 0.0, -1.0, 1.0]          # portal_in_portal.ron:243-249
    assert tz("b0_mat") == [0.0, 0.0, 1.0, 1.0]          # :252-270 at progress = 0
    assert tz("b1_mat") == [0.0, 0.0, 3.0, 1.0]          # b0 * a^-1 * b0
    assert tz("b2_mat") == [0.0, 0.0, 5.0, 1.0]
    assert all(not math.isfinite(x) for x in u["c0_mat_inv"]["value"])   # scale = violet_progress = 0
    assert u["show_teleported_u"] == {"type": "int", "value": 10}
    assert u["teleport_light_u"]["value"] == 1 and u["progress_u"]["value"] == 0.0
    ids = ir["material_ids"]
    assert ids["room_yellow_M"] == 10 and ids["solid_0_M"] == 19 and ids["portal_grid_violet_M"] == 38
    assert not any(k.startswith("teleport_") for k in ids)      # no Portal objects in this scene
    assert len(ir["objects"]) == 14 and len(ir["materials"]) == 29 and len(ir["intersection_materials"]) == 1


@pytest.mark.parametrize("scene,expect", [
    ("basics", {"teleport_12_1_M": 32, "teleport_12_2_M": 33, "teleport_15_1_M": 34, "teleport_15_2_M": 35, "mirror_M": 22}),
    ("monoportal", {"teleport_6_1_M": 25, "teleport_6_2_M": 26, "room_yellow_M": 10}),
    ("triple_portal", {"teleport_6_1_M": 26, "teleport_20_2_M": 43, "room_black2_M": 25}),
    ("mobius_monoportal", {"teleport_6_1_M": 22, "teleport_6_2_M": 23, "solid_black_M": 21}),
])
def test_material_ids_appendix_a(scene, expect):
    ids = load_ir(scene)["material_ids"]
    for k, v in expect.items():
        assert ids[k] == v


def test_glsl_rewrite():
    sw = set()
    out = gen_oracle.glsl_to_cpp("for (int i = 0; i < 50; i++) { if (i >= n) break; // !FOR_NUMBER!\n"
                                 "for (int i = 0; i < n; i++) { // !FOR_VARIABLE!\n vec3 p = (r.o + r.d * 2.).xyz; float q = 1e-3 + p.x; }", "f", sw)
    assert "50" not in out and ".xyz()" in out and "2.f" in out and "1e-3f" in out and "p.x" in out
    assert sw == {"xyz"}
    assert gen_oracle.glsl_to_cpp("void f(out vec3 a, inout float b, in int c)", "f", set()).split() == \
        "void f( vec3& a, float& b, int c)".split()


@pytest.mark.parametrize("scene", SCENES)
def test_oracle_reproduces_golden_frame(scene):
    ir = load_ir(scene)
    files = [f for f in os.listdir(os.path.join(GOLDEN, "frames")) if f.startswith(scene + "_")]
    assert len(files) == 1
    w, h = map(int, files[0].split("_")[-2].split("x"))
    with np.load(os.path.join(GOLDEN, "frames", files[0])) as z:
        gold, sha = z["frame"], str(z["sha256"])
    assert hashlib.sha256(gold.tobytes()).hexdigest() == sha
    for variant in ("strict", "fast"):
        img = runner.Oracle(ir, variant, textures=load_tex(scene)).render(w, h, DEPTH[scene])
        assert np.array_equal(img.view(np.uint32), gold.view(np.uint32)), f"{scene}/{variant} differs from its pin"
    assert np.all(gold[..., 3] == 1.0) and np.isfinite(gold).all()


def test_oracle_invariants():
    ir = load_ir("portal_in_portal")
    orc = runner.Oracle(ir, "fast")
    black = orc.render(32, 18, 0)                              # depth 0 -> all black (frag.glsl:158)
    assert np.all(black[..., :3] == 0.0) and np.all(black[..., 3] == 1.0)
    full = orc.render(64, 36, 40)
    part = orc.render(64, 36, 40, rows=(10, 20))               # row ranges are independent
    assert np.array_equal(full[10:20], part)
    orc.set_uniforms({"teleport_light_u": 0})                  # no teleports -> every ray ends on its first hit
    _, bounces = orc.render(64, 36, 40, want_bounces=True)
    assert bounces.max() == 1
    # AA: 4 samples differ from 1 sample only by a small amount on a smooth image
    orc.set_uniforms()
    aa = orc.render(64, 36, 40, aa_count=4)
    assert np.abs(aa - full).mean() < 0.05 and not np.array_equal(aa, full)


def test_f64_oracle_flags_few_pixels():
    """float64 arithmetic on the same inputs: differences beyond 1e-4 mark ill-conditioned (edge) pixels."""
    ir = load_ir("triple_portal")
    a = runner.Oracle(ir, "fast").render(160, 90, 40)
    d = runner.Oracle(ir, "f64").render(160, 90, 40)
    bad = (np.abs(a - d).max(axis=-1) > 1e-4).mean()
    assert bad < 0.01


@pytest.mark.parametrize("scene", SCENES)
def test_frontend_regenerates_committed_ir(scene, reference):
    ir = frontend.scene_ir(frontend.load_scene(f"{reference}/scenes/{scene}.ron"), scene)
    gold = load_ir(scene)
    assert list(ir["uniforms"]) == list(gold["uniforms"])
    for k, u in ir["uniforms"].items():
        a, g = np.asarray(u["value"], dtype=np.float64), np.asarray(gold["uniforms"][k]["value"], dtype=np.float64)
        assert np.array_equal(a, g, equal_nan=True), k
    assert ir["objects"] == gold["objects"] and ir["materials"] == gold["materials"] and ir["library"] == gold["library"]
    assert ir["camera_matrix"] == gold["camera_matrix"]
