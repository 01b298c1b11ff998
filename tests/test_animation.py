"""The animation layer between a scene file and one frame's uniforms: stages with cameras, real
animations (time mapping, camera interpolation), named cameras and camera teleportation through portals.
C++ host (`ph_player_*`, portal_b200/csrc/host/ph_anim.cpp) against the oracle's independent restatement
(oracle/animation.py) -- value for value in float64 -- plus hand-checkable facts about the fixture scene."""
import glob
import math
import os

import numpy as np
import pytest

from conftest import ROOT
from portal_b200.capi import PortalB200Error
from portal_b200.host import HostPlayer, HostRenderer, HostScene

FIXTURE = os.path.join(ROOT, "tests", "fixtures", "two_spheres.ron")
ANIMS = [("fly.1", 2.0), ("fly.2", 1.5), ("hold", 1.0), ("through", 4.0)]


def _same(a, b):
    return np.array_equal(np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64), equal_nan=True)


def _assert_same_state(p, hp, s, hs, where):
    a, b = p.camera_state(), hp.camera_state()
    for k in a:
        assert _same(a[k], b[k]), (where, k, a[k], b[k])
    ta, tb = s.uniform_table(), hs.uniform_table()
    assert list(ta) == list(tb), where
    for k in ta:
        assert _same(ta[k][1], tb[k][1]), (where, k)


def _pair(path):
    from oracle import frontend
    from oracle.animation import Player
    s = frontend.load_scene(path)
    hs = HostScene.from_file(path)
    return s, Player(s), hs, HostPlayer(hs)


def test_fixture_animations_match_oracle_player():
    _, _, hs0, hp0 = _pair(FIXTURE)
    assert hp0.animations() == ANIMS
    assert sorted(hp0.camera_names()) == ["at_ball", "before_gate", "behind_gate", "beside_gate", "wide"]
    for name, _ in ANIMS:
        s, p, hs, hp = _pair(FIXTURE)
        p.init_animation(name)
        hp.init_animation(name)
        for t in (0.0, 0.3, 1.0, 1.7, 2.6, 0.2):           # not monotonic: the wrap re-arms `override_matrix`
            p.update(t)
            hp.update(t)
            _assert_same_state(p, hp, s, hs, (name, t))


def test_time_mapping_and_camera_chain():
    """Scene::update (scene.rs:1385-1418): inside a real animation formula `time` = (t % duration) / duration and
    `total_time` adds the durations of the animations before it; cameras: get_start_cam / get_end_cam (:1291-1335)."""
    s, p, hs, hp = _pair(FIXTURE)
    hp.init_animation("fly.2")
    hp.update(0.3)
    st = hp.camera_state()
    assert st["time"] == math.fmod(0.3, 1.5) / 1.5 and st["total_time"] == 2.0 + math.fmod(0.3, 1.5)
    # fly.2 builds on RealAnimation("fly.1") which builds on stage "closed": p from fly.1, spin formula from fly.2
    t = hs.uniform_table()
    assert t["p_u"] == ("float", 0.9) and t["open_u"] == ("int", 0) and t["spin_u"] == ("float", 0.2 + st["time"])
    # use_prev_cam: fly.2 starts where fly.1 ends
    hp.update(0.0)
    st = hp.camera_state()
    assert st["look_at"] == [0.0, 0.5, 0.25] and (st["alpha"], st["beta"], st["r"]) == (2.9, 1.4, 2.2)
    # cam_easing_uniform is clamped to [0, 1]: near the end of fly.2 the camera IS the end camera ("at_ball")
    hp.update(1.49)
    st = hp.camera_state()
    ball = np.asarray(hs.uniform_table()["ball_mat"][1]).reshape(4, 4)[3, :3]       # column-major: translation
    assert (st["alpha"], st["beta"], st["r"]) == (-0.4, 1.3, 1.9)
    assert np.allclose(st["look_at"], ball + 0.001, atol=1e-15)                    # MatrixCenter: centre + 0.001 (camera.rs:117-120)
    # "hold": use_any_cam_as_start = Some(false) -> fly.1's START camera; use_start_cam_as_end -> stays there
    _, _, hs2, hp2 = _pair(FIXTURE)
    hp2.init_animation("hold")
    for tm in (0.0, 0.6):
        hp2.update(tm)
        st = hp2.camera_state()
        assert st["look_at"] == [0.3, 0.1, -0.2] and (st["alpha"], st["beta"], st["r"]) == (2.1, 1.05, 3.6)
    assert hp2.camera_state()["total_time"] == 3.5 + 0.6
    assert hs2.uniform_table()["open_u"] == ("int", 1)                              # Dev stage restored


def test_run_animations_plays_the_whole_sequence():
    """Scene::run_animations (scene.rs:1359-1384): one clock over all real animations (2.0 + 1.5 + 1.0 + 4.0 s here)."""
    s, p, hs, hp = _pair(FIXTURE)
    p.anim.run_animations = True
    hp.set_run_animations(True)
    for t, (name, local) in [(0.5, ("fly.1", 0.25)), (2.75, ("fly.2", 0.5)), (3.9, ("hold", 0.4)), (6.5, ("through", 0.5)),
                              (8.5 + 1.0, ("fly.1", 0.5)), (1.9, ("fly.1", 0.95))]:
        p.update(t)
        hp.update(t)
        _assert_same_state(p, hp, s, hs, t)
        st = hp.camera_state()
        assert p.anim.current_stage == ("real", name)
        assert abs(st["time"] - local) < 1e-12 and abs(st["total_time"] - math.fmod(t, 8.5)) < 1e-12


def test_stage_and_named_cameras():
    s, p, hs, hp = _pair(FIXTURE)
    hp.update(0.0)                                                                  # plain render-frame: the saved camera
    st = hp.camera_state()
    assert st["look_at"] == [0.1, -0.2, 0.0] and (st["alpha"], st["beta"], st["r"]) == (0.83, 1.21, 2.9) and st["time"] == 0.0
    hp.init_stage("closed")                                                         # set_cam: Some(Some(Named("wide")))
    hp.update(0.25)
    st = hp.camera_state()
    assert (st["alpha"], st["beta"], st["r"]) == (2.1, 1.05, 3.6) and st["time"] == 0.25 and st["total_time"] == 0.25
    hp.init_stage("reset")                                                          # set_cam: None -> back to the original camera
    hp.update(0.0)
    assert hp.camera_state()["alpha"] == 0.83
    hp.select_camera("at_ball")
    hp.update(0.0)
    assert hp.camera_state()["r"] == 1.9
    for bad in (hp.init_stage, hp.init_animation, hp.select_camera):
        with pytest.raises(PortalB200Error, match="no (stage|animation|camera) named"):
            bad("nope")
    # same walk on the oracle side
    p.update(0.0)
    p.init_stage("closed")
    p.update(0.25)
    p.init_stage("reset")
    p.update(0.0)
    p.select_camera("at_ball")
    p.update(0.0)
    _assert_same_state(p, hp, s, hs, "stage walk")


def test_camera_teleports_through_the_gate_on_the_oracle():
    """teleport_camera + teleport_matrix (main.rs:1217-1264, 1174-1215) with the CPU oracle as the external-ray
    probe: walking through the open gate costs 1 + 3 probes once, and the finite-difference matrix it recovers is
    portal_b * portal_a^-1 (to the 1e-3 step of the differences)."""
    from oracle import frontend
    from oracle.animation import Player
    from oracle.runner import Oracle
    orc = Oracle(frontend.scene_ir(frontend.load_scene(FIXTURE), "two_spheres"), variant="strict")
    s = frontend.load_scene(FIXTURE)
    p = Player(s, probe=_oracle_probe(orc))
    p.init_animation("through")
    crossed_at, cams = None, []
    for k in range(21):
        p.update(4.0 * k / 20 * 0.999)
        cams.append(p.camera_state())
        if crossed_at is None and p.cam.teleport_matrix != frontend.mat_identity():
            crossed_at = k
            a = s.get_matrix(s.matrix_by_name["portal_a"])
            b = s.get_matrix(s.matrix_by_name["portal_b"])
            want = np.asarray(frontend.mat_mul(b, frontend.mat_inverse(a)))
            assert np.allclose(np.asarray(p.cam.teleport_matrix), want, atol=2e-3)
    assert crossed_at == 13 and p.n_probes == 20 + 3
    before, after = np.asarray(cams[12]["camera"][12:15]), np.asarray(cams[13]["camera"][12:15])
    assert np.linalg.norm(after - before) > 2.0                                    # the eye is now at the other portal
    assert np.allclose(np.asarray(cams[13]["camera_mul_inv"]).reshape(4, 4).T @ np.asarray(p.cam.teleport_matrix).reshape(4, 4).T,
                       np.eye(4), atol=1e-12)


def test_stereo_eye_is_carried_through_the_gate_on_the_oracle():
    """teleport_eye_matrices (main.rs:1121-1172): camera "beside_gate" stands 0.1 in front of the gate with its x axis
    along the gate's normal; with eye_distance 0.25 the left eye lies behind the gate plane and must come out of
    portal_b, the right eye is a plain translation.  Without a probe both eyes are plain translations (C++ == oracle)."""
    from oracle import frontend
    from oracle.animation import Player
    from oracle.runner import Oracle
    orc = Oracle(frontend.scene_ir(frontend.load_scene(FIXTURE), "two_spheres"), variant="strict")
    s = frontend.load_scene(FIXTURE)
    p = Player(s, probe=_oracle_probe(orc))
    p.draw_side_by_side, p.eye_distance = True, 0.25
    p.select_camera("beside_gate")
    p.update(0.0)
    cs = p.camera_state()
    cam, left, right = (np.asarray(cs[k]).reshape(4, 4) for k in ("camera", "left_eye", "right_eye"))
    assert p.n_probes == 2 + 3
    assert np.allclose(right[3, :3], cam[3, :3] + 0.25 * cam[0, :3], atol=1e-15) and np.array_equal(right[:3], cam[:3])
    a, b = s.get_matrix(s.matrix_by_name["portal_a"]), s.get_matrix(s.matrix_by_name["portal_b"])
    t = np.asarray(frontend.mat_mul(b, frontend.mat_inverse(a)))                    # rows = columns (column-major)
    plain_left = np.append(cam[3, :3] - 0.25 * cam[0, :3], 1.0)
    assert np.allclose(left[3, :3], (plain_left @ t)[:3], atol=1e-4)
    assert np.allclose(left[:3, :3], cam[:3, :3] @ t[:3, :3], atol=2e-3)
    # no probe attached: both players place the eyes by translation only, identically
    s2, p2, hs2, hp2 = _pair(FIXTURE)
    p2.draw_side_by_side, p2.eye_distance = True, 0.25
    hp2.set_stereo(True, 0.25)
    for pl in (p2, hp2):
        pl.select_camera("beside_gate")
        pl.update(0.0)
    _assert_same_state(p2, hp2, s2, hs2, "stereo without probe")
    assert np.allclose(np.asarray(hp2.camera_state()["left_eye"]).reshape(4, 4)[3, :3], plain_left[:3], atol=1e-15)


def _oracle_probe_for_host(orc, hs, hp):
    """The same CPU probe, attached to the C++ player through ph_player_set_probe."""
    def probe(a, b):
        orc.set_uniforms({k: v for k, (_, v) in hs.uniform_table().items()})
        cs = hp.camera_state()
        pos, _, enc, chg = orc.probe(a, b, camera=cs["camera"], camera_scale=cs["scale"], camera_mul_inv=cs["camera_mul_inv"],
                                     camera_in_subspace=int(cs["in_subspace"]))
        have = not (pos[0] == 0 and pos[1] == 0 and pos[2] == 0)
        return ([float(x) for x in pos] if have else None, enc, chg)
    return probe


def test_cpp_player_teleports_like_the_oracle_player_on_the_cpu():
    """teleport_camera / teleport_matrix / teleport_eye_matrices of the C++ player, driven by the CPU oracle's probe through
    ph_player_set_probe, against the oracle player driven by the same probe: every camera, eye and teleport matrix and the
    probe count, bit for bit -- the walk through the gate and the stereo pair straddling it, no GPU involved."""
    from oracle import frontend
    from oracle.animation import Player
    from oracle.runner import Oracle
    orc = Oracle(frontend.scene_ir(frontend.load_scene(FIXTURE), "two_spheres"), variant="strict")
    s = frontend.load_scene(FIXTURE)
    p = Player(s, probe=_oracle_probe(orc))
    hs = HostScene.from_file(FIXTURE)
    hp = HostPlayer(hs)
    hp.set_probe(_oracle_probe_for_host(orc, hs, hp))
    p.init_animation("through")
    hp.init_animation("through")
    for k in range(21):
        t = 4.0 * k / 20 * 0.999
        p.update(t)
        hp.update(t)
        _assert_same_state(p, hp, s, hs, ("through", k))
        assert hp.camera_state()["n_probes"] == p.n_probes
    assert p.n_probes == 23 and p.cam.teleport_matrix != frontend.mat_identity()
    # stereo pair straddling the gate
    s2 = frontend.load_scene(FIXTURE)
    p2 = Player(s2, probe=_oracle_probe(orc))
    p2.draw_side_by_side, p2.eye_distance = True, 0.25
    hs2 = HostScene.from_file(FIXTURE)
    hp2 = HostPlayer(hs2)
    hp2.set_probe(_oracle_probe_for_host(orc, hs2, hp2))
    hp2.set_stereo(True, 0.25)
    for pl in (p2, hp2):
        pl.select_camera("beside_gate")
        pl.update(0.0)
    _assert_same_state(p2, hp2, s2, hs2, "stereo")
    assert hp2.camera_state()["n_probes"] == 5
    hp2.set_probe(None)                                                              # detached: plain translations again
    hp2.update(0.0)
    assert hp2.camera_state()["n_probes"] == 5


def _oracle_probe(orc):
    def probe(player, a, b):
        table = player.scene.uniform_table()
        orc.set_uniforms({k: v for k, (_, v) in table.items()})
        cs = player.camera_state()
        pos, _, enc, chg = orc.probe(a, b, camera=cs["camera"], camera_scale=cs["scale"], camera_mul_inv=cs["camera_mul_inv"],
                                     camera_in_subspace=int(cs["in_subspace"]))
        have = not (pos[0] == 0 and pos[1] == 0 and pos[2] == 0)                    # main.rs:1399
        return ([float(x) for x in pos] if have else None, enc, chg)
    return probe


def test_reference_scene_animations_match_oracle_player(reference):
    """Every reference scene: its first animations at four times, camera + full uniform table, C++ == oracle."""
    n = 0
    for path in sorted(glob.glob(f"{reference}/scenes/*.ron")):
        if os.path.basename(path) == "empty.ron":
            continue
        _, p0, _, hp0 = _pair(path)
        names = [a["name"] for a in p0.anim.animations]
        assert [a for a, _ in hp0.animations()] == names
        for an in names[:3]:
            s, p, hs, hp = _pair(path)
            p.init_animation(an)
            hp.init_animation(an)
            dur = p.anim.animations[p.anim.animation_by_name[an]]["duration"]
            for tt in (0.0, 0.37 * dur, 0.99 * dur, 1.5 * dur):
                p.update(tt)
                hp.update(tt)
                _assert_same_state(p, hp, s, hs, (path, an, tt))
                n += 1
    assert n >= 250


@pytest.mark.gpu
def test_player_teleports_on_the_gpu_like_the_oracle(torch_cuda):
    """The same walk through the gate with pe_probe_ray as the probe: every camera matrix, the teleport matrix and
    the probe count equal the oracle-driven player's bit for bit; the frame after the crossing equals the oracle's."""
    from oracle import frontend
    from oracle.animation import Player
    from oracle.runner import Oracle
    orc = Oracle(frontend.scene_ir(frontend.load_scene(FIXTURE), "two_spheres"), variant="strict")
    s = frontend.load_scene(FIXTURE)
    p = Player(s, probe=_oracle_probe(orc))
    hs = HostScene.from_file(FIXTURE)
    hr = HostRenderer(hs)
    hp = HostPlayer(hs, hr)
    p.init_animation("through")
    hp.init_animation("through")
    for k in range(21):
        t = 4.0 * k / 20 * 0.999
        p.update(t)
        hp.update(t)
        a, b = p.camera_state(), hp.camera_state()
        for key in a:
            assert _same(a[key], b[key]), (k, key)
        assert b["n_probes"] == p.n_probes
    assert hp.camera_state()["n_probes"] == 23
    cs = p.camera_state()
    orc.set_uniforms({k: v for k, (_, v) in s.uniform_table().items()})
    want = orc.render(192, 108, 12, camera=cs["camera"], camera_scale=cs["scale"], camera_mul_inv=cs["camera_mul_inv"],
                      camera_in_subspace=int(cs["in_subspace"]))
    got = hp.render_frame(192, 108, 12)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


@pytest.mark.gpu
def test_cli_render_frame_animation_and_render_loop(torch_cuda, tmp_path):
    """`portal_b200_render render-frame --animation/--time` and `render --animations` (C++ only) against the same
    calls made through the Python bindings."""
    import subprocess
    exe = os.path.join(ROOT, "portal_b200", "portal_b200_render")
    out = tmp_path / "f.rgba"
    r = subprocess.run([exe, "render-frame", FIXTURE, "--width", "160", "--height", "90", "--render-depth", "12", "--animation", "fly.2",
                        "--time", "0.6", "--output", str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    got = np.frombuffer(out.read_bytes(), dtype=np.uint8).reshape(90, 160, 4)
    hs = HostScene.from_file(FIXTURE)
    hr = HostRenderer(hs)
    hp = HostPlayer(hs, hr)
    hp.init_animation("fly.2")
    hp.update(0.6)
    assert np.array_equal(got, hp.render_frame(160, 90, 12, rgba8=True))
    r = subprocess.run([exe, "render-frame", FIXTURE, "--animation", "nope"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 1 and "has no animation named `nope`" in r.stderr
    # the offline loop: 2 of the 4.0 s * 5 fps = 20 frames of "through", 3 motion-blur sub-frames each
    r = subprocess.run([exe, "render", FIXTURE, "--animations", "through", "--fps", "5", "--motion-blur-frames", "3", "--width", "96",
                        "--height", "54", "--render-depth", "8", "--aa-count", "1", "--out-dir", str(tmp_path / "video"), "--max-frames", "2"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    hs = HostScene.from_file(FIXTURE)
    hr = HostRenderer(hs)
    hp = HostPlayer(hs, hr)
    hp.init_animation("through")
    hp.update(0.0)
    for i in range(2):
        want = hp.render_motion_blur_frame(96, 54, 8, i, 20, 3, 4.0)
        raw = (tmp_path / "video" / "through" / f"frame_{i}.ppm").read_bytes()
        assert raw.startswith(b"P6\n96 54\n255\n")
        got = np.frombuffer(raw[len(b"P6\n96 54\n255\n"):], dtype=np.uint8).reshape(54, 96, 3)
        assert np.array_equal(got, want[..., :3])


@pytest.mark.gpu
def test_stereo_frame_through_the_gate_on_the_gpu(torch_cuda):
    """Eye placement with pe_probe_ray == the oracle-driven player's, bit for bit; the side-by-side frame rendered
    with those eye cameras equals the oracle's frame."""
    from oracle import frontend
    from oracle.animation import Player
    from oracle.runner import Oracle
    orc = Oracle(frontend.scene_ir(frontend.load_scene(FIXTURE), "two_spheres"), variant="strict")
    s = frontend.load_scene(FIXTURE)
    p = Player(s, probe=_oracle_probe(orc))
    p.draw_side_by_side, p.eye_distance = True, 0.25
    hs = HostScene.from_file(FIXTURE)
    hr = HostRenderer(hs)
    hp = HostPlayer(hs, hr)
    hp.set_stereo(True, 0.25)
    for pl in (p, hp):
        pl.select_camera("beside_gate")
        pl.update(0.0)
    a, b = p.camera_state(), hp.camera_state()
    for key in a:
        assert _same(a[key], b[key]), key
    assert b["n_probes"] == 5
    orc.set_uniforms({k: v for k, (_, v) in s.uniform_table().items()})
    want = orc.render(256, 72, 12, camera=a["camera"], camera_scale=a["scale"], camera_mul_inv=a["camera_mul_inv"],
                      camera_in_subspace=int(a["in_subspace"]), draw_side_by_side=1,
                      camera_left_eye=a["left_eye"], camera_right_eye=a["right_eye"],
                      left_eye_in_subspace=int(a["left_eye_in_subspace"]), right_eye_in_subspace=int(a["right_eye_in_subspace"]),
                      left_eye_scale=frontend.camera_scale(p.left_eye_matrix), right_eye_scale=frontend.camera_scale(p.right_eye_matrix))
    got = hp.render_frame(256, 72, 12)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def _random_animation_scene(n, seed):
    """The fixture scene with its animations replaced by n random ones: every stage kind, Changed / CopyPrev parts, camera
    chains through use_prev_cam / use_start_cam_as_end / use_any_cam_* (cycles included), all easings, easing uniforms."""
    import random
    rng = random.Random(seed)
    cams = ["wide", "at_ball", "before_gate", "behind_gate", "beside_gate"]
    names = [f"an{i}" for i in range(n)]

    def cam():
        k = rng.random()
        if k < 0.25:
            return "None"
        if k < 0.7:
            return f'Some(Named("{rng.choice(cams)}"))'
        la = (f"Coordinate(({rng.uniform(-1, 1):.3f}, {rng.uniform(-1, 1):.3f}, {rng.uniform(-1, 1):.3f}))" if rng.random() < 0.7
              else 'MatrixCenter(Some(Named("ball")))')
        return (f"Some(Inline((look_at: {la}, alpha: {rng.uniform(-3, 3):.4f}, beta: {rng.uniform(0.2, 2.9):.4f}, r: {rng.uniform(0.5, 4):.3f}, "
                f"in_subspace: {rng.choice(['true', 'false'])}, free_movement: {rng.choice(['true', 'false', 'false'])}, "
                "matrix: (1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.5, 0.0, -0.25, 1.0))))")

    def opt_flag():
        return rng.choice(["None", "None", "Some(true)", "Some(false)"])

    def any_name():
        return "None" if rng.random() < 0.3 else f'Some("{rng.choice(names)}")'

    out = []
    for i, nm in enumerate(names):
        stage = rng.choice(["Dev", 'Animation("closed")', 'Animation("reset")'] + ([f'RealAnimation("{rng.choice(names[:i])}")'] if i else []))
        p = rng.choice(["CopyPrev", f"Changed(Some(Inline(Progress({rng.uniform(0, 1):.3f}))))", 'Changed(Some(Inline(Formula(("0.3 + time * 0.5")))))'])
        spin = rng.choice(["CopyPrev", f"Changed(Some(Inline(Angle({rng.uniform(-2, 2):.3f}))))", 'Changed(Some(Named("wobble")))'])
        ball = rng.choice(["CopyPrev", 'Changed(Some(Named("portal_a")))',
                           'Changed(Some(Inline(Lerp(t: Uniform(Some(Inline(Formula(("time"))))), first: Some(Named("portal_a")), second: Some(Named("portal_b"))))))'])
        easing = rng.choice(["Linear", "In", "Out", "InOut", "InOutFast", "ElasticOut"])
        eu = rng.choice(["None", "None", 'Some(Inline(Formula(("easing_in_out(time) * 1.2 - 0.1"))))', 'Some(Named("p"))'])
        out.append(f"""        (name: "{nm}", data: (
            duration: {rng.choice(['0.0', '0.5', '1.0', '2.5', '3.0'])},
            animation_stage: {stage},
            uniforms: ({{"p": {p}, "spin": {spin}, "open": CopyPrev, "count": CopyPrev}}),
            matrices: ({{"portal_a": CopyPrev, "ball": {ball}}}),
            use_prev_cam: {rng.choice(['true', 'false', 'false'])},
            use_start_cam_as_end: {rng.choice(['true', 'false', 'false'])},
            cam_start: {cam()},
            cam_end: {cam()},
            use_any_cam_as_start: {opt_flag()},
            use_any_cam_as_end: {opt_flag()},
            cam_any_start: {any_name()},
            cam_any_end: {any_name()},
            cam_easing: {easing},
            cam_easing_uniform: {eu},
        )),
""")
    text = open(FIXTURE, encoding="utf-8").read()
    i = text.index("    animations: ([")
    j = text.index("    current_stage:", i)
    return text[:i] + "    animations: ([\n" + "".join(out) + "    ]),\n" + text[j:]


@pytest.mark.parametrize("seed", [11, 12])
def test_players_agree_on_random_animations(seed, tmp_path):
    """Differential fuzz of the two animation layers (C++ ph_anim.cpp vs oracle/animation.py): 60 random animations; each is
    initialised and stepped through five times (wrap-around included); cameras, times and uniform tables must be identical."""
    path = tmp_path / "anim.ron"
    path.write_text(_random_animation_scene(60, seed), encoding="utf-8")
    s0, p0, hs0, hp0 = _pair(str(path))
    names = [a for a, _ in hp0.animations()]
    assert names == [a["name"] for a in p0.anim.animations] and len(names) == 60
    n = 0
    for nm in names:
        s, p, hs, hp = _pair(str(path))
        p.init_animation(nm)
        hp.init_animation(nm)
        for t in (0.0, 0.4, 0.93, 2.7, 0.1):
            p.update(t)
            hp.update(t)
            _assert_same_state(p, hp, s, hs, (seed, nm, t))
            n += 1
    assert n == 300
    # one clock over the whole sequence
    s, p, hs, hp = _pair(str(path))
    p.anim.run_animations = True
    hp.set_run_animations(True)
    for t in (0.0, 3.3, 17.0, 41.9, 5.5):
        p.update(t)
        hp.update(t)
        _assert_same_state(p, hp, s, hs, (seed, "run", t))


def test_per_animation_overrides_of_update_inner_variables(reference):
    """SceneRenderer::update_inner_variables (main.rs:1696-1755), applied right after init_animation_by_name as render-frame
    does: `subspace_degree` becomes Int(500) / Int(1000) for the listed animation names, render depth 100 / fps 600 for others;
    a scene WITHOUT `subspace_degree` leaves the function at the `?` -- before the depth override.  C++ player == oracle
    player, uniform table included."""
    seen = {"degree500": 0, "degree1000": 0, "depth": 0, "fps": 0, "early_exit": 0}
    for scene in ("portal_in_portal", "portal_in_portal_cone", "portal_in_portal_plus_ultra", "teleportation_degrees", "recursive_space"):
        path = f"{reference}/scenes/{scene}.ron"
        _, p0, _, _ = _pair(path)
        for an in [a["name"] for a in p0.anim.animations]:
            s, p, hs, hp = _pair(path)
            p.init_animation(an)
            hp.init_animation(an)
            ov = hp.animation_overrides()
            assert ov == {"render_depth": p.render_depth_override, "fps": p.fps_override}, (scene, an)
            p.update(0.1)
            hp.update(0.1)
            _assert_same_state(p, hp, s, hs, (scene, an))
            table = hs.uniform_table()
            has_degree = "subspace_degree_u" in table
            if an in p._DEGREE_500 and has_degree:
                want = 1000 if an in ("v2.spiral.4", "v2.spiral.5", "v2.spiral.6") else 500
                assert table["subspace_degree_u"] == ("int", want), (scene, an)
                seen["degree1000" if want == 1000 else "degree500"] += 1
            if an in p._DEGREE_500 and not has_degree:
                assert ov == {"render_depth": 0, "fps": 0}
                seen["early_exit"] += 1
            seen["depth"] += ov["render_depth"] == 100
            seen["fps"] += ov["fps"] == 600
    assert seen["degree500"] >= 1 and seen["depth"] >= 1 and seen["fps"] >= 1, seen


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["portal_in_portal", "triple_portal", "basics"])
def test_animated_states_of_config_scenes_bit_exact_on_the_gpu(scene, torch_cuda):
    """The config scenes are measured at their saved state, where many matrices are pure translations and some are singular
    (`c0`: scale 0, inverse all NaN).  Animations drive exactly those: `violet_progress` opens the third portal, matrices
    stop being translations, structure masks and the finite flags of the specialised program change from frame to frame.
    Every animation of the scene, three times each, through the product's own player (C++ host + GPU) against the oracle
    driven by the oracle's player: camera, uniform tables and every pixel, bit for bit."""
    from conftest import GOLDEN, load_tex
    from oracle import frontend
    from oracle.animation import Player
    from oracle.runner import Oracle
    path = os.path.join(ROOT, "tests", "golden", "ron", f"{scene}.ron")
    depth = {"portal_in_portal": 40, "triple_portal": 40, "basics": 4}[scene]
    tex = load_tex(scene)
    s0 = frontend.load_scene(path)
    names = [a["name"] for a in Player(s0).anim.animations]
    assert len(names) >= 2
    orc = Oracle(frontend.scene_ir(s0, scene), variant="fast", textures=tex)
    hs = HostScene.from_file(path)
    hr = HostRenderer(hs, textures=tex)
    hp = HostPlayer(hs, hr)
    s = frontend.load_scene(path)
    p = Player(s)
    n = 0
    for an in names[:6]:
        p.init_animation(an)
        hp.init_animation(an)
        dur = p.anim.animations[p.anim.animation_by_name[an]]["duration"]
        for frac in (0.13, 0.5, 0.97):
            p.update(frac * dur)
            hp.update(frac * dur)
            _assert_same_state(p, hp, s, hs, (an, frac))
            cs = p.camera_state()
            orc.set_uniforms({k: v for k, (_, v) in s.uniform_table().items()})
            want = orc.render(160, 90, depth, camera=cs["camera"], camera_scale=cs["scale"], camera_mul_inv=cs["camera_mul_inv"],
                              camera_in_subspace=int(cs["in_subspace"]))
            got = hp.render_frame(160, 90, depth)
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (scene, an, frac, int((got.view(np.uint32) != want.view(np.uint32)).any(axis=-1).sum()))
            n += 1
    assert n >= 6
