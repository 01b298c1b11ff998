"""Video textures (SURVEY.md section 8 f1, the last reference scene that did not compile: `boot.dev`).  In the reference a video
is one more `uniform sampler2D <name>_tex` (src/gui/scene.rs:405-409, 703-716) whose image the host replaces every frame with
ONE frame of a clip: frame index = round((frames - 1) * clamp(uniform, 0, 1)) (src/main.rs:862-914, src/gui/video.rs:14-20).
Decoding the clip (ffmpeg -> PNG, video.rs:65-110) is image IO and out of scope; what is in scope and checked here, on
`tests/fixtures/video.ron` (hand-written): both front-ends read the `videos:` section, declare the sampler, agree on the
uniform table and on the frame index at every time; the generated sm_100a program, run on the host harness with the selected
frame bound, gives the oracle's pixels bit for bit; an unbound video sampler reads black.  (No GPU needed: the GPU side is
`pe_set_texture` + a render, which the texture scenes of tests/test_all_scenes_gpu.py cover.)"""
import os

import numpy as np

from conftest import ROOT
from portal_b200.host import HostRenderer, HostScene
from test_host_frontend import _assert_same_table, _oracle_ir
from test_program_on_host import H, W, _bits, _run_on_host

FIXTURE = os.path.join(ROOT, "tests", "fixtures", "video.ron")
IDENTITY = [1.0, 0, 0, 0, 0, 1.0, 0, 0, 0, 0, 1.0, 0, 0, 0, 0, 1.0]      # eye at the origin looking down +z, like tests/test_analytic.py


def _oracle_scene():
    from oracle import frontend
    return frontend.load_scene(FIXTURE)


def test_videos_are_samplers_in_both_front_ends():
    ir = _oracle_ir(FIXTURE, "video", time=3.0)
    assert [t["name"] for t in ir["textures"]] == ["still", "clip", "silent"] and ir["textures"][1] == {"name": "clip", "path": None, "video": True}
    assert ir["videos"] == [{"name": "clip", "path": "clips/clip.mov", "uniform": "clip_pos"}, {"name": "silent", "path": "", "uniform": None}]
    hs = HostScene.from_file(FIXTURE)
    assert hs.videos() == [("clip", "clips/clip.mov", "clip_pos"), ("silent", "", None)]
    assert hs.counts()["videos"] == 2 and hs.counts()["textures"] == 1 and hs.textures() == [("still", "tests/fixtures/still.png")]
    hs.set_time(3.0)
    _assert_same_table(hs.uniform_table(), ir)
    src = HostRenderer(hs, device=-1).source()                 # the product's front-end declares the samplers too (NVRTC accepts it)
    assert "clip_tex" in src and "silent_tex" in src and "still_tex" in src


def test_frame_selection_known_answers_and_agreement():
    sc, hs = _oracle_scene(), HostScene.from_file(FIXTURE)
    # clip_pos = time / 8;  index = round((n - 1) * clamp(clip_pos, 0, 1)), halves away from zero (Rust's f64::round)
    for time, n, want in [(0.0, 5, 0), (4.0, 5, 2), (1.0, 5, 1), (2.0, 5, 1), (3.0, 5, 2), (8.0, 5, 4), (100.0, 5, 4), (-3.0, 5, 0),
                          (4.0, 100, 50), (1.0, 100, 12), (5.0, 1, 0), (4.0, 2, 1), (3.9, 2, 0)]:
        sc.time = sc.total_time = time
        hs.set_time(time)
        assert sc.video_frame_index(0, n) == want and hs.video_frame_index(0, n) == want, (time, n)
    assert sc.video_frame_index(0, 0) is None and hs.video_frame_index(0, 0) is None          # no frames: nothing to show
    assert sc.video_frame_index(1, 7) is None and hs.video_frame_index(1, 7) is None          # a video without a uniform
    assert hs.video_frame_index(2, 7) is None                                                  # no such video
    rng = np.random.default_rng(3)
    for _ in range(300):
        time, n = float(rng.uniform(-2, 10)), int(rng.integers(1, 500))
        sc.time = sc.total_time = time
        hs.set_time(time)
        assert sc.video_frame_index(0, n) == hs.video_frame_index(0, n), (time, n)


def test_the_selected_frame_reaches_the_pixels(tmp_path):
    from oracle.runner import Oracle
    rng = np.random.default_rng(8)
    frames = [rng.integers(0, 256, size=(18, 32, 4), dtype=np.uint8) for _ in range(3)]
    still = rng.integers(0, 256, size=(8, 8, 4), dtype=np.uint8)
    sc = _oracle_scene()
    seen = []
    for time in (0.0, 4.0, 8.0):
        ir = _oracle_ir(FIXTURE, "video", time=time)
        sc.time = sc.total_time = time
        k = sc.video_frame_index(0, len(frames))
        tex = {"still": still, "clip": frames[k]}              # `silent` stays unbound
        got, _ = _run_on_host(tmp_path, f"t{int(time)}", "video", ir=ir, tex=tex, depth=4, attrs={"camera_matrix": IDENTITY})
        want = Oracle(ir, "strict", textures=tex).render(W, H, 4, camera=IDENTITY, camera_scale=1.0)
        assert np.array_equal(_bits(got), _bits(want)), time
        seen.append((k, got))
    assert [k for k, _ in seen] == [0, 1, 2]
    assert not np.array_equal(seen[0][1], seen[1][1]) and not np.array_equal(seen[1][1], seen[2][1])   # the clip plays
    # an unbound video sampler reads (0, 0, 0, 1): the screen is black, the frame around it is not
    ir = _oracle_ir(FIXTURE, "video", time=0.0)
    got, _ = _run_on_host(tmp_path, "unbound", "video", ir=ir, tex={"still": still}, depth=4, attrs={"camera_matrix": IDENTITY})
    want = Oracle(ir, "strict", textures={"still": still}).render(W, H, 4, camera=IDENTITY, camera_scale=1.0)
    assert np.array_equal(_bits(got), _bits(want))
    assert (got[H // 2, W // 2, :3] == 0).all() and got[H // 2, W // 2, 3] == 1 and got[:, :, :3].max() > 0


def test_the_references_video_scene_compiles_now(reference):
    """`boot.dev` was the one reference scene of 82 the generators rejected (`video1_tex` undefined): both front-ends now give
    it four video samplers, the same uniform table, and the sm_100a generator + NVRTC accept the program."""
    from portal_b200.renderer import SceneRenderer
    path = os.path.join(reference, "scenes", "boot.dev.ron")
    ir = _oracle_ir(path, "boot.dev")
    assert [v["name"] for v in ir["videos"]] == ["video1", "video2", "video3", "video4"]
    assert [v["uniform"] for v in ir["videos"]] == [f"video{i}_frame" for i in (1, 2, 3, 4)]
    hs = HostScene.from_file(path)
    assert [v[0] for v in hs.videos()] == ["video1", "video2", "video3", "video4"]
    _assert_same_table(hs.uniform_table(), ir)
    r = SceneRenderer(ir, device=-1)
    assert len(r.cubin()) > 100_000 and "video3_tex" in r.source()
    r.close()
    assert "video3_tex" in HostRenderer(hs, device=-1).source()
