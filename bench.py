#!/usr/bin/env python
"""bench.py -- Mpixels/s of the portal ray loop on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scene S] [--orbit N]
                    [--mode owner|p2p|gather] [--format f32|rgba8] [--frontend ron|ir] [--dump-outputs DIR]

A "step" is one frame of the workload (default: the headline config, portal_in_portal.ron 3840x2160 depth 40, saved
camera, aa 1): uniform-block upload + ONE launch of the scene's sm_100a ray-loop kernel per GPU.
  value   frames timed with CUDA events on the launching stream, scene resident on the GPU(s), float RGBA frames.
          N > 1: the frame is sharded by cyclic 16-row strips (`pe_sharder_*`, C ABI); default mode "owner" -- every rank's
          strips stay in the HBM of the GPU that rendered them (what a consumer then pulls); "p2p" -- every kernel stores
          into rank 0's frame over NVLink; "gather" -- ONE NCCL gather + de-interleave (what north_star names).  The
          rank-0-assembled rates are measured too and reported under `assembled`.
  e2e     the reference-facing call: scene file -> the product's own host front-end (`ph_scene_*`, C++) -> per frame
          float64 scene evaluation + uniform upload (`ph_frame_uniforms`) -> render -> RGBA8 frame in HOST memory
          (`pe_submit_host_rgba8` / `pe_wait_host`; N > 1: `pe_sharder_*` host delivery over every GPU's own PCIe link).
  parity  sha256 of the frames the timed loops produced (value: the last float frame, gathered from the ranks with one
          NCCL gather when N > 1; e2e: the last RGBA8 host frame) against tests/golden/fullsize_sha256.json -- the CPU
          oracle's frames at the full BASELINE.json sizes.
`--impl reference` times the CPU oracle (oracle/, the restatement of the reference's GLSL path -- the reference has no CPU
implementation and cannot be built here, SURVEY.md section 0.1) on the host cores, in a clean subprocess
(oracle/bench_cpu.py), on a bounded sample of the same frame; `cpu_baseline` of the default arm is the same measurement.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SCENE_DIR = os.path.join(ROOT, "tests", "golden", "scenes")
RON_DIR = os.path.join(ROOT, "tests", "golden", "ron")
WORKLOADS = {  # BASELINE.json configs
    "portal_in_portal": (3840, 2160, 40),
    "triple_portal": (3840, 2160, 40),
    "monoportal": (1920, 1080, 20),
    "mobius_monoportal": (7680, 4320, 64),
    "basics": (256, 256, 4),
}
STRIP_ROWS = 16


def metric_name(scene, w, h, depth):
    return f"Mpixels/s @ {w}x{h} depth-{depth} {scene}"


def workload_name(args):
    """One string for both arms (the driver compares them)."""
    return (f"{args.scene}.ron {args.width}x{args.height} depth {args.depth}, " +
            (f"{args.orbit}-frame camera orbit" if args.orbit else "saved camera") + ", aa 1")


def load_ir(scene):
    with open(os.path.join(SCENE_DIR, f"{scene}.scene.json")) as f:
        return json.load(f)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def golden_pins(scene, w, h, depth, orbit=0, k=None):
    """sha256 pins of the oracle's frame for this workload (tests/golden/fullsize_sha256.json), or None."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "fullsize_sha256.json")) as f:
            rec = json.load(f).get(scene)
    except OSError:
        return None
    if not rec:
        return None
    if (rec["width"], rec["height"], rec["depth"]) != (w, h, depth):
        rec = rec.get(f"{w}x{h}")
        if not rec or rec.get("depth") != depth:
            return None
    if orbit:
        return rec.get(f"orbit_{orbit}", {}).get(str(k))
    return rec


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.idx = device_index
        self.proc = None
        self.path = f"/tmp/_pe_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self, t0=None, t1=None, t2=None):
        """t0, t1: wall-clock (time.time()) bounds of the timed region.  If it was too short to contain two samples
        (nvidia-smi cannot sample faster than ~20 ms) the samples up to t2 -- the end of an untimed repeat of the very
        same steps that run_ours() appends in that case -- are used, and failing that everything since start()."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        import datetime
        rows = []
        for line in open(self.path):
            p = [x.strip() for x in line.split(",")]
            if len(p) < 10:
                continue
            try:
                ts = datetime.datetime.strptime(p[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(p[2]), float(p[3]), p[6:10]))
            except ValueError:
                continue
        inside = [r for r in rows if t0 is not None and t0 <= r[0] <= t1]
        window = "timed region"
        if len(inside) < 2 and t2 is not None:
            inside = [r for r in rows if t0 <= r[0] <= t2]
            window = "timed region + untimed repeat of the same steps (timed region shorter than the sampling period)"
        if len(inside) < 2:
            inside, window = rows, "warm-up + timed region (timed region shorter than the sampling period)"
        sm = sorted(r[1] for r in inside)
        reasons = set()
        for r in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": inside[0][2] if inside else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ------------------------------------------------------------------------------ CPU oracle legs
def cpu_oracle(args, budget_s, steps=1, warmup=1, threads=0):
    """The oracle's fast build on a bounded sample of the frame, in a CLEAN subprocess (oracle/bench_cpu.py resets the CPU
    affinity and the OpenMP environment that torchrun narrows).  Returns the parsed JSON line."""
    env = {k: v for k, v in os.environ.items() if not (k.startswith(("OMP_", "KMP_", "GOMP_", "MKL_")) or k == "PORTAL_B200_BENCH_CPU_REEXEC")}
    cmd = [sys.executable, "-m", "oracle.bench_cpu", "--scene", args.scene, "--width", str(args.width), "--height", str(args.height),
           "--depth", str(args.depth), "--budget", str(budget_s), "--steps", str(steps), "--warmup", str(warmup), "--threads", str(threads)]
    p = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    if p.returncode != 0:
        raise RuntimeError("oracle.bench_cpu failed: " + (p.stderr or p.stdout)[-2000:])
    return json.loads(p.stdout.strip().splitlines()[-1])


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w, h, depth = args.width, args.height, args.depth
    t0 = time.perf_counter()
    res = cpu_oracle(args, budget_s=60.0, steps=args.steps, warmup=min(max(args.warmup, 1), 3))
    dt = time.perf_counter() - t0
    v = res["value"]
    print(json.dumps({
        "impl": "reference", "metric": metric_name(args.scene, w, h, depth), "value": round(v, 4), "unit": "Mpixels/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(w * h / (v * 1e6) * 1e3, 3),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args)},
        "cpu_baseline": {"value": round(v, 4), "unit": "Mpixels/s", "cores": res["threads_used"], "kind": "port", "sample": res["sample"]},
        "e2e": {"value": round(v, 4), "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": f"CPU oracle (restatement of the reference's GLSL path; the reference itself has no CPU path), clean subprocess; wall {dt:.1f} s",
    }))


# ------------------------------------------------------------------------------ our arm
def sha(buf) -> str:
    return hashlib.sha256(memoryview(buf).cast("B")).hexdigest()


DUMP_PIXELS = 1 << 20      # --dump-outputs: pixels kept per frame (two frames + their indices: 40 MB of .npy files)


def dump_frame(d, name, frame):
    """--dump-outputs: DIR/<name>.npy = the (h, w, 4) frame's pixels as float32 (n, 4) -- every pixel, or a fixed seeded
    sample of DUMP_PIXELS of them -- and DIR/pixel_index.npy = their row-major indices (float64)."""
    import numpy as np
    n = frame.shape[0] * frame.shape[1]
    idx = np.arange(n) if n <= DUMP_PIXELS else np.sort(np.random.default_rng(0).choice(n, DUMP_PIXELS, replace=False))
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(d, f"{name}.npy"), np.ascontiguousarray(frame).reshape(n, 4)[idx].astype(np.float32))


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from portal_b200 import distributed as D
    from portal_b200.renderer import SceneRenderer, load_textures

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    w, h, depth = args.width, args.height, args.depth
    textures = load_textures(os.path.join(SCENE_DIR, f"{args.scene}.textures.npz"))
    options = {}
    if args.tile_w:
        options["tile_w"] = args.tile_w
    stream = torch.cuda.Stream()          # a real (non-NULL) stream: NULL means "the context's own stream" to the C ABI
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream
    assert sptr != 0

    # ---- the scene: `ron` = the product's own host front-end (RON text -> ph_scene_* -> pe_*), `ir` = the JSON scene IR
    if args.frontend == "ron":
        from portal_b200.host import HostRenderer, HostScene
        hscene = HostScene.from_file(os.path.join(RON_DIR, f"{args.scene}.ron"))
        r = HostRenderer(hscene, device=local, textures=textures, persistent=bool(args.persistent), options=options)
        cam0 = hscene.camera()

        def frame_uniforms(k=None):
            cam = None
            if k is not None:
                cam = dict(cam0, alpha=cam0["alpha"] + 2.0 * math.pi * k / args.orbit)
            r.frame_uniforms(w, h, depth, camera=cam)
    else:
        r = SceneRenderer(load_ir(args.scene), textures=textures, device=local, persistent=bool(args.persistent), options=options)
        r.render_depth = depth
        cam0 = dict(r.cam)

        def frame_uniforms(k=None):
            if k is not None:
                r.set_cam(cam0["look_at"], cam0["alpha"] + 2.0 * math.pi * k / args.orbit, cam0["beta"], cam0["r"])
            r.set_uniforms()
    lib, ctx = r._lib, r._ctx

    def check(rc):
        if rc:
            raise RuntimeError(lib.pe_last_error(ctx).decode(errors="replace"))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value leg set-up
    mode = args.mode if (world > 1 or not args.no_overlap) else "single"
    if world == 1 and mode != "single":
        mode = "owner"                     # one GPU: the same sharder, one rank (so that every N runs the same code)
    fmt = args.format
    bpp = 16 if fmt == "f32" else 4
    tdtype = torch.float32 if fmt == "f32" else torch.uint8
    frame_counter = [0]
    sharder = None
    if mode == "single":
        target = r.full_target(w, h) if hasattr(r, "full_target") else SceneRenderer.full_target(w, h)
        # ring of output frames larger than the 126 MB L2: >= 2 float frames (265 MB at 4K) / >= 6 RGBA8 frames
        n_outs = max(2, int(math.ceil(192e6 / (w * h * bpp))) + 1)
        outs = [torch.empty((h, w, 4), dtype=tdtype, device="cuda") for _ in range(n_outs)]
        n_px_local = w * h
    elif mode == "gather":
        target = D.make_target(w, h, rank, world, STRIP_ROWS, full_frame=False)
        spr = D.strips_per_rank(h, world, STRIP_ROWS)
        n_outs = max(2, int(math.ceil(192e6 / max(spr * STRIP_ROWS * w * 16, 1))) + 1)
        local_bufs = [torch.zeros((spr, STRIP_ROWS, w, 4), dtype=torch.float32, device="cuda") for _ in range(n_outs)]
        gathered = torch.empty((world, spr, STRIP_ROWS, w, 4), dtype=torch.float32, device="cuda") if rank == 0 else None
        frame_dev = torch.empty((h, w, 4), dtype=torch.float32, device="cuda") if rank == 0 else None
        fmt, bpp = "f32", 16
        n_px_local = int(lib.pe_target_pixels(C.byref(target)))
    else:
        sharder = D.NativeSharder(r, w, h, rank, world, mode, fmt, STRIP_ROWS)
        target = sharder.target
        n_px_local = sum(1 for y in D.local_rows(h, rank, world, STRIP_ROWS) if y >= 0) * w
    last = {"ptr": None}
    overlapped = mode == "owner" and not args.no_overlap and not args.persistent

    def render_once(i):
        """Enqueue one frame (this rank's part of it) on the stream."""
        if mode == "single":
            out = outs[i % len(outs)]
            check(lib.pe_render(ctx, C.byref(target), out.data_ptr(), None, sptr) if fmt == "f32" else
                  lib.pe_render_rgba8(ctx, C.byref(target), out.data_ptr(), sptr))
            last["ptr"] = out
        elif mode == "gather":
            out = local_bufs[i % len(local_bufs)]
            check(lib.pe_render(ctx, C.byref(target), out.data_ptr(), None, sptr))
            dist.gather(out, list(gathered.unbind(0)) if rank == 0 else None, dst=0)       # torch's current stream == `stream`
            if rank == 0:
                check(lib.pe_deinterleave_strips(ctx, gathered.data_ptr(), frame_dev.data_ptr(), w, h, STRIP_ROWS, world, spr, sptr))
            last["ptr"] = out
        elif overlapped:
            sharder.render_overlapped(sptr)    # two frames in flight: the tail of one runs under the head of the next
        else:
            last["ptr"] = sharder.render(sptr)
            sharder.release(sptr)              # p2p, rank 0: the frame's consumer (nothing, here) has been enqueued

    def step(i):
        if args.orbit:
            # BASELINE config 5: alpha_k = alpha_0 + 2*pi*k/orbit (SURVEY.md section 8d); only `_camera` changes
            frame_uniforms(frame_counter[0] % args.orbit)
            frame_counter[0] += 1
        render_once(i)

    frame_uniforms(0 if args.orbit else None)
    # ---- per-scene autotuning (pe_autotune): block size 512 / 1024 x canonical rays on / off, same pixels, timed on this
    # rank's own part of the frame; untimed set-up, like the scene compilation itself
    tuned = None
    if not args.no_autotune and not args.persistent:
        tt = D.make_target(w, h, rank, world, STRIP_ROWS, full_frame=False) if mode != "single" else target
        if tt.n_strips > 0:
            buf = C.create_string_buffer(2048)
            check(lib.pe_autotune(ctx, C.byref(tt), 5, buf, len(buf)))
            tuned = buf.value.decode().strip().splitlines()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                      # nvidia-smi needs ~0.2 s to produce its first sample: start it early
    for i in range(max(args.warmup, 3)):
        step(i)
    barrier()
    frame_counter[0] = 0
    # ---- timed region: K steps, device time, max over ranks
    l0 = int(lib.pe_launch_count(ctx))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_epoch0 = time.time()
    ev[0].record(stream)
    for i in range(args.steps):
        kev[i][0].record(stream)
        step(i)
        kev[i][1].record(stream)
    if overlapped:
        last["ptr"] = sharder.flush(sptr)      # the stream now waits for the frames still in flight: they are inside the timed region
    ev[1].record(stream)
    barrier()
    t_epoch1 = time.time()
    launches = torch.tensor([int(lib.pe_launch_count(ctx)) - l0], dtype=torch.int64, device="cuda")
    ms = torch.tensor([ev[0].elapsed_time(ev[1])], dtype=torch.float64, device="cuda")
    kms = torch.tensor([sum(a.elapsed_time(b) for a, b in kev) / args.steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(kms, op=dist.ReduceOp.MAX)
        dist.all_reduce(launches, op=dist.ReduceOp.SUM)        # every rank's kernels count
    total_ms, kernel_ms = float(ms.item()), float(kms.item())
    if overlapped:
        kernel_ms = total_ms / args.steps      # launches overlap: per-launch events mean nothing, the frame period does

    # ---- parity of the value leg: the LAST frame the timed loop produced, hashed against the oracle's pin.  A camera orbit has
    # pins for frames 0 and orbit / 2 only: those two are rendered once more, untimed, through the very same step.
    last_k = (args.steps - 1) % args.orbit if args.orbit else None
    parity = {}

    def assembled_last_frame():
        """bytes of the whole last frame on rank 0 (None elsewhere)."""
        if mode == "single":
            return last["ptr"].cpu().numpy()
        if world == 1:                     # the sharder's buffer of the one rank IS the frame
            out = np.empty((h, w, 4), dtype=np.float32 if fmt == "f32" else np.uint8)
            check(lib.pe_memcpy_d2h(ctx, out.ctypes.data, last["ptr"], out.nbytes, sptr))
            return out
        if mode == "gather":
            return frame_dev.cpu().numpy() if rank == 0 else None
        if mode == "p2p":
            if rank != 0:
                return None
            out = np.empty((h, w, 4), dtype=np.float32 if fmt == "f32" else np.uint8)
            check(lib.pe_memcpy_d2h(ctx, out.ctypes.data, last["ptr"], out.nbytes, sptr))
            return out
        # owner: ONE NCCL gather of every rank's strips (exactly the buffers the last timed step wrote) + de-interleave
        spr_ = D.strips_per_rank(h, world, STRIP_ROWS)
        mine = torch.zeros((spr_, STRIP_ROWS, w, 4), dtype=tdtype, device="cuda")
        nb = n_px_local * bpp
        if nb:
            # device-to-device: the sharder's buffer (a raw device pointer of the C ABI) seen as a tensor
            class _DevBuf:
                __cuda_array_interface__ = {"shape": (nb,), "typestr": "|u1", "data": (int(last["ptr"]), False), "version": 3}
            mine.view(torch.uint8).reshape(-1)[:nb].copy_(torch.as_tensor(_DevBuf(), device="cuda"))
        g = torch.empty((world,) + tuple(mine.shape), dtype=tdtype, device="cuda") if rank == 0 else None
        dist.gather(mine, list(g.unbind(0)) if rank == 0 else None, dst=0)
        if rank != 0:
            return None
        if fmt == "f32":
            fr = torch.empty((h, w, 4), dtype=torch.float32, device="cuda")
            check(lib.pe_deinterleave_strips(ctx, g.data_ptr(), fr.data_ptr(), w, h, STRIP_ROWS, world, spr_, sptr))
            torch.cuda.synchronize()
            return fr.cpu().numpy()
        return D.deinterleave_numpy(g.cpu().numpy(), h, world, STRIP_ROWS)

    def hash_value_frame(k):
        frame = assembled_last_frame()
        if rank != 0:
            return None
        pins = golden_pins(args.scene, w, h, depth, args.orbit, k)
        key = "sha256_f32_rgba" if fmt == "f32" else "sha256_rgba8"
        got = sha(np.ascontiguousarray(frame))
        how = "as rendered" if world == 1 else ("every rank's strips through one NCCL gather" if mode == "owner" else "assembled on rank 0")
        return {"what": f"{'orbit frame %d' % k if args.orbit else 'last timed frame, saved camera'}, {fmt}, {how}", "sha256": got,
                "golden": pins.get(key) if pins else None, "match": (got == pins.get(key)) if pins and pins.get(key) else None}

    if args.dump_outputs:
        frame = assembled_last_frame()          # every rank takes part: owner mode gathers the strips on rank 0
        if rank == 0:
            dump_frame(args.dump_outputs, f"frame_{fmt}", frame)
        del frame
    if not args.orbit:
        rec = hash_value_frame(None)
        if rank == 0:
            parity["value_frame"] = rec
    else:
        recs = []
        for k in (0, args.orbit // 2):
            frame_counter[0] = k
            step(args.steps + k)
            if overlapped:
                last["ptr"] = sharder.flush(sptr)
            barrier()
            recs.append(hash_value_frame(k))
        if rank == 0:
            parity["value_frame"] = {"what": "orbit frames rendered once more (untimed) by the timed step", "frames": recs,
                                     "match": all(r["match"] for r in recs) if all(r["match"] is not None for r in recs) else None}

    # A timed region of a few tens of ms (many GPUs, short frames) ends before nvidia-smi delivers two samples: keep the
    # GPUs under the identical load, untimed, for ~1.5 s so that the clocks / throttle reasons are observed under it.
    if total_ms < 100.0:
        extra = max(1, min(50000, int(1500.0 / max(total_ms / args.steps, 1e-3))))
        for i in range(extra):
            step(args.steps + i)
        barrier()
    clocks = sampler.stop(t_epoch0, t_epoch1, time.time()) if rank == 0 else None
    if sharder is not None:
        barrier()
        sharder.close()
        sharder = None

    # ---- N > 1: the same frames ASSEMBLED on rank 0 by the render kernels' own NVLink stores (float and RGBA8 frames)
    assembled = None
    if world > 1 and not args.no_assembled:
        assembled = {}
        for afmt in ("f32", "rgba8"):
            sh = D.NativeSharder(r, w, h, rank, world, "p2p", afmt, STRIP_ROWS)
            n = min(args.steps, 100)
            for _ in range(3):
                sh.render(sptr); sh.release(sptr)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(n):
                sh.render(sptr); sh.release(sptr)
            e1.record(stream)
            barrier()
            t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            rec = {"value": round(w * h * n / (float(t.item()) * 1e-3) / 1e6, 2), "unit": "Mpixels/s", "steps": n}
            if rank == 0 and not args.orbit:
                out = np.empty((h, w, 4), dtype=np.float32 if afmt == "f32" else np.uint8)
                check(lib.pe_memcpy_d2h(ctx, out.ctypes.data, sh.frame_ptr, out.nbytes, sptr))
                pins = golden_pins(args.scene, w, h, depth)
                key = "sha256_f32_rgba" if afmt == "f32" else "sha256_rgba8"
                rec["frame_matches_golden"] = (sha(out) == pins[key]) if pins and key in pins else None
            assembled[f"p2p_{afmt}"] = rec
            barrier()
            sh.close()

    # ---- e2e: the reference-facing call with HOST buffers (RGBA8 frame = get_texture_data), per-frame host work included
    e2e_steps = args.steps          # filling and draining the pipeline (one kernel + one copy) costs about one frame of the loop
    e2e_k = [0]

    def e2e_uniforms():
        k = None
        if args.orbit:
            k = e2e_k[0] % args.orbit
        e2e_k[0] += 1
        frame_uniforms(k)                     # ron: float64 scene evaluation + upload; ir: camera -> `_camera` + upload
        return k

    e2e_sync_rate = None
    e2e_last_k = None
    if world == 1:
        with D.gpu_numa_affinity(local):      # pinned pages on the GPU's NUMA node: the D2H copy stays off the socket interconnect
            ring = [torch.empty((h, w, 4), dtype=torch.uint8).pin_memory() for _ in range(2)]
        t8 = SceneRenderer.full_target(w, h)

        def blocking(n):
            for _ in range(n):
                e2e_uniforms()
                check(lib.pe_render_host_rgba8(ctx, C.byref(t8), ring[0].data_ptr()))

        def pipelined(n):
            prev, k = None, None
            for i in range(n):
                k = e2e_uniforms()
                tk = C.c_uint64()
                check(lib.pe_submit_host_rgba8(ctx, C.byref(t8), ring[i % 2].data_ptr(), C.byref(tk)))
                if prev is not None:
                    check(lib.pe_wait_host(ctx, prev))     # frame i-1 is in host memory: the consumer may read it now
                prev = tk.value
            check(lib.pe_wait_host(ctx, prev))
            return k, ring[(n - 1) % 2]
        blocking(2)
        t0 = time.perf_counter()
        blocking(e2e_steps)
        e2e_sync_rate = w * h * e2e_steps / (time.perf_counter() - t0) / 1e6
        pipelined(3)
        check(lib.pe_sync(ctx))
        e2e_k[0] = (args.orbit // 2 - (e2e_steps - 1)) if args.orbit else 0      # an orbit's e2e loop ends on pinned frame orbit / 2
        t0 = time.perf_counter()
        e2e_last_k, host_frame = pipelined(e2e_steps)
        e2e_rate = w * h * e2e_steps / (time.perf_counter() - t0) / 1e6
        host_bytes = host_frame.numpy()
    else:
        hs = D.NativeSharder(r, w, h, rank, world, "host", "rgba8", STRIP_ROWS)

        LAG = D.NativeSharder.PIPELINE_DEPTH - 1     # a rank keeps this many frames in flight behind the one it submits

        prof = {"uniforms": 0.0, "submit": 0.0, "complete": 0.0, "wait_frame": 0.0}
        debug = bool(os.environ.get("PORTAL_B200_DEBUG"))

        def pipelined_n(n):
            k, fr, done = None, None, 0

            def finish(f, last):
                t_ = time.perf_counter()
                hs.complete(f)
                prof["complete"] += time.perf_counter() - t_
                if rank == 0:
                    t_ = time.perf_counter()
                    v = hs.wait_frame(f, view=last)          # the whole frame f is in host memory: the consumer may read it
                    prof["wait_frame"] += time.perf_counter() - t_
                    if last:
                        return (v, f)                        # held, not released: the checker hashes it after the clock has stopped
                    hs.release_frame(f)
                return None
            first = None
            for i in range(n):
                t_ = time.perf_counter()
                k = e2e_uniforms()
                t1_ = time.perf_counter()
                f = hs.submit()
                prof["uniforms"] += t1_ - t_
                prof["submit"] += time.perf_counter() - t1_
                if first is None:
                    first = f
                if i >= LAG:
                    finish(first + done, False)
                    done += 1
            while done < n:
                fr = finish(first + done, done == n - 1)
                done += 1
            return k, fr
        held = pipelined_n(2 * LAG + 2)[1]
        if rank == 0:
            hs.release_frame(held[1])
        barrier()
        e2e_k[0] = (args.orbit // 2 - (e2e_steps - 1)) if args.orbit else 0      # an orbit's e2e loop ends on pinned frame orbit / 2
        t0 = time.perf_counter()
        e2e_last_k, held = pipelined_n(e2e_steps)
        barrier()
        e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        e2e_rate = w * h * e2e_steps / float(e2e_s.item()) / 1e6
        host_bytes = None
        if rank == 0:                      # outside the timed region: a private copy of the delivered frame for the hash, then its slot is released
            host_bytes = held[0].copy()
            hs.release_frame(held[1])
        if debug:
            print(f"[bench] rank {rank}: e2e host time per frame (us): " + ", ".join(f"{k} {v / (e2e_steps + 2 * LAG + 2) * 1e6:.0f}" for k, v in prof.items()) +
                  f"; period {float(e2e_s.item()) / e2e_steps * 1e6:.0f}", file=sys.stderr, flush=True)
        barrier()
        hs.close()
    if rank == 0:
        if args.dump_outputs:
            dump_frame(args.dump_outputs, "e2e_frame_rgba8", host_bytes)
        pins = golden_pins(args.scene, w, h, depth, args.orbit, e2e_last_k)
        got = sha(np.ascontiguousarray(host_bytes))
        parity["e2e_frame"] = {"what": "last RGBA8 frame delivered to host memory by the e2e loop", "sha256": got,
                               "golden": pins.get("sha256_rgba8") if pins else None,
                               "match": (got == pins.get("sha256_rgba8")) if pins and pins.get("sha256_rgba8") else None}

    if rank == 0:
        peaks, peak_src = measured_peaks()
        value = w * h * args.steps / (total_ms * 1e-3) / 1e6
        # roofline of the dominant kernel (pe_render_kernel): algorithmic bytes = 16 B/pixel written
        # (SURVEY.md section 8d) x pixels one launch shades, / its mean launch duration (CUDA events)
        alg_bytes = float(bpp) * n_px_local
        achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp) and world == 1 and not args.orbit:
            with open(tp) as f:
                traffic = json.load(f).get(f"{args.scene}_{w}x{h}_d{depth}") if fmt == "f32" else None
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            res = cpu_oracle(args, budget_s=15.0, steps=0)       # about 15 s of wall on all host threads: whole passes over the frame when one is shorter
            res1 = cpu_oracle(args, budget_s=4.0, threads=1)
            cpu = {"value": round(res["value"], 4), "unit": "Mpixels/s", "cores": res["threads_used"], "kind": "port", "sample": res["sample"],
                   "single_thread_value": round(res1["value"], 4)}
        par = {"single": "1 GPU",
               "owner": f"{world} GPU{'s' if world > 1 else ''} x cyclic {STRIP_ROWS}-row strips (pe_sharder_*, C ABI), every rank's strips stay in its own HBM; no collective on the data path" +
                        ("; two frames in flight per GPU (alternating streams and program instances) so that a frame's last wave overlaps the next frame's first" if overlapped else ""),
               "p2p": f"{world} GPUs x cyclic {STRIP_ROWS}-row strips, kernels store into rank 0's frame over NVLink (CUDA IPC), stream-ordered flag words, no collective",
               "gather": f"{world} GPUs x cyclic {STRIP_ROWS}-row strips + 1 NCCL gather + de-interleave"}[mode]
        frame_mb = w * h * bpp / 1e6
        line = {
            "metric": metric_name(args.scene, w, h, depth), "value": round(value, 2), "unit": "Mpixels/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": round(total_ms / args.steps, 4), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args),
                       "parallelism": par,
                       "scheduler": "persistent warps + per-bounce refill" if args.persistent else
                                    f"one thread per pixel, {args.tile_w or 8}x{32 // (args.tile_w or 8)} warp tiles, <= 64 regs; " +
                                    (f"pe_autotune on rank 0: {tuned[-1]}" if tuned else "512-thread blocks, canonical rays (no autotune)"),
                       "autotune": tuned,
                       "frame_format": "float RGBA (16 B/pixel)" if fmt == "f32" else "RGBA8 quantised by the kernel (4 B/pixel)",
                       "front_end": "scene .ron -> C++ host front-end (ph_scene_*) -> C ABI" if args.frontend == "ron" else "JSON scene IR -> Python SceneRenderer -> C ABI",
                       "l2": f"each step writes {'a' if world == 1 else 'its part of a'} {frame_mb:.1f} MB frame into a ring of buffers larger than "
                             f"the 126 MB L2; inputs are a <8 KB constant block"},
            "kernel_ms": round(kernel_ms, 4),
            "roofline": {"bound": "hbm", "achieved": round(achieved, 2), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": round(achieved / peaks["hbm_gbs"], 5), "traffic": traffic, "peak_source": peak_src,
                         "note": f"{int(bpp)} B/pixel algorithmic x {n_px_local} px per launch; the loop is fp32-issue bound (DESIGN.md section 6): "
                                 f"issue-slot utilisation and instructions per pixel are in profiles/"},
            "clocks": clocks,
            "e2e": {"value": round(e2e_rate, 2), "unit": "Mpixels/s", "h2d_bytes_per_step": e2e_h2d_bytes(r) * world,
                    "d2h_bytes_per_step": w * h * 4, "steps": e2e_steps,
                    "call": ("ph_frame_uniforms + " if args.frontend == "ron" else "set_cam/set_uniforms + ") +
                            ("pe_submit_host_rgba8 / pe_wait_host per frame (RGBA8 into pinned host memory, 2 frames in flight)" if world == 1 else
                             f"pe_sharder_submit / complete on every rank, wait_frame / release_frame on rank 0: RGBA8 strips over {world} PCIe links "
                             f"into one shared pinned host frame, no gather")},
            "parity": parity,
            "gpu_launches": int(launches.item()),
        }
        if e2e_sync_rate is not None:
            line["e2e"]["sync_call_value"] = round(e2e_sync_rate, 2)
            line["e2e"]["sync_call"] = "pe_render_host_rgba8 (one blocking call per frame)"
        if assembled:
            line["assembled"] = assembled
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    r.close()


def e2e_h2d_bytes(r):
    """Bytes of the constant uniform block uploaded every step (scene matrices + camera + scalars)."""
    import re
    src = r.source()
    m = re.search(r"sizeof\(PeConstBlock\) == (\d+)", src)
    return int(m.group(1)) if m else 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scene", default="portal_in_portal")
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--depth", type=int, default=0)
    ap.add_argument("--persistent", type=int, default=0)
    ap.add_argument("--tile-w", type=int, default=0, choices=[0, 8, 16, 32], help="warp tile width (0: the library default, 8)")
    ap.add_argument("--orbit", type=int, default=0, help="camera orbit of this many frames per turn (config 5: 360)")
    ap.add_argument("--mode", default="owner", choices=["owner", "p2p", "gather"],
                    help="N > 1, the timed `value` steps: owner = strips stay in the rendering GPU's HBM; p2p = kernels store into rank 0's "
                         "frame over NVLink; gather = one NCCL gather + de-interleave")
    ap.add_argument("--frontend", default="ron", choices=["ron", "ir"],
                    help="ron = the product's C++ host front-end on tests/golden/ron/<scene>.ron; ir = the JSON scene IR (oracle front-end's export)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-autotune", action="store_true", help="keep the library defaults (512-thread blocks, canonical rays) instead of pe_autotune")
    ap.add_argument("--no-overlap", action="store_true", help="N > 1, owner mode: one frame in flight per GPU instead of two")
    ap.add_argument("--no-assembled", action="store_true", help="N > 1: skip the extra rank-0-assembled measurements")
    ap.add_argument("--format", default="f32", choices=["f32", "rgba8"],
                    help="frame format of the timed steps: f32 = float RGBA, 16 B/pixel (the metric's definition, SURVEY.md 8d); "
                         "rgba8 = what the reference's RGBA8 render target holds, 4 B/pixel, quantised by the kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last frame of the timed loop (frame_<format>.npy) and the last host "
                         "RGBA8 frame of the e2e loop (e2e_frame_rgba8.npy) to DIR as float32 (n, 4) arrays: every pixel, or a "
                         f"fixed seeded sample of {DUMP_PIXELS} pixels whose row-major indices are in pixel_index.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm renders a sample of the frame in a subprocess; it dumps nothing")
    w, h, d = WORKLOADS[args.scene]
    args.width, args.height, args.depth = args.width or w, args.height or h, args.depth or d
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
