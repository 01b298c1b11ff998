"""The PNG codec either side of the path (portal_b200/csrc/host/ph_png.cpp, through the C ABI ph_png_*): textures reach the
reference as PNG files (Texture2D::from_file_with_format, src/main.rs:1066-1085), frames leave as PNG (Image::export_png,
src/main.rs:2939-2943).  The image has no libpng / zlib for C++, so the codec is written out; here Python's zlib and PIL are the
independent checkers: our encoder's files decode to the same pixels in PIL, PIL's files -- every colour type, bit depth,
compression level (stored / fixed / dynamic Huffman blocks) and filter choice PIL produces -- decode to PIL's RGBA pixels in
ours, so do the reference's scenes/img textures (five of its ten are stored), and damaged files are refused with a message,
never a crash."""
import ctypes as C
import io
import os
import zlib

import numpy as np
import pytest
from PIL import Image

Image.MAX_IMAGE_PIXELS = None

from portal_b200 import capi
from portal_b200.capi import PortalB200Error
from portal_b200.host import png_decode, png_encode


def _pil_png(img, **kw):
    buf = io.BytesIO()
    img.save(buf, format="PNG", **kw)
    return buf.getvalue()


def _rgba(rng, h, w, kind):
    if kind == "noise":
        return rng.integers(0, 256, size=(h, w, 4), dtype=np.uint8)
    if kind == "flat":
        return np.full((h, w, 4), 200, np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]                      # smooth gradients + a repeated tile: long matches, every filter type useful
    return np.stack([(xx * 3) % 256, (yy * 5) % 256, ((xx // 8 + yy // 8) % 2) * 255, 255 - (xx + yy) % 256], axis=-1).astype(np.uint8)


@pytest.mark.parametrize("kind", ["noise", "flat", "gradient"])
def test_encoder_output_is_a_png_pil_reads_back_exactly(kind):
    rng = np.random.default_rng(1)
    for h, w in ((1, 1), (3, 5), (64, 64), (90, 160), (257, 33)):
        px = _rgba(rng, h, w, kind)
        data = png_encode(px)
        back = np.asarray(Image.open(io.BytesIO(data)).convert("RGBA"))
        assert Image.open(io.BytesIO(data)).mode == "RGBA" and np.array_equal(back, px), (kind, h, w)
        assert np.array_equal(png_decode(data), px)                      # and our decoder reads our encoder
    big = _rgba(rng, 270, 480, "gradient")
    assert len(png_encode(big)) < big.nbytes // 4                        # LZ77 + filters do compress a rendered-looking frame


def test_decoder_reads_what_pil_writes_in_every_format():
    rng = np.random.default_rng(2)
    base = _rgba(rng, 37, 53, "gradient")
    base[::3, ::2, :3] = rng.integers(0, 256, size=base[::3, ::2, :3].shape, dtype=np.uint8)
    rgba = Image.fromarray(base, "RGBA")
    images = {
        "RGBA": rgba, "RGB": rgba.convert("RGB"), "L": rgba.convert("L"), "LA": rgba.convert("LA"),
        "P": rgba.convert("RGB").quantize(colors=200), "P16": rgba.convert("RGB").quantize(colors=16),
        "P4": rgba.convert("RGB").quantize(colors=4), "P2": rgba.convert("RGB").quantize(colors=2), "1": rgba.convert("1"),
    }
    ptrans = rgba.convert("RGB").quantize(colors=64)
    for name, img in images.items():
        for level in (0, 1, 6, 9):                       # 0 = stored blocks, 1 = mostly fixed codes, 6 / 9 = dynamic codes
            for optimize in (False, True):
                data = _pil_png(img, compress_level=level, optimize=optimize)
                want = np.asarray(Image.open(io.BytesIO(data)).convert("RGBA"))
                assert np.array_equal(png_decode(data), want), (name, level, optimize)
    # transparency chunks: palette alpha, grey key, RGB key
    for name, img, kw in (("P+tRNS", ptrans, {"transparency": bytes(range(0, 256, 4))}), ("L+tRNS", images["L"], {"transparency": int(np.asarray(images["L"])[5, 7])}),
                          ("RGB+tRNS", images["RGB"], {"transparency": tuple(int(v) for v in np.asarray(images["RGB"])[4, 9])})):
        data = _pil_png(img, **kw)
        want = np.asarray(Image.open(io.BytesIO(data)).convert("RGBA"))
        got = png_decode(data)
        assert np.array_equal(got, want), name
        assert (got[..., 3] < 255).any(), name


def test_zlib_streams_against_pythons_zlib():
    lib = capi.lib()
    rng = np.random.default_rng(3)
    for n in (0, 1, 2, 3, 100, 70_000, 300_000):
        for kind in ("noise", "runs", "text"):
            raw = (rng.integers(0, 256, n, dtype=np.uint8) if kind == "noise" else
                   np.repeat(rng.integers(0, 256, n // 50 + 1, dtype=np.uint8), 50)[:n] if kind == "runs" else
                   np.frombuffer((b"the quick brown fox jumps over the lazy dog; " * (n // 40 + 1))[:n], dtype=np.uint8)).tobytes()
            # our encoder's stream, wrapped in a one-row-per-4-bytes PNG, is covered above; here the raw zlib layer through PNG IDAT:
            w = max(1, n // 4)
            if n % 4 == 0 and n:
                px = np.frombuffer(raw, dtype=np.uint8).reshape(1, w, 4)
                data = png_encode(px)
                idat, pos = b"", 8
                while pos < len(data):
                    ln = int.from_bytes(data[pos:pos + 4], "big")
                    if data[pos + 4:pos + 8] == b"IDAT":
                        idat += data[pos + 8:pos + 8 + ln]
                    assert zlib.crc32(data[pos + 4:pos + 8 + ln]) == int.from_bytes(data[pos + 8 + ln:pos + 12 + ln], "big")
                    pos += 12 + ln
                assert len(zlib.decompress(idat)) == n + 1                      # Python's inflate accepts our deflate: filter byte + row


def test_reference_textures_decode_like_pil(reference):
    img = os.path.join(reference, "scenes", "img")
    names = sorted(n for n in os.listdir(img) if n.endswith(".png"))
    assert len(names) == 5
    for name in names:
        data = open(os.path.join(img, name), "rb").read()
        want = np.asarray(Image.open(io.BytesIO(data)).convert("RGBA"))
        assert np.array_equal(png_decode(data), want), name


def test_damaged_files_are_refused_with_a_message():
    rng = np.random.default_rng(4)
    good = _pil_png(Image.fromarray(_rgba(rng, 20, 30, "gradient"), "RGBA"), compress_level=6)
    for bad, what in ((b"", "signature"), (good[:7], "signature"), (b"JFIF" + good[4:], "signature"), (good[:40], "IEND"),
                      (good[:-12], "IEND"), (good[:60] + bytes([good[60] ^ 0x55]) + good[61:], "CRC")):
        with pytest.raises(PortalB200Error) as e:
            png_decode(bad)
        assert what in str(e.value), (what, str(e.value))
    # interlaced and 16-bit files: refused by name, not mis-decoded
    with pytest.raises(PortalB200Error, match="interlaced"):
        png_decode(_fix_crc(good[:28] + b"\x01" + good[29:]))
    arr16 = (rng.integers(0, 65536, size=(4, 4), dtype=np.uint16))
    with pytest.raises(PortalB200Error, match="16-bit"):
        png_decode(_pil_png(Image.fromarray(arr16)))
    # fuzz: random single-byte damage anywhere never crashes the process; it either still decodes or raises
    for _ in range(300):
        b = bytearray(good)
        k = int(rng.integers(0, len(b)))
        b[k] ^= int(rng.integers(1, 256))
        try:
            out = png_decode(bytes(b))
            assert out.shape[2] == 4
        except PortalB200Error:
            pass
    for cut in range(0, len(good), 7):
        try:
            png_decode(good[:cut])
        except PortalB200Error:
            pass


def _fix_crc(data: bytes) -> bytes:
    """Recompute every chunk's CRC (after an intentional header edit)."""
    out, pos = bytearray(data[:8]), 8
    while pos + 12 <= len(data):
        ln = int.from_bytes(data[pos:pos + 4], "big")
        body = data[pos + 4:pos + 8 + ln]
        out += data[pos:pos + 4] + body + zlib.crc32(body).to_bytes(4, "big")
        pos += 12 + ln
    return bytes(out)


def test_video_frames_dir_rule():
    lib = capi.lib()
    buf = C.create_string_buffer(256)
    for path, want in (("video1.mov", "video_png/video1"), ("clips/intro.final.mp4", "video_png/intro.final"), ("a/b/c", "video_png/c"),
                       ("x/.hidden", "video_png/.hidden"), ("dir/", "video_png/dir"), ("", "")):
        n = lib.ph_video_frames_dir(path.encode(), buf, len(buf))
        assert buf.value.decode() == want and n == len(want), path


def test_codec_survives_damage_under_sanitizers(tmp_path):
    """tests/host_harness/sanitize_png.cpp built with AddressSanitizer + UndefinedBehaviorSanitizer: round trips, every prefix
    and thousands of mutated files (chunk CRCs repaired, so the damage reaches inflate / filters / palettes) -- no report."""
    import subprocess
    from conftest import ROOT
    host = os.path.join(ROOT, "portal_b200", "csrc", "host")
    exe = str(tmp_path / "sanitize_png")
    cc = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-omit-frame-pointer", "-I", host,
                         os.path.join(ROOT, "tests", "host_harness", "sanitize_png.cpp"), os.path.join(host, "ph_png.cpp"), "-o", exe],
                        capture_output=True, text=True, timeout=600)
    assert cc.returncode == 0, cc.stderr[-3000:]
    run = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert run.returncode == 0 and "no crash" in run.stdout and "runtime error" not in run.stderr and "AddressSanitizer" not in run.stderr, (run.stdout + run.stderr)[-3000:]
