#!/usr/bin/env python
"""Write tests/golden/reference_scenes.tar.xz: every scene file of the reference (optozorax/portal, `scenes/*.ron`) and a
sample of the PNG textures under its `scenes/img`, so that the tests that read the reference's scenes need nothing outside
the repository.  The archive is deterministic (sorted names, zero times and owners).

    python tools/export_reference_scenes.py <reference checkout>
"""
import io
import lzma
import os
import sys
import tarfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "reference_scenes.tar.xz")
# the four 500x500 scene textures (iCCP / pHYs chunks, one to three IDATs) and one 3840x2160 frame in five IDATs; the other
# five images (0.2 - 2.4 MB each) are the same colour type and bit depth
IMAGES = ["border.png", "mobius.png", "mobius_monoportal.png", "monoportal.png", "monoportal_offset.png"]


def main():
    ref = sys.argv[1]
    scenes = os.path.join(ref, "scenes")
    names = sorted(f for f in os.listdir(scenes) if f.endswith(".ron")) + [f"img/{f}" for f in IMAGES]
    buf = io.BytesIO()
    with tarfile.open(fileobj=buf, mode="w", format=tarfile.USTAR_FORMAT) as t:
        for n in names:
            with open(os.path.join(scenes, n), "rb") as f:
                data = f.read()
            info = tarfile.TarInfo(f"scenes/{n}")
            info.size, info.mode, info.mtime = len(data), 0o644, 0
            t.addfile(info, io.BytesIO(data))
    with open(OUT, "wb") as f:
        f.write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))
    print(f"{OUT}: {len(names)} files, {os.path.getsize(OUT)} bytes")


if __name__ == "__main__":
    main()
