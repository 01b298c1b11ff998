import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
SCENES = ["basics", "monoportal", "triple_portal", "portal_in_portal", "mobius_monoportal"]
# depth per BASELINE.json config
DEPTH = {"basics": 4, "monoportal": 20, "triple_portal": 40, "portal_in_portal": 40, "mobius_monoportal": 64}
# Oracle and kernel share one pinned numeric profile, transcendentals included (DESIGN.md section 4): every
# config scene must agree bit for bit.  (exp/log/pow would be the exception; no config scene calls them.)
BIT_EXACT = ["basics", "monoportal", "triple_portal", "portal_in_portal", "mobius_monoportal"]
# The reference's scene files (every scenes/*.ron) and a sample of its scenes/img textures (tools/export_reference_scenes.py)
REFERENCE_ARCHIVE = os.path.join(GOLDEN, "reference_scenes.tar.xz")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    # On a machine without a GPU the tests JIT many program variants that no GPU run will ever ask for (option sweeps,
    # synthetic snippets): keep them out of portal_b200/_cache, which build() fills for the config scenes and which travels
    # to the GPU box with the repository snapshot.
    if not os.path.exists("/dev/nvidiactl") and "PORTAL_B200_CACHE_DIR" not in os.environ:
        scratch = os.path.join("/tmp", f"portal_b200_cache_cpu_tests_{os.getuid()}")
        os.environ["PORTAL_B200_CACHE_DIR"] = scratch
        # ... seeded with what build() already compiled, so a fresh machine does not JIT those programs twice
        shipped = os.path.join(ROOT, "portal_b200", "_cache")
        if os.path.isdir(shipped):
            import shutil
            os.makedirs(scratch, exist_ok=True)
            for f in os.listdir(shipped):
                if not os.path.exists(os.path.join(scratch, f)):
                    shutil.copy2(os.path.join(shipped, f), os.path.join(scratch, f))


def load_ir(name):
    with open(os.path.join(GOLDEN, "scenes", f"{name}.scene.json")) as f:
        return json.load(f)


def load_tex(name):
    p = os.path.join(GOLDEN, "scenes", f"{name}.textures.npz")
    if not os.path.exists(p):
        return {}
    with np.load(p) as z:
        return {k: np.ascontiguousarray(z[k]) for k in z.files}


@pytest.fixture(scope="session")
def reference(tmp_path_factory):
    """A directory laid out like the reference checkout: scenes/*.ron and scenes/img/*.png, unpacked from REFERENCE_ARCHIVE."""
    import tarfile
    d = tmp_path_factory.mktemp("reference")
    with tarfile.open(REFERENCE_ARCHIVE) as t:
        t.extractall(d, filter="data")
    return str(d)


@pytest.fixture(scope="session", autouse=True)
def _built_library():
    """Everything (CPU and GPU tests) talks to the in-tree libportal_b200.so."""
    from portal_b200 import build
    build.build()
    return True


@pytest.fixture(scope="session")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch
