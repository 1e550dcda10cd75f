"""The per-stream lifecycle entry points (reset, retune, capture detach / attach) are part of the published ABI: declared in
navtex_b200.h and listed in engine.EXPORTS, which test_abi checks against the built library.  No GPU needed."""
import os
import re

from navtex_b200 import engine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("nvx_engine_reset_streams", "nvx_engine_retune_stream", "nvx_capture_detach", "nvx_capture_attach")


def test_lifecycle_entry_points_are_declared_and_exported():
    with open(os.path.join(ROOT, "include", "navtex_b200.h")) as f:
        header = f.read()
    for name in NAMES:
        assert name in engine.EXPORTS, name
        assert re.search(r"\bint " + name + r"\(", header), name
