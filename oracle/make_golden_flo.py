"""TEST INFRASTRUCTURE — generates tests/golden/flo_24x40.npz with the UNMODIFIED reference's .flo functions
(src/utils/frame_utils.py writeFlow / readFlow, located through ref_shim.REF_ROOT).  Runs only where the reference tree exists.

    python oracle/make_golden_flo.py

The fixture holds the seeded flow field, the bytes the reference's writeFlow puts on disk for it, and what the reference's
readFlow returns for those bytes; tests/test_flo_cpu.py compares gimmvfi_b200.flo against both.
"""
import importlib.util
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import ref_shim  # noqa: E402


def main():
    spec = importlib.util.spec_from_file_location("ref_frame_utils", os.path.join(ref_shim.REF_ROOT, "src", "utils", "frame_utils.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    uv = np.random.default_rng(1).standard_normal((24, 40, 2)).astype(np.float32)
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "ref.flo")
        ref.writeFlow(p, uv)
        raw = np.fromfile(p, np.uint8)
        read = ref.readFlow(p)
    out = os.path.join(ROOT, "tests", "golden", "flo_24x40.npz")
    np.savez_compressed(out, uv=uv, flo_bytes=raw, ref_read=read)
    print(out, raw.size, "bytes")


if __name__ == "__main__":
    main()
