"""`.flo` IO (src/utils/frame_utils.py:24-44, :84-113): byte-identical files and values vs the reference's own functions."""
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR
from gimmvfi_b200.flo import flo_to_tensor, read_flo, write_flo


def test_flo_round_trip_and_format(tmp_path):
    rng = np.random.default_rng(0)
    uv = rng.standard_normal((37, 53, 2)).astype(np.float32) * 7
    p = tmp_path / "a.flo"
    write_flo(p, uv)
    raw = open(p, "rb").read()
    assert len(raw) == 12 + 37 * 53 * 2 * 4
    assert np.frombuffer(raw[:4], "<f4")[0] == np.float32(202021.25) and tuple(np.frombuffer(raw[4:12], "<i4")) == (53, 37)
    assert np.array_equal(read_flo(p), uv)
    t = flo_to_tensor(p)
    assert tuple(t.shape) == (1, 2, 37, 53) and np.array_equal(t[0, 0].numpy(), uv[..., 0])
    write_flo(tmp_path / "b.flo", uv[..., 0], uv[..., 1])                      # (u, v) form
    assert open(tmp_path / "b.flo", "rb").read() == raw
    open(tmp_path / "bad.flo", "wb").write(b"\x00" * 20)
    with pytest.raises(ValueError):
        read_flo(tmp_path / "bad.flo")
    open(tmp_path / "short.flo", "wb").write(raw[:100])
    with pytest.raises(ValueError):
        read_flo(tmp_path / "short.flo")


def test_flo_matches_reference_functions(tmp_path):
    """tests/golden/flo_24x40.npz (oracle/make_golden_flo.py): the bytes the reference's writeFlow wrote for a seeded field and what
    its readFlow returned for them."""
    g = np.load(os.path.join(GOLDEN_DIR, "flo_24x40.npz"))
    uv = np.random.default_rng(1).standard_normal((24, 40, 2)).astype(np.float32)
    assert np.array_equal(uv, g["uv"])
    write_flo(tmp_path / "ours.flo", uv)
    assert open(tmp_path / "ours.flo", "rb").read() == g["flo_bytes"].tobytes()
    (tmp_path / "ref.flo").write_bytes(g["flo_bytes"].tobytes())
    assert np.array_equal(g["ref_read"], read_flo(tmp_path / "ref.flo"))
