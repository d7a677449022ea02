"""Dynamic-patch tiling of still images (SURVEY.md 8f-4, image_processor.py:263-285, 404-448) - CPU side.

* the product's grid chooser (`long_vita_b200.preprocess.dynamic_tile_grid`, host arithmetic) against the reference's own
  `dynamic_preprocess` (a recorded run, tests/golden/ref_recorded.pt), the oracle and the committed fixture;
* the per-element bodies of the CUDA kernels (`csrc/preprocess_core.h`, the text the kernels compile) built with gcc
  and driven with the product's own tables and grid: bit-identical bf16 tiles to the reference fixture.
The kernels themselves (launch geometry, device pointers) are the business of tests/test_gpu_preprocess.py.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD = os.path.join(HERE, "golden")
sys.path.insert(0, ROOT)

from long_vita_b200 import preprocess as PP          # noqa: E402
from oracle import preprocess as OP                  # noqa: E402
from tests.util import recorded                      # noqa: E402


def _sizes():
    rng = np.random.default_rng(7)
    s = [(448, 448), (896, 448), (448, 896), (1000, 1000), (1344, 448), (640, 480), (1920, 1080), (1080, 1920), (4000, 300),
         (300, 4000), (449, 448), (448 * 3, 448 * 2), (672, 448), (448, 672), (1, 1), (5000, 5000), (200, 100)]
    s += [(int(a), int(b)) for a, b in rng.integers(1, 3000, (300, 2))]
    return s


def test_tile_grid_equals_the_oracle_and_the_fixture():
    for w, h in _sizes():
        for lo, hi in ((1, 12), (1, 6), (2, 9)):
            assert PP.dynamic_tile_grid(w, h, lo, hi, 448) == OP.dynamic_grid(w, h, lo, hi, 448), (w, h, lo, hi)
    g = torch.load(os.path.join(GOLD, "ref_preprocess_dynamic.pt"))
    S = g["image_size"]
    for im, gp in zip(g["images"], g["grid_pixels"]):
        gx, gy = PP.dynamic_tile_grid(im.shape[1], im.shape[0], g["min_patch_grid"], g["max_patch_grid"], S)
        assert (gx * S, gy * S) == tuple(gp)


def test_tile_grid_equals_the_references_own_dynamic_preprocess():
    sys.path.insert(0, GOLD)
    from make_golden import reference_dynamic_grid

    cases = [(w, h, 448, 1, 12) for w, h in _sizes()] + [(w, h, 336, 1, 6) for w, h in _sizes()[:40]]
    want = recorded("dynamic_grid", lambda: [tuple(reference_dynamic_grid(w, h, S, lo, hi)) for w, h, S, lo, hi in cases])
    assert len(want) == len(cases)
    for (w, h, S, lo, hi), grid in zip(cases, want):
        assert PP.dynamic_tile_grid(w, h, lo, hi, S) == grid, (w, h, S)


def test_vectorised_resampling_tables_equal_the_oracle_loop():
    """long_vita_b200.preprocess.resample_table (numpy, one column of the window at a time) against the oracle's
    per-pixel restatement of Pillow's precompute_coeffs / normalize_coeffs_8bpc: windows and 22-bit weights identical."""
    rng = np.random.default_rng(0)
    pairs = [(1920, 448), (448, 448), (448, 1792), (3840, 1792), (2160, 896), (1, 28), (5, 3), (3, 5), (5376, 448), (448, 5376),
             (1000, 999), (999, 1000)] + [(int(a), int(b)) for a, b in rng.integers(1, 2500, (60, 2))]
    for a, b in pairs:
        xm, cn, kk = OP.resample_coeffs(a, b)
        x2, c2, r2, k2 = PP.resample_table(a, b)
        assert kk.shape[1] == k2 and x2.dtype == c2.dtype == r2.dtype == np.int32, (a, b)
        assert np.array_equal(xm, x2) and np.array_equal(cn, c2) and np.array_equal(kk, r2), (a, b)


@pytest.fixture(scope="module")
def host_kernels(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("pre_host") / "libpre_tiles_host.so")
    cmd = ["gcc", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-I", os.path.join(ROOT, "long-vita_b200", "csrc"),
           os.path.join(HERE, "native", "pre_tiles_host.c"), "-o", so]
    subprocess.run(cmd, check=True)
    lib = C.CDLL(so)
    p = C.c_void_p
    lib.lv_host_resize_h.argtypes = [p, p, p, p, p, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.lv_host_resize_v_tiles.argtypes = [p, p, p, p, p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, p, p]
    lib.lv_host_resize_h.restype = lib.lv_host_resize_v_tiles.restype = None
    return lib


def _table(n_in, n_out):
    xmin, cnt, rows, ksize = PP.resample_table(n_in, n_out)
    return (np.asarray(xmin, np.int32), np.asarray(cnt, np.int32), np.ascontiguousarray(np.asarray(rows, np.int32)), ksize)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _host_tiles(lib, img, out, out_h, out_w, S, tile_base, mean, std):
    """What long_vita_b200.preprocess._tiles_call asks lv_image_tiles_preprocess to do, on the host build."""
    H, W, _ = img.shape
    xt, yt = _table(W, out_w), _table(H, out_h)
    tmp = np.empty((H, out_w, 3), np.uint8)
    lib.lv_host_resize_h(_ptr(img), _ptr(tmp), _ptr(xt[0]), _ptr(xt[1]), _ptr(xt[2]), xt[3], H, W, out_w)
    m, s = np.asarray(mean, np.float32), np.asarray(std, np.float32)
    lib.lv_host_resize_v_tiles(_ptr(tmp), _ptr(out), _ptr(yt[0]), _ptr(yt[1]), _ptr(yt[2]), yt[3], out_h, out_w, S, tile_base,
                               _ptr(m), _ptr(s))


def _host_dynamic(lib, img, lo, hi, S):
    img = np.ascontiguousarray(img)
    gx, gy = PP.dynamic_tile_grid(img.shape[1], img.shape[0], lo, hi, S)
    thumb = 1 if gx * gy > 1 else 0
    out = np.full((gx * gy + thumb, 3, S, S), 0xFFFF, np.uint16)          # a bit pattern no pixel produces (NaN)
    _host_tiles(lib, img, out, gy * S, gx * S, S, thumb, PP.IMAGENET_DEFAULT_MEAN, PP.IMAGENET_DEFAULT_STD)
    if thumb:
        _host_tiles(lib, img, out, S, S, S, 0, PP.IMAGENET_DEFAULT_MEAN, PP.IMAGENET_DEFAULT_STD)
    return torch.from_numpy(out.view(np.int16)).view(torch.bfloat16), (gx * S, gy * S)


def test_kernel_bodies_on_the_host_match_the_references_own_process_dynamic_fixture(host_kernels):
    g = torch.load(os.path.join(GOLD, "ref_preprocess_dynamic.pt"))
    for im, ref, gp in zip(g["images"], g["out"], g["grid_pixels"]):
        got, grid = _host_dynamic(host_kernels, im.numpy(), g["min_patch_grid"], g["max_patch_grid"], g["image_size"])
        assert grid == tuple(gp)
        assert got.shape == ref.shape
        assert torch.equal(got.view(torch.int16), ref.to(torch.bfloat16).view(torch.int16)), tuple(im.shape)


def test_kernel_bodies_on_the_host_match_the_oracle_at_448(host_kernels):
    """Full tile size, a 700 x 1400 image (tie between the 1 x 2 and 2 x 4 grids, decided by the area rule): scaled up
    on both axes, 2 x 4 tiles + thumbnail."""
    rng = np.random.default_rng(11)
    base = rng.integers(0, 256, (90, 50, 3)).repeat(16, axis=0).repeat(16, axis=1)[:1400, :700]
    img = np.clip(base + rng.integers(-30, 31, base.shape), 0, 255).astype(np.uint8)
    ref, grid_ref = OP.process_dynamic(img, 1, 12, 448)
    got, grid = _host_dynamic(host_kernels, img, 1, 12, 448)
    assert grid == grid_ref == (896, 1792) and got.shape[0] == 9
    assert torch.equal(got.view(torch.int16), torch.from_numpy(ref).to(torch.bfloat16).view(torch.int16))
