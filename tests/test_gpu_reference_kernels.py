"""This repo's CUDA path and the C oracle against what the reference's REAL CUDA kernels computed.
face_index_map and weight_map must be bit-identical.

The reference's kernels are not part of this repository; their outputs are stored as
tests/golden/ref_kernel_*.npz (tests/golden/make_ref_kernel_golden.py) and the inputs are regenerated
from seeds.  The files of ``ref_kernel_inputs`` were written by the reference's kernels on a B200.  Those
of ``stress_inputs`` were written by the C oracle (their ``source``): at commit 8e6a457 this module
compared the reference's kernels on a B200 with the C oracle and this repo's kernels on exactly these
inputs and passed, and neither the kernels nor the oracle nor the inputs have changed since.  Maps too
large to store whole are checked at the stored sample of pixels and, everywhere, through the SHA-256 of
the whole map."""
import os
import sys

import numpy as np
import pytest
import torch

import oracle

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLDEN)
import make_ref_kernel_golden as mk  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def nr():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import neural_renderer_v2_pytorch_b200 as nr_
    return nr_


def stored(name, faces):
    """The stored reference output of case `name`, after checking that `faces` are its inputs."""
    d = np.load(os.path.join(GOLDEN, "ref_kernel_%s.npz" % name))
    assert abs(float(d["faces_checksum"]) - faces.astype(np.float64).sum()) < 1e-9, "inputs not reproduced"
    return d


def assert_maps(d, fim, wm, what):
    """fim [B,S,S] and wm [B,S,S,3] are the stored maps of `d`, bit for bit."""
    if "pixels" not in d:
        assert np.array_equal(fim, d["face_index_map"]), "%s: %d px differ" % (what, (fim != d["face_index_map"]).sum())
        assert np.array_equal(wm, d["weight_map"]), "%s: weight map differs" % what
        return
    assert fim.shape == tuple(d["shape"]), what
    px = d["pixels"]
    f, w = fim.reshape(-1)[px], wm.reshape(-1, 3)[px]
    assert np.array_equal(f, d["face_index_map"]), "%s: %d of %d sampled px differ" % (
        what, (f != d["face_index_map"]).sum(), px.size)
    assert np.array_equal(w, d["weight_map"]), "%s: weight map differs at the sampled px" % what
    assert mk.digest(fim, np.int32) == str(d["face_index_map_sha256"]), "%s: face_index_map differs" % what
    assert mk.digest(wm, np.float32) == str(d["weight_map_sha256"]), "%s: weight map differs" % what


def c_oracle(faces, S, near, far, bs):
    fim = oracle.face_index_map(faces, S, near, far, bool(bs))
    return fim, oracle.weight_map(faces, fim)


def ours(nr, faces, S, near, far, bs):
    f = torch.from_numpy(faces).cuda().contiguous()
    B, nf = f.shape[:2]
    fim = torch.empty(B * S * S, dtype=torch.int32, device="cuda")
    nr.face_index_map_forward_safe(f, fim, nf, S, near, far, bs, 1e-8, 1e-4)
    wm = torch.zeros((B * S * S, 3), dtype=torch.float32, device="cuda")
    nr.compute_weight_map_c(f, fim, wm, nf, S)
    return fim.reshape(B, S, S).cpu().numpy(), wm.reshape(B, S, S, 3).cpu().numpy()


def ours_dense(nr, faces, S, near, far, bs):
    """The same maps from the fused forward with the face-parallel raster kernel (nr_raster_dense.cu)."""
    from neural_renderer_v2_pytorch_b200 import rasterize as rz
    B, nf = faces.shape[:2]
    v = torch.from_numpy(np.ascontiguousarray(faces, dtype=np.float32)).reshape(B, nf * 3, 3).cuda()
    idx = torch.arange(nf * 3, dtype=torch.int32).reshape(nf, 3).cuda()
    rz.FORCE_DENSE_RASTER = True
    try:
        hp = nr.RasterizeHyperparam(image_size=S, near=near, far=far, anti_aliasing=False, draw_backside=bool(bs),
                                    draw_rgb=False, draw_depth=False)
        maps = nr.rasterize_maps(v, idx, nr.RasterizeParam(), hp)
    finally:
        rz.FORCE_DENSE_RASTER = None
    return maps["face_index_map"].cpu().numpy(), maps["weight_map"].cpu().numpy()


@pytest.mark.parametrize("name", sorted(mk.ref_kernel_inputs().keys()))
def test_three_way(nr, name):
    faces, S, near, far, bs = mk.ref_kernel_inputs()[name]
    d = stored(name, faces)
    assert_maps(d, *c_oracle(faces, S, near, far, bs), "C oracle")
    assert_maps(d, *ours(nr, faces, S, near, far, bs), "CUDA path")
    assert_maps(d, *ours_dense(nr, faces, S, near, far, bs), "dense raster kernel")


def test_full_size_teapot_512(nr):
    """BASELINE config 2 geometry (teapot, 512^2), 8 views: 2.1 M pixels, bit-exact vs the reference kernel."""
    faces, S, near, far, bs = mk.stress_inputs()["teapot_512"]
    d = stored("teapot_512", faces)
    fim_c, wm_c = c_oracle(faces, S, near, far, bs)
    assert (fim_c >= 0).mean() > 0.05
    assert_maps(d, fim_c, wm_c, "C oracle")
    assert_maps(d, *ours(nr, faces, S, near, far, bs), "CUDA path")
    assert_maps(d, *ours_dense(nr, faces, S, near, far, bs), "dense raster kernel")


def test_dense_random_1024(nr):
    """Config-4 style stress at reduced face count: 200k random ~5 px triangles at 1024^2."""
    faces, S, near, far, bs = mk.stress_inputs()["random_1024"]
    d = stored("random_1024", faces)
    assert_maps(d, *c_oracle(faces, S, near, far, bs), "C oracle")
    assert_maps(d, *ours(nr, faces, S, near, far, bs), "CUDA path")
    assert_maps(d, *ours_dense(nr, faces, S, near, far, bs), "dense raster kernel")


@pytest.mark.parametrize("n,jitter", [(300, 2e-4), (5000, 3e-4), (5000, 5e-2)])
def test_dense_path_with_piles_of_near_ties(nr, n, jitter):
    """The z-buffer rasterizer on its worst case: thousands of faces over the same pixels with depths inside
    (and around) the 1e-4 hysteresis.  Every covered pixel is contested, a CTA's (face, contested pixel) pairs
    outgrow their shared-memory queue, pixels hold more candidates than the resolve pass sorts (it then replays
    the reference's loop over all faces), and with the default pool the candidate nodes overflow on the first
    call.  The map must still be the reference kernel's, bit for bit."""
    name = "ties_%d_%g" % (n, jitter)
    faces, S, near, far, bs = mk.stress_inputs()[name]
    d = stored(name, faces)
    assert (d["face_index_map"] >= 0).sum() > 50
    fim_c = oracle.face_index_map(faces, S)
    assert np.array_equal(fim_c, d["face_index_map"]), "C oracle != reference kernel"
    fim_o, wm_o = ours(nr, faces, S, near, far, bs)
    assert np.array_equal(fim_o, d["face_index_map"]), "tile pipeline: %d px differ" % (fim_o != d["face_index_map"]).sum()
    for attempt in range(3):        # the host grows the candidate pool from the statistics of earlier calls
        fim_d, wm_d = ours_dense(nr, faces, S, near, far, bs)
        assert_maps(d, fim_d, wm_d, "z-buffer path, call %d" % attempt)
        torch.cuda.synchronize()
