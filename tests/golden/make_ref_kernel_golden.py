"""Run the REFERENCE's real CUDA kernels (oracle/_ref, built by oracle/build_ref.py from the
reference's sources) on a B200 and store their outputs as fixtures in this directory.

    python tests/golden/make_ref_kernel_golden.py [OUT_DIR]

These pin the C restatement (oracle/nr_oracle.c) and this repo's kernels: tests/test_oracle.py checks
the oracle against them without a GPU, tests/test_gpu_reference_kernels.py checks both on the GPU.
Inputs are regenerated from seeds by ``ref_kernel_inputs`` and ``stress_inputs`` (also used by the
tests), so only the outputs are stored.  The maps of ``stress_inputs`` are too large to store whole:
their files hold the maps at a seeded sample of foreground pixels plus a SHA-256 of the whole maps.

``--oracle`` computes the maps of ``stress_inputs`` with the C oracle instead, for a machine without the
reference's kernels (the files of ``ref_kernel_inputs`` are left alone); each file records in ``source``
which of the two wrote it.
"""
import importlib.util
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def load_reference_extension():
    import torch  # noqa: F401  (the extension links against libtorch)
    so = os.path.join(ROOT, "oracle", "_ref", "nr_ref_rasterize_cuda.so")
    if not os.path.exists(so):
        return None
    spec = importlib.util.spec_from_file_location("nr_ref_rasterize_cuda", so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def teapot_faces(B, seed, distance=2.732):
    """Teapot seen from B seeded cameras, as gathered screen-space faces [B,nf,3,3] (numpy, CPU math)."""
    import torch
    import neural_renderer_v2_pytorch_b200 as nr
    d = np.load(os.path.join(HERE, "teapot.npz"))
    g = torch.Generator().manual_seed(seed)
    vw = torch.from_numpy(d["vertices"])[None].repeat(B, 1, 1)
    eye = nr.get_points_from_angles(torch.full((B,), distance), torch.rand(B, generator=g) * 80 - 20,
                                    torch.rand(B, generator=g) * 360)
    vs = nr.perspective(nr.look_at(vw, eye))
    return vs[:, torch.from_numpy(d["faces"]).long()].numpy().astype(np.float32)


def random_faces(B, nf, seed, size=0.05):
    rng = np.random.RandomState(seed)
    c = rng.uniform(-1.1, 1.1, size=(B, nf, 1, 2))
    xy = c + rng.normal(0, size, size=(B, nf, 3, 2))
    z = rng.uniform(1.0, 3.0, size=(B, nf, 1, 1)) + rng.normal(0, 0.02, size=(B, nf, 3, 1))
    return np.concatenate([xy, z], -1).astype(np.float32)


def ref_kernel_inputs():
    """name -> (faces [B,nf,3,3], image_size, near, far, draw_backside)"""
    return {
        "teapot_128": (teapot_faces(4, 31), 128, 0.1, 100.0, 1),
        "teapot_cull_96": (teapot_faces(2, 32), 96, 0.1, 100.0, 0),
        "teapot_clip_100": (teapot_faces(2, 33), 100, 2.2, 2.9, 1),
        "random_128": (random_faces(2, 4000, 34), 128, 0.1, 100.0, 1),
        "random_big_64": (random_faces(1, 300, 35, size=0.8), 64, 0.1, 100.0, 0),
    }


def stacked_faces(n, seed, jitter, box=0.08, views=1):
    """n triangles that all cover the same few dozen pixels at depths within `jitter` of each other: every pixel
    under them is a near-tie, i.e. the order-dependent z-test (rasterize_cuda_kernel.cu:145-148) decides."""
    rng = np.random.RandomState(seed)
    c = rng.uniform(-0.5, 0.5, size=(views, 1, 1, 2)).astype(np.float32)
    xy = (c + rng.uniform(-box, box, size=(views, n, 3, 2))).astype(np.float32)
    z = (1.5 + rng.uniform(-jitter, jitter, size=(views, n, 3, 1))).astype(np.float32)
    return np.ascontiguousarray(np.concatenate([xy, z], -1))


def stress_inputs():
    """name -> (faces, image_size, near, far, draw_backside): config-2 geometry at full size, config-4 style
    density, and piles of faces within (and around) the 1e-4 depth hysteresis of each other."""
    out = {
        "teapot_512": (teapot_faces(8, 77), 512, 0.1, 100.0, 1),
        "random_1024": (random_faces(1, 200000, 78, size=0.005), 1024, 0.1, 100.0, 1),
    }
    for n, jitter in ((300, 2e-4), (5000, 3e-4), (5000, 5e-2)):
        out["ties_%d_%g" % (n, jitter)] = (stacked_faces(n, 1234 + n, jitter), 128, 0.1, 100.0, 1)
    return out


WHOLE = 1 << 18     # maps of up to this many pixels are stored whole
SAMPLE = 4096       # foreground pixels stored per map when the whole map is too large to store


def digest(a, dtype):
    """SHA-256 of a map's values (-0.0 counted as 0.0, as np.array_equal does)."""
    import hashlib
    return hashlib.sha256((np.ascontiguousarray(a, dtype=dtype) + dtype(0)).tobytes()).hexdigest()


def outputs_to_store(faces, fim, wm, source):
    """The arrays of one fixture: the whole maps when they are small, else the maps at a seeded sample of
    foreground pixels (``pixels``: flat indices into [B, S, S]) and the SHA-256 of the whole maps."""
    out = dict(faces_checksum=np.float64(faces.astype(np.float64).sum()), source=source)
    if fim.size <= WHOLE:
        return dict(out, face_index_map=fim, weight_map=wm)
    fg = np.flatnonzero(fim.reshape(-1) >= 0)
    px = np.sort(np.random.default_rng(0).choice(fg, min(SAMPLE, fg.size), replace=False)).astype(np.int32)
    return dict(out, shape=np.array(fim.shape, np.int32), pixels=px, face_index_map=fim.reshape(-1)[px],
                weight_map=wm.reshape(-1, 3)[px], face_index_map_sha256=digest(fim, np.int32),
                weight_map_sha256=digest(wm, np.float32))


def run_reference(mod, faces, S, near, far, backside):
    import torch
    f = torch.from_numpy(faces).cuda().contiguous()
    B, nf = f.shape[:2]
    fim = torch.zeros(B * S * S, dtype=torch.int32, device="cuda") - 1
    mod.face_index_map_forward_safe(f, fim, nf, S, near, far, backside, 1e-8, 1e-4)
    wm = torch.zeros((B * S * S, 3), dtype=torch.float32, device="cuda")
    mod.compute_weight_map_c(f, fim, wm, nf, S)
    torch.cuda.synchronize()
    return fim.reshape(B, S, S).cpu().numpy(), wm.reshape(B, S, S, 3).cpu().numpy()


def main():
    args = sys.argv[1:]
    use_oracle = "--oracle" in args
    args = [a for a in args if a != "--oracle"]
    out_dir = args[0] if args else HERE
    if use_oracle:
        import oracle
        source = "C oracle (oracle/nr_oracle.c)"

        def maps(faces, S, near, far, bs):
            fim = oracle.face_index_map(faces, S, near, far, bool(bs))
            return fim, oracle.weight_map(faces, fim)
    else:
        mod = load_reference_extension()
        assert mod is not None, "oracle/_ref/nr_ref_rasterize_cuda.so missing: run oracle/build_ref.py first"
        source = "reference CUDA kernels"

        def maps(faces, S, near, far, bs):
            return run_reference(mod, faces, S, near, far, bs)
    os.makedirs(out_dir, exist_ok=True)
    cases = stress_inputs() if use_oracle else dict(ref_kernel_inputs(), **stress_inputs())
    for name, (faces, S, near, far, bs) in cases.items():
        fim, wm = maps(faces, S, near, far, bs)
        path = os.path.join(out_dir, "ref_kernel_%s.npz" % name)
        np.savez_compressed(path, **outputs_to_store(faces, fim, wm, source))
        print("wrote", path, os.path.getsize(path), "bytes; foreground", int((fim >= 0).sum()))


if __name__ == "__main__":
    main()
