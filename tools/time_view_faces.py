#!/usr/bin/env python
"""Cost of per-view faces ([B, nf, 3], NR_VIEW_FACES), in one call:

  bench     bench.py --workload cfg1 .. cfg5 (and cfg2s, cfg2r) of this tree and of --parent-root (a built checkout of
            the commit before per-view faces), alternated round by round, one process per run;
  expanded  config 2 (teapot, 64 views, 512^2, RGBA, forward + backward replayed from a CUDA graph) with its faces
            passed as [64, nf, 3] against [nf, 3];
  distinct  64 different meshes (teapot / UV sphere / textured model cycled, each with its own camera, padded to
            common nv and nf), 512^2, RGBA, forward + backward replayed from a CUDA graph: the batched call, 64
            single-view calls, and the gather workaround (vertices gathered to [64, 3 nf, 3], faces = arange; unlit).

    python tools/time_view_faces.py --parent-root /path/to/parent/tree [--rounds 3]

Prints the card's name, power limit and maximum SM clock, then one line per measurement."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKLOADS = ["cfg1", "cfg2", "cfg2s", "cfg2r", "cfg3", "cfg4", "cfg5"]


def timed(run, reps=200):
    """Best of three windows of `reps` replays, ms per replay (CUDA events)."""
    import torch
    for _ in range(20):
        run()
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            run()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / reps)
    return best


def child_expanded():
    sys.path.insert(0, ROOT)
    import torch
    import bench
    import neural_renderer_v2_pytorch_b200 as nr
    dev = torch.device("cuda:0")
    w = dict(bench.WORKLOADS["cfg2"])
    inp = bench.make_inputs(w, 1000, dev, nr)
    B, S = w["views"], w["S"]
    faces, G = inp["faces"].to(dev), inp["G"].to(dev)
    vt, ft = inp["vt"].to(dev), inp["ft"].to(dev)
    v = inp["vertices"].to(dev).requires_grad_(True)
    tex = inp["textures"].to(dev).requires_grad_(True)
    res = {}
    for arm in ("shared", "expanded", "shared", "expanded"):
        f = faces if arm == "shared" else faces[None].expand(B, *faces.shape).contiguous()
        t = ft if arm == "shared" else ft[None].expand(B, *ft.shape).contiguous()

        def step():
            hp = nr.RasterizeHyperparam(image_size=S, anti_aliasing=False)
            img = nr.rasterize_rgba(v, f, nr.RasterizeParam(vertices_textures=vt, faces_textures=t, textures=tex), hp)
            img.backward(G)
            return img
        run = nr.capture_step(step, params=[v, tex], warmup=3)
        res[arm] = min(res.get(arm, 1e9), timed(run))
    print("RESULT " + json.dumps({"expanded": res}), flush=True)


def child_distinct():
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    import bench
    import neural_renderer_v2_pytorch_b200 as nr
    dev = torch.device("cuda:0")
    B, S, H, W = 64, 512, 12, 8
    g = torch.Generator().manual_seed(0)
    d = np.load(os.path.join(ROOT, "tests", "golden", "teapot.npz"))
    sv, sf = bench.sphere_mesh(40)
    mv, mf, mvt, mft, mtex = nr.load_obj(os.path.join(ROOT, "tests", "golden", "textured", "m.obj"), load_textures=True)
    rnd_vt = lambda n: torch.rand((n, 2), generator=g) * torch.tensor([W - 1., H - 1.])
    base = [(torch.from_numpy(d["vertices"]), torch.from_numpy(d["faces"]).int(), None, None),
            (sv, sf, None, None),
            (torch.from_numpy(mv), torch.from_numpy(mf).int(), torch.from_numpy(mvt), torch.from_numpy(mft).int())]
    meshes = []
    for b in range(B):
        v, f, vt, ft = base[b % 3]
        if vt is None:
            vt, ft = rnd_vt(v.shape[0]), f
        meshes.append((v, f, vt, ft))
    nv = max(m[0].shape[0] for m in meshes)
    nf = max(m[1].shape[0] for m in meshes)
    nvt = max(m[2].shape[0] for m in meshes)
    eye = nr.get_points_from_angles(torch.full((B,), 2.732), torch.rand(B, generator=g) * 60 - 20, torch.rand(B, generator=g) * 360)
    V = torch.zeros((B, nv, 3))
    F = torch.zeros((B, nf, 3), dtype=torch.int32)
    VT = torch.zeros((B, nvt, 2))
    FT = torch.zeros((B, nf, 3), dtype=torch.int32)
    for b, (v, f, vt, ft) in enumerate(meshes):
        V[b, :v.shape[0]] = nr.perspective(nr.look_at(v[None].float(), eye[b:b + 1]))[0]
        F[b, :f.shape[0]] = f
        VT[b, :vt.shape[0]] = vt
        FT[b, :ft.shape[0]] = ft
    T = torch.rand((B, 3, H, W), generator=g)
    Gr = torch.randn((B, 4, S, S), generator=g)
    V, F, VT, FT, T, Gr = (t.to(dev) for t in (V, F, VT, FT, T, Gr))
    v = V.clone().requires_grad_(True)
    tex = T.clone().requires_grad_(True)
    hp = lambda: nr.RasterizeHyperparam(image_size=S, anti_aliasing=False)
    singles = [(m[0].shape[0], F[b, :m[1].shape[0]].contiguous(), VT[b:b + 1, :m[2].shape[0]].contiguous(),
                FT[b, :m[1].shape[0]].contiguous()) for b, m in enumerate(meshes)]
    idx = torch.arange(3 * nf, dtype=torch.int32, device=dev).reshape(nf, 3)
    bidx = torch.arange(B, device=dev)[:, None, None]

    def batched():
        img = nr.rasterize_rgba(v, F, nr.RasterizeParam(vertices_textures=VT, faces_textures=FT, textures=tex), hp())
        img.backward(Gr)
        return img

    def single():
        for b, (n, f, vt, ft) in enumerate(singles):
            img = nr.rasterize_rgba(v[b:b + 1, :n], f, nr.RasterizeParam(vertices_textures=vt, faces_textures=ft,
                                                                         textures=tex[b:b + 1]), hp())
            img.backward(Gr[b:b + 1])

    def gather():
        vg = v[bidx, F.long()].reshape(B, 3 * nf, 3)
        vtg = VT[bidx, FT.long()].reshape(B, 3 * nf, 2)
        img = nr.rasterize_rgba(vg, idx, nr.RasterizeParam(vertices_textures=vtg, faces_textures=idx, textures=tex), hp())
        img.backward(Gr)
        return img

    res = {"views": B, "nv": nv, "nf": nf}
    for arm, fn in (("batched", batched), ("single_view_calls", single), ("gather", gather)) * 2:
        run = nr.capture_step(fn, params=[v, tex], warmup=3)
        res[arm] = min(res.get(arm, 1e9), timed(run, 50 if arm == "single_view_calls" else 200))
    print("RESULT " + json.dumps({"distinct": res}), flush=True)


def bench_line(root, workload, steps):
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--workload", workload,
                          "--steps", str(steps), "--warmup", "20", "--no-cpu-baseline"], cwd=root,
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout
    for ln in out.splitlines():
        if ln.startswith("{"):
            j = json.loads(ln)
            return j.get("ms_per_step"), j.get("kernels_ms")
    print(out[-3000:])
    return None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-root", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--child", choices=["expanded", "distinct"])
    args = ap.parse_args()
    if args.child:
        {"expanded": child_expanded, "distinct": child_distinct}[args.child]()
        return
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    print("card (name, power.limit, clocks.max.sm): %s" % q.stdout.strip(), flush=True)
    parent = os.path.abspath(args.parent_root)
    for r in range(1, args.rounds + 1):
        for w in WORKLOADS:
            # the order alternates from round to round, so that a drift of the card's clocks favours neither build
            for arm, root in (("parent", parent), ("new", ROOT))[::1 if r % 2 else -1]:
                ms, kern = bench_line(root, w, args.steps)
                print("%-6s %-5s r%d step %s ms  kernels %s" % (arm, w, r, ms, json.dumps(kern)), flush=True)
    for child in ("expanded", "distinct"):
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--parent-root", parent, "--child", child],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout
        lines = [ln[7:] for ln in out.splitlines() if ln.startswith("RESULT ")]
        print(lines[0] if lines else out[-3000:], flush=True)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    print("card (after): %s" % q.stdout.strip(), flush=True)


if __name__ == "__main__":
    main()
