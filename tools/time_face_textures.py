#!/usr/bin/env python
"""Cost of per-face texture cubes ([B, nf, ts, ts, ts, 3], NR_FACE_TEXTURES), in one call:

  cubes  config 2's geometry (teapot, 64 views, 512^2, RGBA, forward + backward replayed from a CUDA graph) with a
         Mesh-style cube set [64, 2464, 4, 4, 4, 3], and config 2's own uv-textured step in the same process for context;
  bench  bench.py --workload cfg1 .. cfg5 (and cfg2s, cfg2r) of this tree and of --parent-root (a built checkout of
         the commit before per-face texture cubes), alternated round by round, one process per run.

    python tools/time_face_textures.py --parent-root /path/to/parent/tree [--rounds 2]

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


def child_cubes():
    sys.path.insert(0, ROOT)
    import torch
    import bench
    import neural_renderer_v2_pytorch_b200 as nr
    dev = torch.device("cuda:0")
    w = dict(bench.WORKLOADS["cfg2"])
    inp = bench.make_inputs(w, 1000, dev, nr)
    B, S, ts = w["views"], w["S"], 4
    faces, G = inp["faces"].to(dev), inp["G"].to(dev)
    vt, ft = inp["vt"].to(dev), inp["ft"].to(dev)
    v = inp["vertices"].to(dev).requires_grad_(True)
    tex = inp["textures"].to(dev).requires_grad_(True)
    nf = faces.shape[0]
    g = torch.Generator().manual_seed(0)
    cubes = torch.sigmoid(torch.randn((B, nf, ts, ts, ts, 3), generator=g)).to(dev).requires_grad_(True)
    hp = lambda: nr.RasterizeHyperparam(image_size=S, anti_aliasing=False)

    def uv():
        img = nr.rasterize_rgba(v, faces, nr.RasterizeParam(vertices_textures=vt, faces_textures=ft, textures=tex), hp())
        img.backward(G)
        return img

    def cube():
        img = nr.rasterize_rgba(v, faces, nr.RasterizeParam(textures=cubes), hp())
        img.backward(G)
        return img

    res = {"views": B, "S": S, "nf": nf, "ts": ts}
    for arm, fn, params in (("uv_cfg2", uv, [v, tex]), ("cubes_ts4", cube, [v, cubes])) * 2:
        run = nr.capture_step(fn, params=params, warmup=3)
        res[arm] = min(res.get(arm, 1e9), timed(run))
    # kernel split of the cube step (bench.py's per-launch CUDA events, outside the timed windows)
    L = nr._lib.lib()
    import ctypes
    for arm, fn in (("uv_cfg2", uv), ("cubes_ts4", cube)):
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        L.nr_profile_enable(1)
        for _ in range(50):
            fn()
        torch.cuda.synchronize()
        ms = (ctypes.c_float * nr._lib.NR_PROF_SLOTS)()
        cnt = (ctypes.c_int32 * nr._lib.NR_PROF_SLOTS)()
        L.nr_profile_collect(ms, cnt)
        L.nr_profile_enable(0)
        res[arm + "_kernels_ms"] = {nr._lib.PROF_SLOT_NAMES[i]: round(ms[i] / 50, 4) for i in range(nr._lib.NR_PROF_SLOTS)
                                    if cnt[i]}
    print("RESULT " + json.dumps({"cubes": res}), flush=True)


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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-root", required=True)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--child", choices=["cubes"])
    args = ap.parse_args()
    if args.child:
        child_cubes()
        return
    print("card (name, power.limit, clocks.max.sm): %s" % card(), flush=True)
    parent = os.path.abspath(args.parent_root)
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "--parent-root", parent, "--child", "cubes"],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout
    lines = [ln[7:] for ln in out.splitlines() if ln.startswith("RESULT ")]
    print(lines[0] if lines else out[-3000:], flush=True)
    for r in range(1, args.rounds + 1):
        for w in WORKLOADS:
            # the order alternates from round to round, so that a drift of the card's clocks favours neither build
            for arm, root in (("parent", parent), ("new", ROOT))[::1 if r % 2 else -1]:
                ms, kern = bench_line(root, w, args.steps)
                print("%-6s %-5s r%d step %s ms  kernels %s" % (arm, w, r, ms, json.dumps(kern)), flush=True)
    print("card (after): %s" % card(), flush=True)


if __name__ == "__main__":
    main()
