#!/usr/bin/env python
"""Cost of light gradients at config 2 lit: teapot, 64 views at 512^2, RGB, directional + ambient + specular light,
forward + backward replayed from a CUDA graph.  Three arms, alternated round by round in one call (boxes differ by
~2 %, see tools/exp_step.py):

    parent  constant lights, the package and library of another tree (--parent-root, e.g. a checkout of the
            commit before light gradients, built)
    const   constant lights, this tree
    grad    every light tensor requires grad, this tree (the backward also sums d loss / d light data)

    python tools/time_light_gradients.py --parent-root /path/to/parent/tree [--rounds 3]

Prints the device name and power limit, then one line per (round, arm) and a JSON summary (best ms per arm)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def child(root, arm):
    sys.path.insert(0, root)
    import torch
    import bench
    import neural_renderer_v2_pytorch_b200 as nr
    if arm == "parent":
        # Before light gradients, pack_lights copied the light types from the host on every call, which a graph
        # capture refuses.  Give that module a torch whose tensor() hands back the tensor it made the first time.
        import types as _types
        from neural_renderer_v2_pytorch_b200 import lights as lm
        made = {}

        def tensor(data, *a, **k):
            key = repr((data, a, sorted(k.items())))
            if key not in made:
                made[key] = torch.tensor(data, *a, **k)
            return made[key]
        lm.torch = _types.SimpleNamespace(**{n: getattr(torch, n) for n in dir(torch) if not n.startswith("__")})
        lm.torch.tensor = tensor
    dev = torch.device("cuda:0")
    w = dict(bench.WORKLOADS["cfg2"], mode="rgb")
    inp = bench.make_inputs(w, 1000, dev, nr)
    B, S = w["views"], w["S"]
    faces, G = inp["faces"].to(dev), inp["G"].to(dev)
    vt, ft = inp["vt"].to(dev), inp["ft"].to(dev)
    v = inp["vertices"].to(dev).requires_grad_(True)
    tex = inp["textures"].to(dev).requires_grad_(True)
    g = torch.Generator().manual_seed(7)
    grad = arm == "grad"
    mk = lambda *s: (torch.rand(*s, generator=g)).to(dev).requires_grad_(grad)
    L = dict(dc=mk(B, 3), dd=(torch.tensor([0., 0., -1.]) + 0.3 * torch.randn(B, 3, generator=g)).to(dev).requires_grad_(grad),
             ac=mk(B, 3), sc=mk(B, 3), sa=(1. + 4. * torch.rand(B, generator=g)).to(dev).requires_grad_(grad))
    lights = [nr.DirectionalLight(L["dc"], L["dd"]), nr.AmbientLight(L["ac"]), nr.SpecularLight(L["sc"], L["sa"])]

    def step():
        hp = nr.RasterizeHyperparam(image_size=S, anti_aliasing=False)
        p = nr.RasterizeParam(vertices_textures=vt, faces_textures=ft, textures=tex, lights=lights)
        img = nr.rasterize_rgb(v, faces, p, hp)
        img.backward(G)
        return img

    params = [v, tex] + (list(L.values()) if grad else [])
    run = nr.capture_step(step, params=params, warmup=3)
    for _ in range(20):
        run()
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(200):
            run()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / 200)
    extra = (" |d light| %.6g" % sum(float(t.grad.double().abs().sum()) for t in L.values())) if grad else ""
    # where the time goes: the library's kernels bracketed by CUDA events (nr_profile_enable), over eager steps
    import ctypes
    from neural_renderer_v2_pytorch_b200 import _lib
    lib = _lib.lib()
    ms, launches = (ctypes.c_float * _lib.NR_PROF_SLOTS)(), (ctypes.c_int32 * _lib.NR_PROF_SLOTS)()
    lib.nr_profile_collect(ms, launches)
    lib.nr_profile_enable(1)
    for _ in range(20):
        step()
    torch.cuda.synchronize()
    lib.nr_profile_collect(ms, launches)
    lib.nr_profile_enable(0)
    split = "  kernels ms/step: " + ", ".join("%s %.4f" % (n, ms[i] / 20) for i, n in enumerate(_lib.PROF_SLOT_NAMES)
                                              if launches[i])
    print("ARM %s %.4f ms/step  |d v| %.6g%s  (%s)%s" % (arm, best, float(v.grad.double().abs().sum()), extra,
                                                         os.path.relpath(nr.__file__, root), split), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-root", default=None, help="tree of the build to compare with (constant lights only)")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import torch
    print("device: %s" % torch.cuda.get_device_name(0))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,power.max_limit", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    print("nvidia-smi name, power.limit, power.max_limit: %s" % q.stdout.strip(), flush=True)
    arms = ([("parent", os.path.abspath(args.parent_root))] if args.parent_root else []) + [("const", ROOT), ("grad", ROOT)]
    res = {a: [] for a, _ in arms}
    for r in range(args.rounds):
        for arm, root in arms:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", root, arm],
                                 stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout
            line = [ln for ln in out.splitlines() if ln.startswith("ARM ")]
            if not line:
                print(out)
                raise SystemExit("arm %s failed" % arm)
            print("round %d %s" % (r, line[0]), flush=True)
            res[arm].append(float(line[0].split()[2]))
    summary = {a: dict(best_ms=min(v), all_ms=v) for a, v in res.items()}
    print(json.dumps(dict(workload="cfg2 lit (rgb, directional + ambient + specular, 64 x 512^2, graph replay)",
                          device=torch.cuda.get_device_name(0), power=q.stdout.strip(), arms=summary)))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--child":
        child(sys.argv[2], sys.argv[3])
    else:
        main()
