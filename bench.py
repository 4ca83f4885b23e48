#!/usr/bin/env python
"""Benchmark of the rasterize -> sample -> approximate-gradient hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2] [--dump-outputs DIR]

One "step" = one forward + backward of ``rasterize_rgba`` over one batch of synthetic views
(BASELINE.json config 2: teapot, a batch of 64 views, 512x512, no anti-aliasing, RGBA with a
texture_size-4 atlas; upstream gradient G ~ N(0,1) fixed, SURVEY.md section 8d).  Metric:
megapixel-views per second = views * S^2 / 1e6 / time.  For N > 1 the driver launches this file under
torchrun and config 2's batch of 64 is SHARDED over the ranks (64 / N views per GPU, "scaling":
"strong", as BASELINE.json configs[1] says; no data-path collective: views are independent); the step
time is the max over ranks, `value` the aggregate.  ``--scaling weak`` keeps 64 views per GPU instead.
Config 3 (one shared mesh, 8 views per GPU, gradient all-reduce) is weak-scaled by definition.

Prints ONE JSON line (rank 0).  Keys beyond the base contract: `roofline`, `cpu_baseline`,
`e2e`, `gpu_launches`, `clocks`, `kernels_ms`.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

if "reference" in sys.argv[1:]:
    # the CPU arm uses every host core; torchrun exports OMP_NUM_THREADS=1, and the OpenMP runtime reads it
    # once, when torch loads it
    try:
        os.environ["OMP_NUM_THREADS"] = str(len(os.sched_getaffinity(0)))
    except AttributeError:
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    # views = the batch BASELINE.json names (global batch when strong-scaled, per GPU when weak-scaled)
    # config 2: the configuration the metric is quoted on; its batch of 64 shards over the GPUs
    "cfg2": dict(views=64, S=512, aa=False, mode="rgba", ts=4, mesh="teapot", scaling="strong"),
    "cfg2s": dict(views=64, S=512, aa=False, mode="silhouettes", ts=0, mesh="teapot", scaling="strong"),
    # config 1: examples_pytorch defaults, one view from (2.732, 30, 40), 256^2 with 2x anti-aliasing, ts 16
    "cfg1": dict(views=1, S=256, aa=True, mode="rgba", ts=16, mesh="teapot", camera=(2.732, 30., 40.)),
    # config 5: texture optimisation as examples_pytorch/example3.py: orthographic camera (:40), elevation 0 and
    # a random azimuth (:53), textures = tanh(parameter) (:54), render_rgb with 2x anti-aliasing
    "cfg5": dict(views=32, S=512, aa=True, mode="rgb", ts=4, mesh="teapot", ortho=True, tanh=True, elevation0=True),
    # config 2 through the Renderer facade: world-space vertices -> camera transform -> rasterize
    "cfg2r": dict(views=64, S=512, aa=False, mode="rgba", ts=4, mesh="teapot", renderer=True, scaling="strong"),
    # config 3: multi-view optimisation of ONE shared 100k-face mesh, 8 views per GPU: gradient all-reduce
    "cfg3": dict(views=8, S=512, aa=False, mode="silhouettes", ts=0, mesh="sphere", shared=True),
    # config 4: 1M independent ~5 px triangles: stresses binning and z-test contention
    "cfg4": dict(views=16, S=1024, aa=False, mode="silhouettes", ts=0, mesh="random1m"),
}
METRIC = "megapixel-views/sec fwd+bwd"
UNIT = "Mpix-views/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def algorithmic_bytes(nv, nf, T, P, C, S, depth=False):
    """SURVEY.md section 8(d): per view, forward and backward shares."""
    fwd = 12 * nv + 12 * nf + 12 * T + 4 * P + 12 * P + (4 * P if depth else 0) + 4 * C * S * S
    bwd = 4 * C * S * S + 16 * P + (4 * P if depth else 0) + 12 * nv + 12 * T + 12 * T
    return fwd, bwd


def sphere_mesh(n=225, perturb=0.0, seed=0):
    """UV sphere, n x n vertices (n=225: 50 625 vertices, 100 352 faces); radius 0.8 times a seeded
    low-frequency perturbation (SURVEY.md section 8d, config 3)."""
    i = torch.arange(n, dtype=torch.float32)
    theta = (i / (n - 1) * 3.14159265)[:, None].expand(n, n)
    phi = (i / (n - 1) * 2 * 3.14159265)[None, :].expand(n, n)
    r = torch.full((n, n), 0.8)
    if perturb:
        g = torch.Generator().manual_seed(seed)
        for _ in range(6):
            a, kt, kp, ph = (torch.rand(1, generator=g).item() for _ in range(4))
            r = r * (1 + perturb * (a - 0.5) * torch.sin((1 + int(kt * 4)) * theta + 6.28 * ph) *
                     torch.cos((1 + int(kp * 4)) * phi))
    v = torch.stack((r * torch.sin(theta) * torch.cos(phi), r * torch.cos(theta), r * torch.sin(theta) * torch.sin(phi)), -1)
    idx = (torch.arange(n - 1)[:, None] * n + torch.arange(n - 1)[None, :]).reshape(-1)
    f = torch.cat((torch.stack((idx, idx + 1, idx + n), 1), torch.stack((idx + 1, idx + n + 1, idx + n), 1)), 0)
    return v.reshape(-1, 3).contiguous(), f.to(torch.int32).contiguous()


def random_triangle_mesh(nf=1000000, seed=0):
    """nf independent triangles: centres U(-1,1)^3, corner offsets N(0, 0.01^2); faces = arange."""
    g = torch.Generator().manual_seed(seed)
    c = torch.rand((nf, 1, 3), generator=g) * 2 - 1
    v = (c + torch.randn((nf, 3, 3), generator=g) * 0.01).reshape(-1, 3)
    v = v - v.min(0).values[None]                       # load_obj-style normalisation (load_obj.py:157-161)
    v = v / v.abs().max() * 2
    v = v - v.max(0).values[None] / 2
    return v.contiguous(), torch.arange(nf * 3, dtype=torch.int32).reshape(nf, 3)


def shard_of(w, rank, world, scaling):
    """(global views, first view, one-past-last view) of `rank`.  Strong scaling: the workload's batch is
    split over the ranks (balanced, contiguous).  Weak: every rank has the workload's batch."""
    V = w["views"]
    if scaling == "strong":
        base, extra = divmod(V, world)
        lo = rank * base + min(rank, extra)
        return V, lo, lo + base + (1 if rank < extra else 0)
    return V * world, rank * V, (rank + 1) * V


def make_inputs(w, seed, device, nr, lo=0, hi=None, total=None):
    """Synthetic inputs of views [lo, hi) out of a batch of `total` views drawn from one seeded stream
    (so a sharded run renders exactly the views of the single-GPU run)."""
    total = w["views"] if total is None else total
    hi = total if hi is None else hi
    B, S = hi - lo, w["S"]
    g = torch.Generator().manual_seed(seed)
    elev = torch.rand(total, generator=g) * 80. - 20.
    azim = torch.rand(total, generator=g) * 360.
    dist_ = torch.full((total,), 2.732)
    if w.get("camera"):
        dist_, elev, azim = (torch.full((total,), float(x)) for x in w["camera"])
    if w.get("elevation0"):
        elev = torch.zeros(total)
    eye = nr.get_points_from_angles(dist_, elev, azim)[lo:hi]
    mesh = w.get("mesh", "teapot")
    if mesh == "teapot":
        d = np.load(os.path.join(ROOT, "tests", "golden", "teapot.npz"))
        v_world, faces = torch.from_numpy(d["vertices"]), torch.from_numpy(d["faces"])
    elif mesh == "sphere":
        v_world, faces = sphere_mesh(225, perturb=0.3, seed=0)
    else:
        v_world, faces = random_triangle_mesh(1000000, seed=0)
    tdev = device if (mesh == "random1m" and str(device) != "cpu") else "cpu"   # 3M vertices x 16 views: transform on the GPU
    vs = nr.look_at(v_world.to(tdev)[None].expand(B, -1, -1), eye.to(tdev))
    if not w.get("ortho"):
        vs = nr.perspective(vs)
    vs = vs.contiguous()
    out = dict(vertices=vs, faces=faces, nv=vs.shape[1], nf=faces.shape[0], T=0, eye=eye, v_world=v_world)
    if w["mode"] in ("rgb", "rgba"):
        vt_np, ft_np, tex_np = nr.create_textures(faces.shape[0], w["ts"])
        gt = torch.Generator().manual_seed(0)
        out["textures"] = torch.rand((total,) + tex_np.shape, generator=gt)[lo:hi].contiguous()
        out["vt"] = torch.from_numpy(vt_np)[None].repeat(B, 1, 1).contiguous()
        out["ft"] = torch.from_numpy(ft_np)
        out["T"] = tex_np.shape[1] * tex_np.shape[2]
    C = {"rgba": 4, "rgb": 3, "silhouettes": 1, "depth": 1}[w["mode"]]
    gg = torch.Generator().manual_seed(1)
    shape = (total, C, S, S) if C > 1 else (total, S, S)
    out["G"] = torch.randn(shape, generator=gg)[lo:hi].contiguous()
    out["C"] = C
    return out


def config_of(name, w, inp, world, scaling, local_views, global_views, step_bytes):
    """The `config` object of the JSON line; both arms build it with this function."""
    rgb = w["mode"] in ("rgb", "rgba")
    extras = "".join((", orthographic camera" if w.get("ortho") else "", ", textures = tanh(parameter)" if w.get("tanh") else "",
                      ", one shared mesh (gradient all-reduced over the ranks)" if w.get("shared") else "",
                      ", through Renderer.render (fused camera transform)" if w.get("renderer") else ""))
    return {"workload": "%s: %s (%d v / %d f), batch of %d views, %dx%d, anti_aliasing=%s, %s%s%s"
                        % (name, w.get("mesh", "teapot"), inp["nv"], inp["nf"], global_views, w["S"], w["S"], w["aa"], w["mode"],
                           (", texture_size %d (T=%d texels/view)" % (w["ts"], inp["T"])) if rgb else "", extras),
            "views_per_gpu": local_views, "global_views": global_views, "image_size": w["S"],
            "parallelism": "dp%d" % world,
            "l2": "per-GPU per-step working set %.3f GB vs 126 MB L2, no explicit flush" % (step_bytes / 1e9)}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.active = False                 # samples count only while the timed region runs
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def sample(self):
        """One NVML query; it is kept only while a timed region runs (the queries before it warm NVML up: the
        first ones take tens of milliseconds)."""
        if not self.ok:
            return
        nv = self.nv
        try:
            mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            if not self.active:
                return
            self.samples.append(mhz)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
                     0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}
            for bit, name in names.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        while not self._stop_evt.is_set():
            self.sample()
            self._stop_evt.wait(0.004)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=1.0)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, arrays):
    """Writes every tensor of `arrays` as out_dir/<name>.npy in float32, DUMP_BYTES in all.  The smallest go
    first, whole; a tensor larger than its share of what is left is written as a sample of its flattened
    elements: ascending indices drawn by a generator seeded with 0, so runs with the same arguments write the
    same elements and two builds can be compared element for element."""
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES
    for i, (name, t) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].numel())):
        a = t.detach().float()
        share = (left // (len(arrays) - i) - 4096) // 4     # elements; 4 KB for the .npy header
        if a.numel() > share:
            idx = np.unique(np.random.default_rng(0).integers(0, a.numel(), size=share))
            a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())
        left -= a.numel() * 4 + 4096


def physical_gpu_index(local):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except (ValueError, IndexError):
            return local
    return local


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs NVML reports as local to the GPU, BEFORE any pinned buffer is
    allocated, so the staging memory of the end-to-end arm lives on the GPU's NUMA node."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return 0


# ------------------------------------------------------------------------------------------ ours
def run_ours(args):
    import torch.distributed as dist
    import neural_renderer_v2_pytorch_b200 as nr
    from neural_renderer_v2_pytorch_b200 import _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback "
                         "(use --impl reference for the CPU baseline)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa_cpus = bind_to_gpu_numa_node(physical_gpu_index(local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its "NCCL version ..." banner (NCCL_DEBUG=VERSION / WARN) on stdout, next to the JSON
        # line; send its log to stderr instead
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    w = dict(WORKLOADS[args.workload])
    if args.views:
        w["views"] = args.views
    scaling = args.scaling or w.get("scaling", "weak")
    S = w["S"]
    R = S * 2 if w["aa"] else S
    V, lo, hi = shard_of(w, rank, world, scaling)
    B = hi - lo
    if B <= 0:
        raise SystemExit("bench.py: %d views cannot be split over %d ranks" % (V, world))
    if scaling == "strong":
        inp = make_inputs(w, seed=1000, device=dev, nr=nr, lo=lo, hi=hi, total=V)
    else:       # every rank draws its own views
        inp = make_inputs(w, seed=1000 + rank, device=dev, nr=nr)
    C = inp["C"]
    L = _lib.lib()

    faces = inp["faces"].to(dev)
    G = inp["G"].to(dev)
    rgb = w["mode"] in ("rgb", "rgba")
    ft = inp["ft"].to(dev) if rgb else None
    vt = inp["vt"].to(dev) if rgb else None
    fn = {"rgba": nr.rasterize_rgba, "rgb": nr.rasterize_rgb, "silhouettes": nr.rasterize_silhouettes,
          "depth": nr.rasterize_depth}[w["mode"]]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- the differentiable inputs of the step live in ONE flat device buffer (views of it are the
    # leaves), so the end-to-end arm uploads them with one copy; same for the gradients it reads back
    shared = bool(w.get("shared"))
    if shared:
        leaves_host = [inp["v_world"][None].contiguous()]
        leaf_names = ["vertices_world"]
    elif w.get("renderer"):
        leaves_host = [inp["v_world"][None].repeat(B, 1, 1).contiguous(), inp["textures"]]
        leaf_names = ["vertices_world", "textures"]
    else:
        leaves_host = [inp["vertices"].cpu()] + ([inp["textures"]] if rgb else [])
        leaf_names = ["vertices"] + (["textures"] if rgb else [])
    sizes = [t.numel() for t in leaves_host]
    offs = [sum(sizes[:i]) for i in range(len(sizes))]
    flat_in = torch.empty(sum(sizes), dtype=torch.float32, device=dev)
    params = []
    for t, o, n in zip(leaves_host, offs, sizes):
        flat_in[o:o + n].copy_(t.reshape(-1))
        params.append(flat_in[o:o + n].view(t.shape).requires_grad_(True))

    if shared:
        # ONE mesh parameter for all views of all ranks: world -> screen transform inside the step,
        # squared-error loss against the unperturbed sphere (examples_pytorch/example2.py:39-41), gradient
        # summed over the local views and over the ranks
        param = params[0]
        eye_d = inp["eye"].to(dev)
        tv, _ = sphere_mesh(225, 0.0)
        with torch.no_grad():
            target = fn(nr.perspective(nr.look_at(tv.to(dev)[None].expand(B, -1, -1), eye_d)), faces,
                        nr.RasterizeParam(), nr.RasterizeHyperparam(image_size=S, anti_aliasing=w["aa"]))
        rend = nr.Renderer()
        rend.image_size, rend.anti_aliasing, rend.viewpoints = S, w["aa"], eye_d

        def step_fn():
            # Renderer.render_silhouettes on the shared [1,nv,3] mesh with [B,3] viewpoints: the fused camera
            # transform projects it into every local view; its backward sums the gradient over the views in
            # registers, and share_across_ranks all-reduces the [1,nv,3] result over the ranks (parallel.py)
            shared_param = param if args.no_collective else nr.parallel.share_across_ranks(param)
            images = rend.render_silhouettes(shared_param, faces)
            ((images - target) ** 2).sum().backward()
            return images
    elif w.get("renderer"):
        # the call a user of the reference makes: Renderer.render(world vertices, ...)
        v_dev, tex_dev = params
        rend = nr.Renderer()
        rend.image_size, rend.anti_aliasing, rend.viewpoints = S, w["aa"], inp["eye"].to(dev)
        rend.fused_camera = not args.unfused_camera

        def step_fn():
            images = rend.render(v_dev, faces, vt, ft, tex_dev)
            images.backward(G)
            return images
    else:
        v_dev = params[0]
        tex_dev = params[1] if rgb else None

        def step_fn():
            hp = nr.RasterizeHyperparam(image_size=S, anti_aliasing=w["aa"])
            tex = torch.tanh(tex_dev) if (rgb and w.get("tanh")) else tex_dev       # example3.py:54
            p = nr.RasterizeParam(vertices_textures=vt, faces_textures=ft, textures=tex) if rgb else nr.RasterizeParam()
            images = fn(v_dev, faces, p, hp)
            images.backward(G)           # == ((images * G).sum()).backward(), SURVEY.md 8(d)
            return images

    def eager_step():
        for p_ in params:
            p_.grad = None
        return step_fn()

    for _ in range(max(args.warmup, 3)):
        eager_step()
    barrier()
    # the whole step (forward + backward, a handful of launches, and for a shared mesh the NCCL
    # all-reduce of its gradient) is captured once in a CUDA graph and replayed: every replay does the
    # full work on the device; --eager launches from Python instead
    use_graph = not args.eager
    run_step = eager_step
    if use_graph:
        try:
            run_step = nr.capture_step(step_fn, params=params, warmup=2)
        except Exception as e:      # e.g. a collective that cannot be captured on this NCCL build
            if not (shared and world > 1):
                raise
            sys.stderr.write("bench.py: graph capture with the all-reduce failed (%s); launching eagerly\n" % e)
            use_graph = False
            torch.cuda.synchronize(dev)
    for _ in range(max(args.warmup, 3)):      # warm replays: clocks ramp up, lazy kernel loading is over
        run_step()
    # ... and a dress rehearsal of the timed loop (untimed): on a fresh box the first few hundred replays can be
    # paced by the host (lazy initialisation in the driver), which is not what the metric is about.  At least
    # twice the timed loop and at least ~0.4 s of replays (short steps need hundreds of them); the count is agreed
    # between the ranks, because with a shared mesh every replay holds a collective.
    # (the NVML sampler thread is set up here, not between the rehearsal and the timed region: its start-up takes
    # milliseconds during which the GPU would idle)
    sampler = ClockSampler(physical_gpu_index(local)) if rank == 0 else None
    if sampler:
        sampler.start()
    t_reh = time.perf_counter()
    for _ in range(args.steps):
        run_step()
    torch.cuda.synchronize(dev)
    t_reh = max(time.perf_counter() - t_reh, 1e-6)
    more = max(args.steps, int(0.4 / t_reh * args.steps))
    if world > 1:
        tm = torch.tensor([more], device=dev, dtype=torch.int64)
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        more = int(tm.item())
    more = min(more, 20000)
    for _ in range(more):
        run_step()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if sampler:
        sampler.active = True
    e0.record()
    t_host0 = time.perf_counter()
    for i in range(args.steps):
        images = run_step()
    host_ms = (time.perf_counter() - t_host0) * 1e3 / args.steps
    e1.record()
    # (no NVML call from this thread while it still has launches to issue: one query can take milliseconds, and a
    # short step would run dry behind it.  Here everything is enqueued and the GPU is still working through it)
    if sampler:
        sampler.sample()
    barrier()
    if sampler:
        sampler.active = False
    ms_total = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps
    total_views = V if scaling == "strong" else B * world
    value = total_views * S * S / 1e6 / (ms_step / 1e3)
    # before anything else runs a step: the captured step's outputs are overwritten by the next one
    if args.dump_outputs and rank == 0:
        outputs = {"images": images}
        outputs.update(("grad_" + n, p_.grad) for n, p_ in zip(leaf_names, params))
        dump_outputs(args.dump_outputs, outputs)

    # ---- per-kernel pass (same inputs, right after the timed region): roofline numbers
    L.nr_profile_enable(1)
    for _ in range(args.steps):
        eager_step()
    torch.cuda.synchronize(dev)
    L.nr_profile_enable(0)
    import ctypes
    ms = (ctypes.c_float * _lib.NR_PROF_SLOTS)()
    cnt = (ctypes.c_int32 * _lib.NR_PROF_SLOTS)()
    L.nr_profile_collect(ms, cnt)
    kern = {n: (ms[i] / cnt[i]) for i, n in enumerate(_lib.PROF_SLOT_NAMES) if cnt[i]}
    if "setup_count" in kern and "scan_tiles" not in kern:
        kern["bin_view"] = kern.pop("setup_count")      # small meshes: the one-kernel cluster binning uses this slot
    # kernels of this library per step (memset nodes not counted)
    launches_per_step = sum(cnt[i] for i, n in enumerate(_lib.PROF_SLOT_NAMES) if n != "memset") / args.steps

    # ---- end-to-end arm: host (pinned) inputs -> H2D -> fwd + bwd -> D2H of every gradient
    # Double-buffered pipeline, as a data loader would drive it: while step i runs on the compute stream,
    # the inputs of step i+1 are uploaded on a copy stream (ONE cudaMemcpyAsync from one pinned buffer into
    # a staging buffer; a device-to-device copy moves them into the static inputs of the captured step)
    # and the gradients of step i-1 go back on a third stream (ONE cudaMemcpyAsync into pinned memory).
    # Every step uploads its own inputs and reads all of its gradients back; all inside the timed region.
    host_in = torch.empty(flat_in.numel(), dtype=torch.float32).pin_memory()
    host_in.copy_(flat_in.cpu())
    n_out = flat_in.numel() + 1                           # every gradient + a checksum of the images
    host_out = [torch.empty(n_out, dtype=torch.float32).pin_memory() for _ in range(2)]
    up_stream, down_stream = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    compute_stream = torch.cuda.current_stream(dev)
    stage_in = [torch.empty_like(flat_in) for _ in range(2)]
    stage_out = [torch.empty(n_out, dtype=torch.float32, device=dev) for _ in range(2)]
    ev_up = [torch.cuda.Event() for _ in range(2)]       # staging set filled
    ev_free = [torch.cuda.Event() for _ in range(2)]     # staging set consumed
    ev_grad = [torch.cuda.Event() for _ in range(2)]     # gradients of the slot gathered
    ev_down = [torch.cuda.Event() for _ in range(2)]     # ... and copied to the host

    # The whole pipelined iteration is itself TWO captured CUDA graphs (one per staging slot), replayed in turn,
    # so that the host issues one launch per step (at 8 views per GPU the ~25 Python calls of an eager pipeline
    # cost more than the step).  Graph `slot`:   [copy stream]  stage_in[slot ^ 1] <- pinned inputs (H2D, the NEXT step's)
    #                                             [copy stream]  pinned gradients <- stage_out[slot ^ 1] (D2H, the PREVIOUS step's)
    #                                             [main]         inputs <- stage_in[slot]; forward + backward; gradients -> stage_out[slot]
    def build_e2e_graphs():
        cap = torch.cuda.Stream(device=dev)
        cap.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(cap):
            for _ in range(3):                  # the rasterizer keeps one workspace per stream: size this stream's
                for p_ in params:
                    p_.grad = None
                step_fn()
                cap.synchronize()
        mode = "thread_local" if world > 1 else "global"
        graphs, pool = [], None
        for slot in (0, 1):
            for p_ in params:
                p_.grad = None
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=cap, pool=pool, capture_error_mode=mode):
                cur = torch.cuda.current_stream(dev)
                up_stream.wait_stream(cur)
                down_stream.wait_stream(cur)
                with torch.cuda.stream(up_stream):
                    stage_in[slot ^ 1].copy_(host_in, non_blocking=True)
                with torch.cuda.stream(down_stream):
                    host_out[slot ^ 1].copy_(stage_out[slot ^ 1], non_blocking=True)
                with torch.no_grad():
                    flat_in.copy_(stage_in[slot])
                images = step_fn()
                with torch.no_grad():
                    for p_, o, nn_ in zip(params, offs, sizes):
                        stage_out[slot][o:o + nn_].copy_(p_.grad.reshape(-1))
                    stage_out[slot][-1:].copy_(images.sum().reshape(1))
                cur.wait_stream(up_stream)
                cur.wait_stream(down_stream)
            pool = g.pool()
            graphs.append(g)
        torch.cuda.synchronize(dev)
        return graphs

    e2e_graphs = None
    if use_graph:
        try:
            e2e_graphs = build_e2e_graphs()
        except Exception as e:
            sys.stderr.write("bench.py: capturing the end-to-end pipeline failed (%s); issuing it from Python\n" % e)
            torch.cuda.synchronize(dev)

    def upload(slot):
        with torch.cuda.stream(up_stream):
            up_stream.wait_event(ev_free[slot])
            stage_in[slot].copy_(host_in, non_blocking=True)
            ev_up[slot].record(up_stream)

    def e2e_run(n, h2d_only=False):
        if e2e_graphs is not None and not h2d_only:
            stage_in[0].copy_(host_in, non_blocking=True)          # the first step's inputs
            for i in range(n):
                e2e_graphs[i & 1].replay()
            host_out[(n - 1) & 1].copy_(stage_out[(n - 1) & 1], non_blocking=True)      # the last step's gradients
            return
        for ev in ev_free + ev_down:
            ev.record(compute_stream)
        upload(0)
        for i in range(n):
            slot = i & 1
            if i + 1 < n:
                upload(slot ^ 1)
            compute_stream.wait_event(ev_up[slot])
            with torch.no_grad():
                flat_in.copy_(stage_in[slot], non_blocking=True)
            ev_free[slot].record(compute_stream)
            if h2d_only:
                continue
            images = run_step()
            compute_stream.wait_event(ev_down[slot])      # the slot's previous read-back has left the device
            with torch.no_grad():
                for p_, o, nn_ in zip(params, offs, sizes):
                    stage_out[slot][o:o + nn_].copy_(p_.grad.reshape(-1), non_blocking=True)
                stage_out[slot][-1:].copy_(images.sum().reshape(1), non_blocking=True)
            ev_grad[slot].record(compute_stream)
            with torch.cuda.stream(down_stream):
                down_stream.wait_event(ev_grad[slot])
                host_out[slot].copy_(stage_out[slot], non_blocking=True)
                ev_down[slot].record(down_stream)
        compute_stream.wait_stream(down_stream)
        compute_stream.wait_stream(up_stream)

    def timed(fn_, n):
        barrier()
        if sampler:
            sampler.active = True
        e0.record()
        fn_(n)
        e1.record()
        barrier()
        if sampler:
            sampler.active = False
        t_ = e0.elapsed_time(e1)
        if world > 1:
            tt = torch.tensor([t_], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_ = float(tt.item())
        return t_ / n

    e2e_run(max(args.warmup, 4))
    ms_e2e = timed(e2e_run, args.steps)
    ms_h2d = timed(lambda n: e2e_run(n, h2d_only=True), args.steps)      # the upload alone, for the scaling diagnosis
    clocks = sampler.stop() if sampler else None
    e2e_value = total_views * S * S / 1e6 / (ms_e2e / 1e3)
    h2d = host_in.numel() * 4
    d2h = n_out * 4
    grad_ok = bool(torch.isfinite(host_out[(args.steps - 1) & 1]).all())

    def finish():
        """Leave without tearing NCCL down: destroy_process_group() can block for minutes on a communicator
        whose all-reduce lives in a captured CUDA graph, and nothing is left to clean up anyway."""
        torch.cuda.synchronize(dev)
        sys.stdout.flush()
        sys.stderr.flush()
        if world > 1:
            dist.barrier()
            os._exit(0)

    if rank != 0:
        finish()
        return

    # statistics of the last forward (nrBinStats; their meaning depends on the path, see include/nr_b200.h)
    bin_stats = None
    try:
        from neural_renderer_v2_pytorch_b200 import rasterize as _rz
        bin_stats = []
        for (di, st_), sc in _rz._Scratch._cache.items():
            if di == dev.index and sc.last_shape is not None:
                sc.poll(block=True)
                t_, m_, o_, b_ = sc.stats.tolist()
                bin_stats.append({"stream": "%x" % st_, "total_pairs": t_, "max_tile_faces": m_, "overflow": o_, "bad_index": b_,
                                  "path": "zbuf" if sc.last_dense else ("one-kernel binning" if sc.last_small else "general binning"),
                                  "dense_shapes": len(sc.dense), "fine_shapes": len(sc.fine_tiles)})
    except Exception:
        pass

    # ---- roofline of the dominant kernel
    peak, peak_src = peaks()
    fwd_b, bwd_b = algorithmic_bytes(inp["nv"], inp["nf"], inp["T"], R * R, C, S)
    shares = {"raster": fwd_b * B, "zbuf_faces": fwd_b * B, "backward": bwd_b * B}
    dom = max((k for k in kern if k in shares), key=lambda k: kern[k])
    achieved = shares[dom] / (kern[dom] / 1e3) / 1e9
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            with open(tpath) as f:
                tj = json.load(f)
            traffic = tj.get(args.workload, {}).get(dom) if B == WORKLOADS[args.workload]["views"] else None
            traffic_src = tj.get("_source")
        except Exception:
            traffic = None
    step_bytes = (fwd_b + bwd_b) * B
    roofline = {"bound": "hbm", "kernel": "k_" + dom, "achieved": round(achieved, 1), "peak": peak,
                "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic,
                "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": shares[dom], "kernel_ms": round(kern[dom], 4),
                "peak_source": peak_src,
                "step_frac": round(step_bytes / (ms_step / 1e3) / 1e9 / peak, 4),
                "how": "CUDA events around every launch on the launch stream, %d profiled steps right after "
                       "the timed region" % args.steps}

    cpu = cpu_baseline_sample(args.workload, budget_s=12.0) if world == 1 and not args.no_cpu_baseline else None

    line = {
        "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms_step, 4), "higher_is_better": True,
        "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(args.workload, w, inp, world, scaling, B, total_views, step_bytes),
        "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": round(ms_e2e, 4), "h2d_only_ms_per_step": round(ms_h2d, 4),
                "host_cpus_bound": numa_cpus, "gradients_finite": grad_ok,
                "pipeline": "per step: ONE pinned H2D copy of every differentiable input (uploaded on a copy stream "
                            "while the previous step runs), fwd+bwd, ONE D2H copy of EVERY gradient the step produces "
                            "+ an image checksum on a third stream; the images themselves stay on the device, as in "
                            "an optimisation loop whose loss is evaluated there; " +
                            ("the pipelined iteration is two captured CUDA graphs replayed in turn"
                             if e2e_graphs is not None else "issued from Python")},
        "gpu_launches": int(round(launches_per_step * args.steps)),
        "launch_mode": "cuda graph replay of the whole step" if use_graph else "eager (python)",
        "collective": (None if not shared or world == 1 else
                       ("none (study: gradient left un-reduced)" if args.no_collective else
                        ("fused into the camera backward kernel over NVLink peer memory"
                         if nr.parallel.fused_allowed(world) and nr.parallel._Exchange.get(inp["nv"], None, dev) is not None
                         else "ncclAllReduce"))),
        "host_ms_per_step": round(host_ms, 4),
        "clocks": clocks,
        "roofline": roofline,
        "kernels_ms": {k: round(v, 4) for k, v in kern.items()},
        "bin_stats": bin_stats,
    }
    if cpu:
        line["cpu_baseline"] = cpu
    print(json.dumps(line))
    finish()


# ------------------------------------------------------------------------------------- CPU side
def oracle_step(inp, w, views):
    """One fwd + bwd of the CPU oracle (C z-buffer / weight map with OpenMP + torch-CPU stages).
    Returns (images, leaves): the leaves carry the gradients."""
    from oracle import pipeline as ref
    v = inp["vertices"][:views].cpu().clone().requires_grad_(True)
    kw = {}
    leaves = [v]
    rgb = w["mode"] in ("rgb", "rgba")
    if rgb:
        tex = inp["textures"][:views].clone().requires_grad_(True)
        leaves.append(tex)
        kw = dict(vertices_textures=inp["vt"][:views], faces_textures=inp["ft"].numpy(),
                  textures=torch.tanh(tex) if w.get("tanh") else tex)
    img = ref.rasterize(v, inp["faces"], w["S"], w["aa"], draw_rgb=rgb,
                        draw_silhouettes=w["mode"] in ("silhouettes", "rgba"), draw_depth=w["mode"] == "depth", **kw)
    G = inp["G"][:views]
    img.backward(G if G.ndim == 4 else G[:, None])
    return img, leaves


def cpu_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_baseline_sample(workload, budget_s=12.0):
    """Times the oracle port on a bounded sample of the workload (about `budget_s` seconds)."""
    import neural_renderer_v2_pytorch_b200 as nr
    w = WORKLOADS[workload]
    cores = cpu_cores()
    torch.set_num_threads(cores)
    os.environ.setdefault("OMP_NUM_THREADS", str(cores))
    inp = make_inputs(w, seed=1000, device="cpu", nr=nr)
    oracle_step(inp, w, 1)                      # warm-up (builds / loads the C library)
    t0 = time.perf_counter()
    oracle_step(inp, w, 1)
    t1 = time.perf_counter() - t0
    views = int(max(1, min(w["views"], budget_s / max(t1, 1e-3))))
    reps, t0 = 0, time.perf_counter()
    while True:                                 # about budget_s seconds of CPU work
        oracle_step(inp, w, views)
        reps += 1
        t = time.perf_counter() - t0
        if t >= budget_s * 0.8 or reps >= 16:
            break
    return {"value": round(reps * views * w["S"] ** 2 / 1e6 / t, 3), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d x (%d of %d views of %s, one fwd+bwd), %.1f s; C z-buffer/weight-map restatement (OpenMP) + "
                      "torch-CPU stages; the reference itself has no CPU z-buffer (rasterize_cuda.cpp:60-61)"
                      % (reps, views, w["views"], workload, t)}


def run_reference(args):
    """--impl reference: the oracle port of the reference's path on the host cores.
    (oracle/_ref holds the reference's CUDA kernels, which need a GPU; the reference ships no CPU
    implementation of the z-buffer, so the CPU arm is kind = "port".)  Every step renders the WHOLE batch
    of the workload (all 64 views of config 2) as long as the run stays within a few minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import neural_renderer_v2_pytorch_b200 as nr
    world = int(os.environ.get("WORLD_SIZE", "1"))
    w = dict(WORKLOADS[args.workload])
    if args.views:
        w["views"] = args.views
    scaling = args.scaling or w.get("scaling", "weak")
    cores = cpu_cores()
    torch.set_num_threads(cores)
    inp = make_inputs(w, seed=1000, device="cpu", nr=nr)
    oracle_step(inp, w, 1)
    t0 = time.perf_counter()
    oracle_step(inp, w, min(4, w["views"]))
    t1 = (time.perf_counter() - t0) / min(4, w["views"])
    total_steps = args.steps + max(args.warmup, 1)
    views = int(max(1, min(w["views"], 280.0 / (t1 * total_steps))))
    for _ in range(max(args.warmup, 1)):
        oracle_step(inp, w, views)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle_step(inp, w, views)
    t = time.perf_counter() - t0
    value = views * w["S"] ** 2 * args.steps / 1e6 / t
    S = w["S"]
    R = S * 2 if w["aa"] else S
    fwd_b, bwd_b = algorithmic_bytes(inp["nv"], inp["nf"], inp["T"], R * R, inp["C"], S)
    V = w["views"] if scaling == "strong" else w["views"] * world
    local = (w["views"] + world - 1) // world if scaling == "strong" else w["views"]
    sample = ("each step = %s views of %s (fwd+bwd) on the host; C z-buffer/weight-map restatement (OpenMP) + "
              "torch-CPU stages" % ("all %d" % views if views == w["views"] else "%d of the %d" % (views, w["views"]),
                                     args.workload))
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 1),
            "ms_per_step": round(t / args.steps * 1e3, 2), "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(args.workload, w, inp, world, scaling, local, V, (fwd_b + bwd_b) * local),
            "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default=None, choices=["strong", "weak"],
                    help="strong: the workload's batch is sharded over the GPUs (default for config 2); "
                         "weak: every GPU renders the workload's batch (default for the others)")
    ap.add_argument("--views", type=int, default=0, help="override the workload's batch (single-GPU studies of the sharded sizes)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-collective", action="store_true",
                    help="cfg3 study only: leave the gradient of the shared mesh un-reduced (isolates the cost of the exchange)")
    ap.add_argument("--unfused-camera", action="store_true", help="cfg2r: camera transform as torch ops")
    ap.add_argument("--eager", action="store_true", help="launch every step from Python instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (the images and the gradient of "
                         "every differentiable input; rank 0's views) as DIR/<name>.npy, float32, at most 64 MB "
                         "in all: a larger output is written as a fixed seeded sample of its elements")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm sizes its batch from a timing, so its "
                 "outputs differ from run to run")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
