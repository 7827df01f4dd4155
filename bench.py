#!/usr/bin/env python
"""bench.py - images/sec of the IR-SDE reverse-diffusion sampler (BASELINE.json metric).

A "step" is ONE complete chain x_T -> x_0 (T network forwards + T fused updates) over one batch of synthetic LQ images.
Default workload (the driver's line) = BASELINE config 2: IR-SDE deraining, 8x3x256x256 per GPU, T=100, ConditionalUNet
nf=64 depth=4, bf16 tcgen05 path, CUDA-graph step replay; weak scaling, every rank owns its own 8 images, no data-path
collective (one weight broadcast before, one gather of x0 after).  The other BASELINE configs are --workload c3 / c4 / c5
(see WORKLOADS); --precision fp32x3 runs the fp32-accurate tensor-core mode (3 x tf32 split MMA) that meets the 1e-3 bound.

  python bench.py --gpus 1 --steps 3 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference                 # the UNMODIFIED reference (baseline/_ref) on the host cores
  python bench.py --impl reference --device cuda   # context number: the reference in PyTorch eager on the B200
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec at 256x256 T=100 IR-SDE"
WORKLOADS = {
    # kind "unet": ConditionalUNet(3,3,nf,depth) chain.  B: images per GPU (weak) or the fixed global batch (strong).
    "c2": dict(kind="unet", mode="sde", B=8, scaling="weak", H=256, W=256, T=100, nf=64, depth=4, max_sigma=10, eps=0.005,
               desc="BASELINE config 2: IR-SDE deraining"),
    "c3": dict(kind="unet", mode="sde", B=32, chunk=8, scaling="strong", H=256, W=256, T=100, nf=64, depth=4, max_sigma=10, eps=0.005,
               desc="BASELINE config 3: IR-SDE dehazing, global batch 32 fixed (32/N images per GPU)"),
    "c5": dict(kind="unet", mode="posterior", B=16, chunk=2, scaling="strong", H=512, W=512, T=400, nf=64, depth=4, max_sigma=10, eps=0.005,
               desc="BASELINE config 5: reverse_posterior, global batch 16 fixed (16/N images per GPU)"),
    # kind "refusion": latent UNet(3,3,64,[1,2,4],4).encode -> ConditionalNAFNet(4, 64, [1,1,1,28], 1, [1,1,1,1]) reverse_sde on
    # the latent, cut into independent tiles (tile x tile latent pixels) that are sharded over the ranks -> decode
    "c4": dict(kind="refusion", mode="sde", B=4, scaling="strong", H=1024, W=1024, T=200, max_sigma=50, eps=0.005, tile=128,
               desc="BASELINE config 4: Refusion latent shadow removal, 4x3x1024x1024 -> 4x4x256x256 latent, tile-sharded"),
    "small": dict(kind="unet", mode="sde", B=2, scaling="weak", H=64, W=64, T=10, nf=16, depth=2, max_sigma=10, eps=0.005,
                  desc="plumbing check only, never a bench line"),
    "c4small": dict(kind="refusion", mode="sde", B=2, scaling="strong", H=128, W=128, T=6, max_sigma=50, eps=0.005, tile=16,
                    desc="plumbing check only, never a bench line"),
}


def synth(B, H, W, seed=1234):
    import torch
    g = torch.Generator().manual_seed(seed)
    lq = torch.rand(B, 3, H, W, generator=g)
    return lq, g


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.p = index, None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out = self.p.communicate(timeout=5)[0]
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, pw, reasons = [], [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        loaded = [s for s, p in zip(sm, pw) if p > 300] or sm
        return {"sm_mhz": statistics.median(loaded) if loaded else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


DUMP_LIMIT = 64 << 20   # bytes written by --dump-outputs at most


def dump_outputs(dirname, arrays, seed=0):
    """Write each float tensor as dirname/<name>.npy in float32 so that two builds can be compared output for output.
    When the arrays together exceed DUMP_LIMIT, each is replaced by the same fixed, seeded sample of its flattened
    elements (sorted positions; the sample depends only on the array's size and `seed`)."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_LIMIT:
            keep = max(1, a.size * DUMP_LIMIT // total)
            idx = np.sort(np.random.default_rng(seed).choice(a.size, keep, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(dirname, name + ".npy"), a)


def build_info():
    d = {}
    try:
        for line in open(os.path.join(ROOT, "image-restoration-sde_b200", "BUILD_INFO")):
            k, _, v = line.strip().partition("=")
            d[k] = v
    except Exception:
        pass
    return d


def ncu_traffic_per_launch():
    """(mean DRAM bytes (read + write) per tcgen05 conv launch, source description) from the newest committed
    `ncu --set full` capture of this workload (profiles/rNN_conv_tc_ncu_full_one_step.csv + .meta.json), or (None, why).
    Not measured live: ncu cannot run inside a timed bench.  The description carries the commit / source hash the capture
    was taken from and whether that equals the build being timed."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_conv_tc_ncu_full_one_step.csv")))
    files = [f for f in files if "_v1_" not in f]
    if not files:
        return None, "no profiles/r*_conv_tc_ncu_full_one_step.csv"
    path = files[-1]
    try:
        rows = list(csv.DictReader(open(path)))[1:]   # first row holds the units (Mbyte)
        tot = sum(float(r["dram__bytes_read.sum"]) + float(r["dram__bytes_write.sum"]) for r in rows)
        meta = {}
        try:
            meta = json.load(open(path[:-4] + ".meta.json"))
        except Exception:
            pass
        bi = build_info()
        same = bool(meta.get("csrc_sha256")) and meta.get("csrc_sha256") == bi.get("csrc_sha256")
        same_conv = bool(meta.get("conv_tc_sha256")) and meta.get("conv_tc_sha256") == bi.get("conv_tc_sha256")
        src = ("%s: mean dram read+write bytes per launch over %d launches of one step, ncu --set full; captured from commit %s "
               "(csrc %s, conv_tc %s); this build: commit %s (csrc %s, conv_tc %s) -> %s" % (
                   os.path.relpath(path, ROOT), len(rows), meta.get("commit", "?"), meta.get("csrc_sha256", "?"),
                   meta.get("conv_tc_sha256", "?"), bi.get("commit", "?"), bi.get("csrc_sha256", "?"), bi.get("conv_tc_sha256", "?"),
                   "same sources" if same else ("same conv kernel sources (conv_tc.cu + common.cuh), other kernels changed" if same_conv
                                                else "DIFFERENT sources")))
        return tot * 1e6 / len(rows), src
    except Exception as e:
        return None, "unreadable %s: %s" % (path, e)


def usable_cores():
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(p))))
    except Exception:
        pass
    # PyTorch's CPU conv stops scaling (and on this pool's 128-thread hosts gets slower) beyond ~32 threads
    return max(1, min(n, 32))


def workload_name(wl):
    w = WORKLOADS[wl]
    if w["kind"] == "unet":
        per = "%d per GPU" % w["B"] if w["scaling"] == "weak" else "global batch %d" % w["B"]
        return ("%s: reverse_%s, %s x3x%dx%d, T=%d, ConditionalUNet nf=%d depth=%d, max_sigma=%d cosine eps=%g"
                % (w["desc"], w["mode"], per, w["H"], w["W"], w["T"], w["nf"], w["depth"], w["max_sigma"], w["eps"]))
    return ("%s: UNet(3,3,64,[1,2,4],4).encode -> ConditionalNAFNet(4,64,[1,1,1,28],1,[1,1,1,1]) reverse_%s T=%d on %dx%d latent "
            "tiles -> decode; global batch %d x3x%dx%d, max_sigma=%d" % (w["desc"], w["mode"], w["T"], w["tile"], w["tile"], w["B"],
                                                                          w["H"], w["W"], w["max_sigma"]))


def metric_name(wl):
    w = WORKLOADS[wl]
    if wl == "c2":
        return METRIC
    return "images/sec at %dx%d T=%d %s" % (w["H"], w["W"], w["T"], "IR-SDE" if w["kind"] == "unet" else "Refusion latent")


# ------------------------------------------------------------------------------------------------------------------
# reference arm: the UNMODIFIED reference (baseline/_ref, staged by baseline/make_ref.py) - its own IRSDE and
# ConditionalUNet classes, its own reverse_sde loop.  Falls back to the oracle port only when the staging is absent.
# ------------------------------------------------------------------------------------------------------------------
def _reference_objects(wl, device):
    """(sde, net, kind): the reference's own classes when baseline/_ref is staged, else None (oracle port)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    try:
        import ref_loader
    except Exception:
        return None
    if not ref_loader.available():
        return None
    w = WORKLOADS[wl]
    util, mods = ref_loader.load("deraining")
    torch.manual_seed(0)
    net = mods.ConditionalUNet(3, 3, w["nf"], w["depth"]).to(device).eval()   # the reference constructor's default init
    sde = util.IRSDE(max_sigma=w["max_sigma"], T=w["T"], schedule="cosine", eps=w["eps"], device=device)
    sde.set_model(net)
    return sde, net


def cpu_reference_sample(wl, steps_per_sample=3, threads=None, objs=None, prewarm=True):
    """The reference on host cores (PyTorch CPU fp32, all usable threads).  Bounded sample = `steps_per_sample` steps of
    the reference's own reverse loop on ONE image of the workload; every step of the chain costs the same, so
    img/s = 1 / (T * s_per_step).  Returns (images_per_s, seconds, description, kind)."""
    import torch
    w = WORKLOADS[wl]
    H, W, T, nf, depth = w["H"], w["W"], w["T"], w["nf"], w["depth"]
    threads = threads or usable_cores()
    torch.set_num_threads(threads)
    lq, g = synth(1, H, W)
    if objs is None:
        objs = _reference_objects(wl, torch.device("cpu"))
    if objs is not None:
        sde, net = objs
        xT = lq + torch.randn(lq.shape, generator=g) * sde.max_sigma
        sde.set_mu(lq)
        with torch.no_grad():
            if prewarm:
                getattr(sde, "reverse_" + w["mode"])(xT, T=1)   # untimed: thread pool / allocator warm-up
            t0 = time.perf_counter()
            getattr(sde, "reverse_" + w["mode"])(xT, T=steps_per_sample)
            dt = time.perf_counter() - t0
        kind, what = "reference", "the reference's own IRSDE.reverse_%s + ConditionalUNet (baseline/_ref)" % w["mode"]
    else:
        from oracle import irsde_oracle as O
        P = O.make_weights(3, 3, nf, depth, seed=0)
        sc = O.Schedule(w["max_sigma"], T, "cosine", w["eps"])
        xT = lq + torch.randn(lq.shape, generator=g) * sc.max_sigma
        zs = torch.randn((steps_per_sample,) + tuple(lq.shape), generator=g)
        net = lambda x, t: O.unet_forward(P, x, lq, t, nf, depth)
        with torch.no_grad():
            t0 = time.perf_counter()
            O.reverse_chain(sc, net, xT, lq, zs, w["mode"], T=steps_per_sample)
            dt = time.perf_counter() - t0
        kind, what = "port", "oracle port of the reference (baseline/_ref not staged)"
    s_per_step = dt / steps_per_sample
    return 1.0 / (T * s_per_step), dt, ("%s: %d steps of 1x3x%dx%d (nf=%d depth=%d) on %d threads; img/s extrapolated as "
                                        "1/(T*s_per_step), T=%d" % (what, steps_per_sample, H, W, nf, depth, threads, T)), kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    wl = args.workload
    w = WORKLOADS[wl]
    if w["kind"] != "unet":
        print(json.dumps({"impl": "reference", "unavailable": "reference arm is implemented for the UNet workloads (c2, c3, c5)"}))
        return
    if args.device == "cuda":
        return run_reference_cuda(args)
    objs = _reference_objects(wl, torch.device("cpu"))
    vals, secs, kind, sample = [], [], "port", ""
    for i in range(args.warmup + args.steps):
        v, dt, sample, kind = cpu_reference_sample(wl, steps_per_sample=1 if i < args.warmup else 2, objs=objs, prewarm=False)
        if i >= args.warmup:
            vals.append(v); secs.append(dt)
    value = len(vals) / sum(1.0 / v for v in vals)  # harmonic mean = total images / total time
    line = {"impl": "reference", "metric": metric_name(wl), "value": value, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * sum(secs) / len(secs),
            "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(wl), "note": "reference on the host cores, PyTorch CPU fp32; each step = a bounded "
                       "sample (2 sampler steps of one image)"},
            "cpu_baseline": {"value": value, "unit": "images/s", "cores": usable_cores(), "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_reference_cuda(args):
    """Context number (BASELINE.md 3): the reference unchanged in PyTorch eager on one B200 - cuDNN / cuBLAS library kernels,
    stock settings (cudnn.allow_tf32 stays at torch's default True, as the reference never touches it) unless --no-tf32."""
    import torch
    wl = args.workload
    w = WORKLOADS[wl]
    dev = torch.device("cuda", 0)
    if args.no_tf32:
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
    objs = _reference_objects(wl, dev)
    if objs is None:
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref not staged"}))
        return
    sde, net = objs
    B = w["B"] if w["scaling"] == "weak" else min(w["B"], w.get("chunk", w["B"]))
    lq, g = synth(B, w["H"], w["W"])
    xT = (lq + torch.randn(lq.shape, generator=g) * sde.max_sigma).to(dev)
    sde.set_mu(lq.to(dev))
    fn = getattr(sde, "reverse_" + w["mode"])
    with torch.no_grad():
        fn(xT, T=max(2, min(10, w["T"] // 10)))
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            x0 = fn(xT)
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    value = B / (ms / 1000.0)
    line = {"impl": "reference", "device": "cuda", "metric": metric_name(wl), "value": value, "unit": "images/s", "n_gpus": 1,
            "steps": args.steps, "warmup": 1, "ms_per_step": ms, "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None,
            "dtype": "f32 (cudnn tf32 %s)" % ("off" if args.no_tf32 else "on: torch default"), "data": "synthetic",
            "config": {"workload": workload_name(wl), "batch": B, "note": "UNMODIFIED reference (baseline/_ref), PyTorch eager on "
                       "the B200: library kernels only; context, not the CPU baseline"},
            "finite": bool(torch.isfinite(x0).all())}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------------------------
def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def _profile(ctx, _lib, run, nsteps):
    """Instrumented pass: CUDA events on the launching stream around every op of `nsteps` sampler steps."""
    ncat = 6
    ms_a, fl_a, n_a, by_a = ((ctypes.c_double * ncat)(), (ctypes.c_double * ncat)(), (ctypes.c_int64 * ncat)(),
                             (ctypes.c_double * ncat)())
    _lib.check(ctx.L.irsde_profile_begin(ctx.h), ctx.h)
    run()
    _lib.check(ctx.L.irsde_profile_end_bytes(ctx.h, ms_a, fl_a, n_a, by_a, ncat), ctx.h)
    names = ["tcgen05_conv", "simt_conv", "layernorm", "attention", "misc", "update"]
    bd = {names[i]: {"ms_per_step": ms_a[i] / nsteps, "ops_per_step": n_a[i] / nsteps,
                     "tflops": (fl_a[i] / (ms_a[i] * 1e-3) / 1e12) if ms_a[i] > 0 and fl_a[i] > 0 else None,
                     "algorithmic_gbs": (by_a[i] / (ms_a[i] * 1e-3) / 1e9) if ms_a[i] > 0 and by_a[i] > 0 else None}
          for i in range(ncat) if n_a[i] > 0}
    return list(ms_a), list(fl_a), list(n_a), list(by_a), bd


def run_b200(args):
    import torch
    import torch.distributed as dist
    import irsde_b200
    from irsde_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = args.workload
    w = WORKLOADS[wl]
    prec = args.precision
    T = w["T"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.manual_seed(0)
    if w["kind"] == "unet":
        # ---- model: random-init weights of the named architecture, broadcast once from rank 0
        net = irsde_b200.ConditionalUNet(3, 3, w["nf"], depth=w["depth"], precision=prec).to(dev)
        if world > 1:
            irsde_b200.broadcast_weights(net, src=0)
        sde = irsde_b200.IRSDE(w["max_sigma"], T, schedule="cosine", eps=w["eps"], device=dev)
        sde.set_model(net)
        sde.use_graph = not args.no_graph
        if w["scaling"] == "weak":
            B_glob, lo, hi = w["B"] * world, rank * w["B"], (rank + 1) * w["B"]
        else:
            B_glob = w["B"]
            lo, hi = irsde_b200.shard_range(B_glob, rank, world)
        B = hi - lo
        chunk = min(w.get("chunk", B), B) if B else 1
        lq_cpu, g = synth(B_glob, w["H"], w["W"], seed=1234)
        xT_cpu = lq_cpu + torch.randn(lq_cpu.shape, generator=g) * sde.max_sigma
        lq_cpu, xT_cpu = lq_cpu[lo:hi].contiguous(), xT_cpu[lo:hi].contiguous()
        lq, xT = lq_cpu.to(dev), xT_cpu.to(dev)
        rev = getattr(sde, "reverse_" + w["mode"])
        ctxs = [net.sync_weights(dev)]

        def chain_resident(Tn=-1):
            outs = []
            for c0 in range(0, B, chunk):
                sde.image_base = lo + c0    # per-image Philox: uid = the image's global index
                sde.set_mu(lq[c0:c0 + chunk])
                outs.append(rev(xT[c0:c0 + chunk], T=Tn))
            return outs

        lq_pin, xT_pin = lq_cpu.pin_memory(), xT_cpu.pin_memory()
        out_pin = torch.empty_like(lq_cpu).pin_memory()

        def chain_e2e():
            ys = []
            for c0 in range(0, B, chunk):
                a = lq_pin[c0:c0 + chunk].to(dev, non_blocking=True)
                b = xT_pin[c0:c0 + chunk].to(dev, non_blocking=True)
                sde.set_mu(a)
                y = rev(b)
                out_pin[c0:c0 + chunk].copy_(y, non_blocking=True)
                ys.append(y)
            if world > 1:  # the job's single gather of results; part of the step
                y = torch.cat(ys) if ys else lq.new_zeros((0,) + tuple(lq.shape[1:]))
                sizes = [irsde_b200.shard_range(B_glob, r, world) if w["scaling"] != "weak" else (r * w["B"], (r + 1) * w["B"])
                         for r in range(world)]
                mx = max(h - l for l, h in sizes)
                pad = y.new_zeros((mx,) + tuple(y.shape[1:]))
                pad[:y.shape[0]] = y
                bufs = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
                dist.gather(pad, bufs, dst=0)
        nbytes_in, nbytes_out = 2 * lq_cpu.numel() * 4, lq_cpu.numel() * 4
        par = "batch-sharded dp%d%s" % (world, ", %d-image chains" % chunk if chunk != B else "")
    else:
        # ---- Refusion: latent autoencoder + NAFNet score network, tile-sharded chain
        ae = irsde_b200.UNet(3, 3, 64, [1, 2, 4], 4, precision=prec).to(dev)
        net = irsde_b200.ConditionalNAFNet(img_channel=4, width=64, middle_blk_num=1, enc_blk_nums=[1, 1, 1, 28],
                                           dec_blk_nums=[1, 1, 1, 1], latent=True, precision=prec).to(dev)
        if world > 1:
            irsde_b200.broadcast_weights(ae, src=0)
            irsde_b200.broadcast_weights(net, src=0)
        sde = irsde_b200.IRSDE(w["max_sigma"], T, schedule="cosine", eps=w["eps"], device=dev)
        sde.set_model(net)
        sde.use_graph = not args.no_graph
        B_glob = w["B"]
        lo, hi = irsde_b200.shard_range(B_glob, rank, world)
        B = hi - lo
        lq_cpu, g = synth(B_glob, w["H"], w["W"], seed=1234)
        lq = lq_cpu.to(dev)
        pipe = irsde_b200.TiledRefusion(ae, sde, tile=w["tile"], mode=w["mode"], seed=7)
        ctxs = [net.sync_weights(dev), ae.sync_weights(dev)]

        def chain_resident(Tn=-1):
            if Tn >= 0:   # instrumented pass: a few steps of the chain on this rank's first tile batch
                z, _ = ae.encode(lq[lo:lo + 1] if B else lq[:1])
                t = w["tile"]
                tiles = torch.cat([z[:, :, y:y + t, x:x + t] for y in range(0, z.shape[2], t) for x in range(0, z.shape[3], t)])
                sde.rng, sde.seed_auto_increment = "philox", False
                sde.set_mu(tiles)
                return [getattr(sde, "reverse_" + w["mode"])(sde.noise_state(tiles), T=Tn)]
            return [pipe.restore(lq)[0]]

        lq_pin = lq_cpu.pin_memory()
        out_pin = torch.empty((B,) + tuple(lq_cpu.shape[1:])).pin_memory()

        def chain_e2e():
            a = lq_pin.to(dev, non_blocking=True)
            y, _ = pipe.restore(a)
            out_pin.copy_(y, non_blocking=True)
            if world > 1:
                mx = max(irsde_b200.shard_range(B_glob, r, world)[1] - irsde_b200.shard_range(B_glob, r, world)[0] for r in range(world))
                pad = y.new_zeros((mx,) + tuple(y.shape[1:]))
                pad[:y.shape[0]] = y
                bufs = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
                dist.gather(pad, bufs, dst=0)
        nbytes_in, nbytes_out = lq_cpu.numel() * 4, out_pin.numel() * 4
        par = "images sharded for encode/decode, %dx%d latent tiles sharded for the chain, dp%d" % (w["tile"], w["tile"], world)

    def launch_total():
        return sum(int(c.L.irsde_launch_count(c.h)) for c in ctxs if c is not None)

    # ---- (1) device-resident throughput: inputs in HBM, in-kernel Philox noise, graph replay
    sde.rng = "philox"
    for _ in range(args.warmup):
        chain_resident()
    barrier()
    l0 = launch_total()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0.record()
    for _ in range(args.steps):
        outs = chain_resident()
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = launch_total() - l0
    value = B_glob * args.steps / (ms_total / 1000.0)
    assert all(torch.isfinite(o).all() for o in outs)
    if args.dump_outputs:   # x0 of the last timed step: this rank's images in global order
        dump_outputs(args.dump_outputs, {"x0" if world == 1 else "x0_rank%d" % rank: torch.cat(outs)})

    # ---- (2) end to end through the public API with HOST buffers (pinned): H2D of the inputs, the sampler exactly as
    #          test.py drives it (UNet workloads: torch RNG, one randn_like per step), D2H of x0, the final gather
    sde.rng = "torch" if w["kind"] == "unet" else "philox"
    for _ in range(max(1, args.warmup // 3)):
        chain_e2e()
    barrier()
    e0.record()
    for _ in range(args.steps):
        chain_e2e()
    e1.record()
    barrier()
    e2e_value = B_glob * args.steps / (max_over_ranks(e0.elapsed_time(e1)) / 1000.0)

    # ---- (3) roofline of the dominant kernel: instrumented pass (CUDA events around every op of a few sampler steps,
    #          same process, right after the timed region; graph replay bypassed so each launch can be bracketed)
    roof, breakdown = None, None
    if rank == 0 and B > 0:
        peaks = _peaks()
        sde.rng = "philox"
        prof_steps = min(T, 5)
        ctx = ctxs[0]
        ms_a, fl_a, n_a, by_a, breakdown = _profile(ctx, _lib, lambda: chain_resident(prof_steps), prof_steps)
        tot_ms = sum(ms_a)
        if w["kind"] == "unet" and prec in ("bf16", "fp32x3") and ms_a[0] > 0:
            peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
            if prec == "fp32x3":
                peak_tf *= 0.5   # kind::tf32 MMA runs at half the bf16 rate; no measured tf32 GEMM peak on this pool
            ach = fl_a[0] / (ms_a[0] * 1e-3) / 1e12
            traffic, traffic_src = ncu_traffic_per_launch() if (wl == "c2" and prec == "bf16") else (None, "no ncu capture of this workload")
            roof = {"kernel": "conv_tc_persist_kernel (tcgen05 tap-GEMM conv%s)" % (", 3 x kind::tf32 split MMA" if prec == "fp32x3" else ""),
                    "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                    "peak_source": ("measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback 1.4 PF sustained "
                                    "(B200_PROFILING.md)") + (" x 0.5 for tf32" if prec == "fp32x3" else ""),
                    "flops_per_launch": fl_a[0] / n_a[0], "avg_launch_ms": ms_a[0] / n_a[0], "launches": int(n_a[0]),
                    "share_of_step": ms_a[0] / tot_ms, "traffic": traffic, "traffic_source": traffic_src,
                    "how": "executed conv FLOPs (x3 MMA passes NOT counted for fp32x3) / summed launch durations; CUDA events "
                           "around each launch, %d sampler steps, non-graph pass after the timed region" % prof_steps}
        elif w["kind"] == "unet" and ms_a[1] > 0:
            ach = fl_a[1] / (ms_a[1] * 1e-3) / 1e12
            roof = {"kernel": "conv_simt_kernel (fp32 FMA)", "bound": "tensor", "achieved": ach, "peak": 75.0, "unit": "TFLOP/s",
                    "frac": ach / 75.0, "peak_source": "nominal fp32 FMA peak (no tensor cores on this path)", "traffic": None,
                    "share_of_step": ms_a[1] / tot_ms}
        elif tot_ms > 0:
            peak_bw = float(peaks.get("hbm_gbs", 6650.0))
            ach = sum(by_a) / (tot_ms * 1e-3) / 1e9
            roof = {"kernel": "whole NAFNet sampler step (1x1-conv GEMMs, depthwise+gate, LayerNorm: HBM-bound, SURVEY 8 d)",
                    "bound": "hbm", "achieved": ach, "peak": peak_bw, "unit": "GB/s", "frac": ach / peak_bw,
                    "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6.65 TB/s", "traffic": None,
                    "bytes_per_step": sum(by_a) / prof_steps, "ms_per_step": tot_ms / prof_steps,
                    "how": "algorithmic bytes (every op's inputs + outputs + weights once) / summed op durations, CUDA events, "
                           "%d steps on one tile batch" % prof_steps}

    # ---- (4) CPU baseline (rank 0, N=1 only): bounded sample of the same workload on host cores
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and w["kind"] == "unet":
        # about 10 s of host work: 12 sampler steps of one 256x256 image (fewer at larger sizes), after one untimed step
        v, dt, sample, kind = cpu_reference_sample(wl, steps_per_sample=max(3, int(round(12 * 65536.0 / (w["H"] * w["W"])))))
        cpu = {"value": v, "unit": "images/s", "cores": usable_cores(), "kind": kind, "sample": sample, "seconds": dt}

    if rank == 0:
        line = {"metric": metric_name(wl), "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": w["scaling"],
                "vs_baseline": None, "dtype": {"bf16": "bf16", "fp32": "f32", "fp32x3": "f32 (3 x tf32 split tensor-core MMA)"}[prec],
                "data": "synthetic",
                "config": {"workload": workload_name(wl), "global_batch": B_glob, "parallelism": par, "graph": sde.use_graph,
                           "l2": "per-step activation working set (>4 GB) exceeds the 126 MB L2; no flush needed",
                           "noise": "in-kernel Philox for `value`; torch.randn_like per step (reference RNG order) for e2e"},
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": nbytes_in, "d2h_bytes_per_step": nbytes_out},
                "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu, "breakdown": breakdown,
                "device_bytes": sum(int(c.L.irsde_device_bytes(c.h)) for c in ctxs if c is not None), "build": dict(build_info(), **{k: os.environ[k] for k in ("IRSDE_HBM_NEW", "IRSDE_LN_PP") if k in os.environ})}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=list(WORKLOADS))
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32", "fp32x3"])
    ap.add_argument("--device", default="cpu", choices=["cpu", "cuda"], help="reference arm only: where the reference runs")
    ap.add_argument("--no-tf32", action="store_true", help="reference arm on cuda: disable cuDNN/cuBLAS TF32")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="B200 arm: write x0 of the last timed step as DIR/x0.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
