#!/usr/bin/env python3
"""bench.py -- headline benchmark (contract in the task statement; layout in DESIGN.md section 5).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-extras] [--step-path module|functional]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = Correlation forward + backward (both input gradients) at BASELINE.json configs[1]:
fp32 [8,256,112,256] per GPU, pad=20,k=1,md=20,s1=1,s2=2 (D=441).  Weak scaling: every rank owns
its own 8-sample shard, no data-path collective (the layers are per-sample; SURVEY 8e).

metric/value : algorithmic GB/s of fwd+bwd (read each input once + write each output once,
               2 218 524 672 B per 8-sample step, SURVEY 8d) summed over ranks, inputs resident in HBM.
e2e          : same metric with HOST buffers: every step copies f1,f2,gradOutput from pinned host
               memory and copies output,gradInput1,gradInput2 back, through the package's
               hostpipe.HostPipeline (H2D / kernels / D2H of consecutive steps overlap on three streams).
roofline     : the dominant kernel (correlation backward) timed alone with CUDA events; achieved =
               its algorithmic bytes per launch / its duration, against MEASURED_PEAKS.json's HBM GB/s.
cpu_baseline : the CPU oracle (oracle/oracle.c, a port -- the reference has no CPU path) on a 1-sample
               slice of the same workload, all host cores.
--impl reference: the reference's OWN CUDA kernels rebuilt for sm_100a (oracle/_ref) on the same
               workload on the same GPU; if they are not built, the CPU oracle port instead.
flownet2     : image-pairs/s of the unmodified reference models (random weights, 448x1024, bs 8 per GPU) on our
               drop-in layers and through flownet2_b200.fused (glue folded into our kernels); `agreement` = max|d|/max|ref|
               of the output flow against the same network on the reference's own kernels, same seeded input,
               deterministic cuDNN, TF32 off (the reference output is computed in a child process: --flow-ref).
Host staging buffers are allocated after binding the rank to its GPU's NUMA node (flownet2_b200.numa).
--dump-outputs DIR: rank 0 writes what the last timed step returned (output, grad_input1, grad_input2) as DIR/<name>.npy,
               float32; the inputs are seeded, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CFG = dict(B=8, C=256, H=112, W=256, pad=20, k=1, md=20, s1=1, s2=2)
D = 441


def alg_bytes(B):
    """SURVEY 8(d): fwd 4*(2*B*C*H*W + B*D*oH*oW); bwd 4*(B*D*oH*oW + 4*B*C*H*W)."""
    chw = CFG["C"] * CFG["H"] * CFG["W"]
    dhw = D * CFG["H"] * CFG["W"]
    fwd = 4 * (2 * B * chw + B * dhw)
    bwd = 4 * (B * dhw + 4 * B * chw)
    bwd_launch = 4 * (B * dhw + 2 * B * chw)     # one gradInput: gradOutput + other input + output
    return fwd, bwd, bwd_launch


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (NVML in a thread, 5 ms period;
    falls back to the nvidia-smi loop of B200_PROFILING.md when pynvml is unusable)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, cuda_index):
        self.idx, self.rows, self._stop, self.h, self.proc, self.t = cuda_index, [], False, None, None, None

    def start(self):
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(self.idx).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
        except Exception:
            self.h = None
            self._start_smi()

    def _nvml_loop(self):
        nv = self.nv
        while not self._stop:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.rows.append((time.time(), sm, self.max_mhz, mask))
            except Exception:
                pass
            time.sleep(0.005)

    def _start_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._smi_loop, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _smi_loop(self):
        bits = [0x8, 0x40, 0x20, 0x4]
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                mask = sum(b for b, v in zip(bits, f[2:6]) if v.lower().startswith("active"))
                self.rows.append((time.time(), float(f[0]), float(f[1]), mask))
            except Exception:
                pass

    def window(self, t0, t1):
        rows = [r for r in self.rows if t0 <= r[0] <= t1]
        sm = sorted(r[1] for r in rows)
        mask = 0
        for r in rows:
            mask |= r[3]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": max(r[2] for r in rows) if rows else None,
                "reasons": sorted(n for b, n in self.REASONS.items() if mask & b), "samples": len(sm)}

    def stop(self):
        self._stop = True
        if self.proc:
            self.proc.terminate()


DUMP_ELEMENTS = 1 << 22     # per array: 16 MB of float32, 48 MB for the three outputs of a step


def dump_outputs(out_dir, arrays):
    """Write each tensor as out_dir/<name>.npy in float32: whole if it has at most DUMP_ELEMENTS elements, else the
    elements at DUMP_ELEMENTS sorted flat indices drawn from a fixed seed (the same positions in every run)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_ELEMENTS:
            idx = torch.randint(t.numel(), (DUMP_ELEMENTS,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def time_loop(fn, steps, warmup, sync, dist_barrier=None):
    """W untimed + K timed calls of fn() between CUDA events on the current stream."""
    import torch
    for _ in range(warmup):
        fn()
    if dist_barrier:
        dist_barrier()
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    sync()
    if dist_barrier:
        dist_barrier()
    t1 = time.time()
    return e0.elapsed_time(e1), t0, t1


def time_cold(fn, iters, flush):
    """Per-iteration event timing with an L2 flush (write > L2 bytes) before each call."""
    import torch
    ms = []
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    ms.sort()
    return ms[len(ms) // 2]


def time_rotating(make_call, nsets, reps=3):
    """Back-to-back launches over `nsets` DISTINCT buffer sets (footprint > 2x L2, so every launch
    sees cold L2) inside ONE event pair: launch latency is amortised, unlike time_cold.
    make_call(i) -> zero-arg callable bound to buffer set i.  Returns median ms per launch."""
    import torch
    calls = [make_call(i) for i in range(nsets)]
    for c in calls:
        c()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for c in calls:
            c()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / nsets)
    out.sort()
    return out[len(out) // 2]


def load_by_path(name, filename):
    import importlib.util
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "flownet2-pytorch_b200", filename))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def numa_bind(local):
    """Pin this rank (CPU affinity + preferred memory node) to its GPU's NUMA node before any pinned allocation."""
    try:
        return load_by_path("_fn2_numa", "numa.py").bind_to_device_node(local)
    except Exception as e:
        return {"node": None, "error": str(e)[:100]}


def profiled_traffic():
    """dram__bytes_read+write per launch of the correlation kernels from a COMMITTED ncu capture (profiles/ncu_traffic.json),
    valid only for the library sources it was taken on: keyed by the product source digest.  None when stale / absent."""
    try:
        digest = load_by_path("_fn2_build", "build.py").product_digest()
        table = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        ent = table.get(digest)
        if ent:
            ent = dict(ent)
            ent["digest"] = digest
        return ent
    except Exception:
        return None


def load_host_pipeline(impl):
    """The package's HostPipeline; for the reference arm the module (stream plumbing only, imports nothing but torch)
    is loaded by path so that libfn2b200.so stays out of that process."""
    if impl == "ours":
        from flownet2_b200.hostpipe import HostPipeline
        return HostPipeline
    import importlib.util
    spec = importlib.util.spec_from_file_location("_fn2_hostpipe", os.path.join(ROOT, "flownet2-pytorch_b200", "hostpipe.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.HostPipeline


FLOW_SEED = 0


def _flow_check_input(batch):
    import torch
    g = torch.Generator().manual_seed(1234)
    return torch.rand(batch, 3, 2, 448, 1024, generator=g) * 255.0


def _build_model(impl, model_name, dev):
    import torch
    from types import SimpleNamespace
    from oracle import ref as oref
    if impl == "ours":
        from flownet2_b200 import compat
        compat.install("B2")
    else:
        oref.install_reference_extensions()
    models = oref.import_reference_models(fresh=True)
    torch.manual_seed(FLOW_SEED)
    return getattr(models, model_name)(SimpleNamespace(rgb_max=255.0, fp16=False)).to(dev).eval()


def _deterministic(on):
    import torch
    torch.backends.cudnn.deterministic = on
    torch.backends.cudnn.benchmark = not on
    torch.backends.cudnn.allow_tf32 = not on
    torch.backends.cuda.matmul.allow_tf32 = not on


def flow_ref_child(model_names, out_dir, batch=8):
    """--flow-ref: the reference kernels' output flow for the seeded check input, one .npy per model (child process of
    the ours arm, so that the reference extensions never share a process with libfn2b200.so)."""
    import numpy as np
    import torch
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    _deterministic(True)
    x = _flow_check_input(batch).to(dev)
    for name in model_names:
        net = _build_model("reference", name, dev)
        with torch.no_grad():
            np.save(os.path.join(out_dir, name + ".npy"), net(x).float().cpu().numpy())
        del net
        torch.cuda.empty_cache()


def flownet2_pairs_per_sec(impl, dev, model_name="FlowNet2", batch=8, steps=5, warmup=2, ref_dir=None):
    """BASELINE configs[3]/[4]: the UNMODIFIED reference models.py (baseline/_ref) on top of our layers
    (B2 hooks) or of the reference's own kernels; random xavier weights, U(0,255) input
    [batch,3,2,448,1024], no_grad; H2D copy of the pinned input and D2H of the flow inside the loop
    (hostpipe.HostPipeline: they overlap with the previous / next batch's kernels, for both arms).
    ours arm: also the fused forwards (flownet2_b200.fused) and the output-flow agreement with the reference kernels."""
    import numpy as np
    import torch
    from oracle import ref as oref
    if not oref.python_tree_available():
        return {"unavailable": "baseline/_ref/flownet2_pytorch not installed (oracle/build_ref.py)"}
    if impl != "ours" and not oref.available():
        return {"unavailable": "oracle/_ref reference extensions not built"}
    net = _build_model(impl, model_name, dev)
    res = {"model": model_name, "batch_per_gpu": batch}
    if impl == "ours":
        from flownet2_b200 import fused
        if ref_dir and os.path.isfile(os.path.join(ref_dir, model_name + ".npy")):
            _deterministic(True)
            ref = np.load(os.path.join(ref_dir, model_name + ".npy"))
            xc = _flow_check_input(batch).to(dev)
            with torch.no_grad():
                o_mod = net(xc).float().cpu().numpy()
            o_fus = fused.fused_forward(net, xc).float().cpu().numpy()
            den = float(np.abs(ref).max())
            res["agreement"] = {"what": "max|d|/max|ref| of the output flow vs the same network on the reference's kernels, "
                                        "448x1024 bs %d, seeded input, deterministic cuDNN, TF32 off" % batch,
                                "drop_in_modules": float(np.abs(o_mod - ref).max() / den),
                                "fused_forward": float(np.abs(o_fus - ref).max() / den), "max_abs_ref": den}
            del xc
        else:
            res["agreement"] = None
    _deterministic(False)
    host = (torch.rand(batch, 3, 2, 448, 1024) * 255.0).pin_memory()
    hout = torch.empty(batch, 2, 448, 1024).pin_memory()
    pipe = load_host_pipeline(impl)([host.shape], [hout.shape], dev, depth=2)

    def timed(forward):
        def compute(din, dout):
            with torch.no_grad():
                dout[0].copy_(forward(din[0]))

        def step():          # H2D of the next batch and D2H of the previous flow overlap with the network
            pipe.submit(compute, (host,), (hout,))
        for _ in range(warmup):
            step()
        pipe.drain()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        pipe.drain()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps
    ms = timed(net)
    res.update({"ms_per_batch": round(ms, 3), "pairs_per_sec_per_gpu": round(batch / ms * 1e3, 2),
                "finite": bool(torch.isfinite(hout).all())})
    if impl == "ours":
        ms_f = timed(lambda x: fused.fused_forward(net, x))
        res["fused"] = {"ms_per_batch": round(ms_f, 3), "pairs_per_sec_per_gpu": round(batch / ms_f * 1e3, 2),
                        "finite": bool(torch.isfinite(hout).all()),
                        "what": "flownet2_b200.fused: correlation + LeakyReLU written into the 473-channel concat; upsample + warp + "
                                "diff + channel-norm + concat groups as one kernel each"}
    del net, pipe
    torch.cuda.empty_cache()
    return res


def cpu_baseline_sample(runs=3):
    """CPU oracle port on ONE sample of the workload (1/8 step), all host cores: median of `runs` warmed runs."""
    import numpy as np
    from oracle import cpu as orc
    rng = np.random.RandomState(0)
    shp = (1, CFG["C"], CFG["H"], CFG["W"])
    a, b = rng.randn(*shp).astype(np.float32), rng.randn(*shp).astype(np.float32)
    prm = (CFG["pad"], CFG["k"], CFG["md"], CFG["s1"], CFG["s2"])
    out = orc.correlation_forward(a, b, *prm)                      # build + warm (threads, pages)
    go = rng.randn(*out.shape).astype(np.float32)
    orc.correlation_backward(a, b, go, *prm)
    tf, tb = [], []
    for _ in range(runs):
        t0 = time.time()
        orc.correlation_forward(a, b, *prm)
        t1 = time.time()
        orc.correlation_backward(a, b, go, *prm)
        t2 = time.time()
        tf.append(t1 - t0)
        tb.append(t2 - t1)
    tf.sort()
    tb.sort()
    fwd, bwd, _ = alg_bytes(1)
    secs = tf[len(tf) // 2] + tb[len(tb) // 2]
    return {"value": round((fwd + bwd) / secs / 1e9, 4), "unit": "GB/s", "cores": os.cpu_count(), "kind": "port",
            "sample": "1 of 8 samples of the cfg2 step, median of %d warmed runs (fwd %.2fs + bwd %.2fs), OpenMP on all cores"
                      % (runs, tf[len(tf) // 2], tb[len(tb) // 2])}


def build_impl(impl, dev):
    """Returns (name, fwd(f1,f2,out), bwd(f1,f2,gO,g1,g2), launches()) for the chosen arm."""
    import torch
    prm = (CFG["pad"], CFG["k"], CFG["md"], CFG["s1"], CFG["s2"])
    if impl == "ours":
        import flownet2_b200
        F2 = flownet2_b200.functional

        state = {"ws": None}     # forward -> backward workspace hand-over, as the autograd Function does

        def fwd(a, b, out):
            _, state["ws"] = F2.correlation_forward(a, b, *prm, 1, out=out, return_workspace=True)

        def bwd(a, b, go, g1, g2):
            F2.correlation_backward(a, b, go, *prm, 1, out1=g1, out2=g2, workspace=state["ws"])
        return "ours", fwd, bwd, F2.launch_count
    from oracle import ref as oref
    ext = oref.load_extension("correlation_cuda")
    if ext is None:
        return None, None, None, None
    scratch = [torch.empty(0, device=dev) for _ in range(2)]
    count = [0]

    def fwd(a, b, out):
        ext.forward(a, b, scratch[0], scratch[1], out, *prm, 1)
        count[0] += 3

    def bwd(a, b, go, g1, g2):
        ext.backward(a, b, scratch[0], scratch[1], go, g1, g2, *prm, 1)
        count[0] += 2 + 2 * a.shape[0]
    return "reference-cuda", fwd, bwd, lambda: count[0]


def extras_ours(dev):
    """cfg3 Resample2d / ChannelNorm kernels and the true FlowNet2 correlation shape: median ms per
    launch over rotating buffer sets (cold L2, launch latency amortised), GB/s of algorithmic bytes.
    Outside the headline timed region."""
    import torch
    import flownet2_b200
    F2 = flownet2_b200.functional
    peak, _ = measured_peak()
    res = {}
    g = torch.Generator(device=dev).manual_seed(0)
    B, H, W = 8, 448, 1024
    hw = B * H * W * 4
    NS = 8

    def rec(name, make_call, nbytes, nsets=NS):
        ms = time_rotating(make_call, nsets)
        res[name] = {"ms": round(ms, 4), "GBps": round(nbytes / ms / 1e6, 1), "frac_hbm": round(nbytes / ms / 1e6 / peak, 3)}

    imgs = [torch.rand(B, 3, H, W, device=dev, generator=g) for _ in range(NS)]
    flows = [torch.randn(B, 2, H, W, device=dev, generator=g) * 4 for _ in range(NS)]
    gos = [torch.randn(B, 3, H, W, device=dev, generator=g) for _ in range(NS)]
    o3 = [torch.empty(B, 3, H, W, device=dev) for _ in range(NS)]
    o2 = [torch.empty(B, 2, H, W, device=dev) for _ in range(NS)]
    o1 = [torch.empty(B, 1, H, W, device=dev) for _ in range(NS)]
    rec("resample2d_fwd", lambda i: (lambda: F2.resample2d_forward(imgs[i], flows[i], out=o3[i])), hw * 8)
    rec("resample2d_bwd", lambda i: (lambda: F2.resample2d_backward(imgs[i], flows[i], gos[i], out1=o3[i], out2=o2[i])), hw * 13)
    rec("channelnorm_fwd_c3", lambda i: (lambda: F2.channelnorm_forward(imgs[i], out=o1[i])), hw * 4)
    rec("channelnorm_bwd_c3", lambda i: (lambda: F2.channelnorm_backward(imgs[i], o1[i], o1[(i + 1) % NS], out=o3[i])), hw * 8)
    rec("channelnorm_fwd_c2", lambda i: (lambda: F2.channelnorm_forward(flows[i], out=o1[i])), hw * 3)
    rec("channelnorm_bwd_c2", lambda i: (lambda: F2.channelnorm_backward(flows[i], o1[i], o1[(i + 1) % NS], out=o2[i])), hw * 6)
    # 16-bit storage variants (SURVEY 8f-4): half the bytes of the fp32 kernels
    himgs = [t.half() for t in imgs]
    ho1 = [torch.empty(B, 1, H, W, device=dev, dtype=torch.float16) for _ in range(NS)]
    ho3 = [torch.empty(B, 3, H, W, device=dev, dtype=torch.float16) for _ in range(NS)]
    rec("channelnorm_fwd_c3_fp16", lambda i: (lambda: F2.channelnorm_forward(himgs[i], out=ho1[i])), hw * 2)
    rec("channelnorm_bwd_c3_fp16", lambda i: (lambda: F2.channelnorm_backward(himgs[i], ho1[i], ho1[(i + 1) % NS], out=ho3[i])), hw * 4)
    del himgs, ho1, ho3
    # hot L2 (the same buffer set every launch; working sets of 117-191 MB vs 126 MB of L2: partly resident)
    rec("resample2d_fwd_hotL2", lambda i: (lambda: F2.resample2d_forward(imgs[0], flows[0], out=o3[0])), hw * 8)
    rec("resample2d_bwd_hotL2", lambda i: (lambda: F2.resample2d_backward(imgs[0], flows[0], gos[0], out1=o3[0], out2=o2[0])), hw * 13)
    rec("channelnorm_fwd_c3_hotL2", lambda i: (lambda: F2.channelnorm_forward(imgs[0], out=o1[0])), hw * 4)
    rec("channelnorm_bwd_c3_hotL2", lambda i: (lambda: F2.channelnorm_backward(imgs[0], o1[0], o1[1], out=o3[0])), hw * 8)
    # sigma = 64 px flows: more than half of the taps clamp to the border (SURVEY 8d cfg3)
    for fl in flows:
        fl.mul_(16.0)
    rec("resample2d_fwd_sigma64", lambda i: (lambda: F2.resample2d_forward(imgs[i], flows[i], out=o3[i])), hw * 8)
    rec("resample2d_bwd_sigma64", lambda i: (lambda: F2.resample2d_backward(imgs[i], flows[i], gos[i], out1=o3[i], out2=o2[i])), hw * 13)
    # SURVEY 8(f)-1/3: upsample + warp + diff + channel-norm + concat as one kernel vs the chain of modules (models.py:130-138)
    xs = [torch.rand(B, 6, H, W, device=dev, generator=g) - 0.5 for _ in range(4)]
    lrs = [torch.randn(B, 2, H // 4, W // 4, device=dev, generator=g) * 0.2 for _ in range(4)]
    cats = [torch.empty(B, 12, H, W, device=dev) for _ in range(4)]
    up = torch.nn.Upsample(scale_factor=4, mode="bilinear")
    rs_m, cn_m = flownet2_b200.Resample2d(), flownet2_b200.ChannelNorm()

    def chain(i):
        def run():
            with torch.no_grad():
                fl = up(lrs[i] * 20.0)
                warped = rs_m(xs[i][:, 3:], fl)
                torch.cat((xs[i], warped, fl / 20.0, cn_m(xs[i][:, :3] - warped)), dim=1, out=cats[i])
        return run
    alg_fused = hw * (6 + 12) + B * 2 * (H // 4) * (W // 4) * 4
    rec("warp_concat_fused", lambda i: (lambda: F2.warp_concat_forward(xs[i], lrs[i], upsample="bilinear", flow_mul=20.0,
                                                                        flow_div=20.0, out=cats[i])), alg_fused, 4)
    rec("warp_concat_chain_of_modules", chain, alg_fused, 4)
    del xs, lrs, cats
    del imgs, flows, gos, o3, o2, o1
    # correlation at the shape FlowNet2 really produces at 448x1024 (SURVEY appendix)
    a = [torch.randn(8, 256, 56, 128, device=dev, generator=g) for _ in range(2)]
    b = [torch.randn(8, 256, 56, 128, device=dev, generator=g) for _ in range(2)]
    o = [torch.empty(8, 441, 56, 128, device=dev) for _ in range(2)]
    gO = [torch.randn(8, 441, 56, 128, device=dev, generator=g) for _ in range(2)]
    g1 = [torch.empty_like(a[0]) for _ in range(2)]
    g2 = [torch.empty_like(a[0]) for _ in range(2)]
    rec("correlation_fwd_56x128", lambda i: (lambda: F2.correlation_forward(a[i], b[i], 20, 1, 20, 1, 2, out=o[i])), 218595328, 2)
    rec("correlation_bwd_56x128", lambda i: (lambda: F2.correlation_backward(a[i], b[i], gO[i], 20, 1, 20, 1, 2, out1=g1[i], out2=g2[i])),
        336035840, 2)
    # fused epilogue (SURVEY 8f-2): LeakyReLU(0.1)(corr) written into channels 32.. of the 473-channel concat buffer
    cat = [torch.empty(8, 473, 56, 128, device=dev) for _ in range(2)]
    rec("correlation_fwd_cat_leaky_56x128", lambda i: (lambda: F2.correlation_forward_cat(a[i], b[i], cat[i], 32, 0.1, 20, 1, 20, 1, 2)),
        218595328, 2)

    def corr_chain(i):
        def run():
            torch.cat((cat[i][:, :32], torch.nn.functional.leaky_relu(F2.correlation_forward(a[i], b[i], 20, 1, 20, 1, 2, out=o[i]), 0.1, inplace=True)), 1)
        return run
    rec("correlation_fwd_then_leaky_then_cat_56x128", corr_chain, 218595328, 2)
    del a, b, o, gO, g1, g2, cat
    # a C < 256 shape (single TMA producer in the forward, 2 k-blocks): [8,128,112,256]
    a = [torch.randn(8, 128, 112, 256, device=dev, generator=g) for _ in range(2)]
    b = [torch.randn(8, 128, 112, 256, device=dev, generator=g) for _ in range(2)]
    o = [torch.empty(8, 441, 112, 256, device=dev) for _ in range(2)]
    g1 = [torch.empty_like(a[0]) for _ in range(2)]
    g2 = [torch.empty_like(a[0]) for _ in range(2)]
    nb_f = 4 * (2 * 8 * 128 * 112 * 256 + 8 * 441 * 112 * 256)
    nb_b = 4 * (8 * 441 * 112 * 256 + 4 * 8 * 128 * 112 * 256)
    rec("correlation_fwd_c128_112x256", lambda i: (lambda: F2.correlation_forward(a[i], b[i], 20, 1, 20, 1, 2, out=o[i])), nb_f, 2)
    rec("correlation_bwd_c128_112x256", lambda i: (lambda: F2.correlation_backward(a[i], b[i], o[i], 20, 1, 20, 1, 2, out1=g1[i], out2=g2[i])),
        nb_b, 2)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--flow-ref", nargs="+", metavar=("OUT_DIR", "MODEL"), help=argparse.SUPPRESS)
    ap.add_argument("--step-path", default="module", choices=["module", "functional"],
                    help="ours arm: time the nn.Module + autograd step (default, the call a user makes) or the functional C-ABI calls")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float32; a fixed sample of large arrays)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.flow_ref:                      # child of the ours arm: reference-kernel output flows for the agreement check
        flow_ref_child(args.flow_ref[1:], args.flow_ref[0])
        return

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_info = numa_bind(local)           # before any pinned allocation: staging buffers on the GPU's own NUMA node
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    name, fwd, bwd, launches = build_impl(args.impl, dev)
    cpu_only_reference = args.impl == "reference" and name is None
    if cpu_only_reference:
        # reference kernels not built: the arm is the CPU oracle port, rank 0 only
        if rank == 0:
            cb = cpu_baseline_sample()
            line = {"impl": "reference", "metric": "correlation_fwd_bwd_algorithmic_GBps", "value": cb["value"],
                    "unit": "GB/s", "n_gpus": args.gpus, "steps": 1, "warmup": 0, "ms_per_step": None,
                    "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                    "data": "synthetic", "config": {"workload": "cfg2 correlation fwd+bwd, 1-sample CPU slice"},
                    "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "GB/s", "h2d_bytes_per_step": 0,
                                                "d2h_bytes_per_step": 0}}
            print(json.dumps(line))
        if dist:
            dist.destroy_process_group()
        return

    B = CFG["B"]
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    shp = (B, CFG["C"], CFG["H"], CFG["W"])
    f1 = torch.randn(*shp, device=dev, generator=g)
    f2 = torch.randn(*shp, device=dev, generator=g)
    out = torch.empty(B, D, CFG["H"], CFG["W"], device=dev)
    gO = torch.randn(B, D, CFG["H"], CFG["W"], device=dev, generator=g)
    g1, g2 = torch.empty_like(f1), torch.empty_like(f2)

    def sync():
        torch.cuda.synchronize()

    def barrier():
        if dist:
            dist.barrier()

    if args.impl == "ours" and args.step_path == "module":
        # the call a user makes: the nn.Module (autograd Function) forward, then backward of both input gradients;
        # the Function keeps the forward's bf16 hi/lo workspace for its backward
        import flownet2_b200
        corr = flownet2_b200.Correlation(CFG["pad"], CFG["k"], CFG["md"], CFG["s1"], CFG["s2"], 1)
        f1.requires_grad_(True)
        f2.requires_grad_(True)
        last = {}

        def step():
            o = corr(f1, f2)
            last["output"] = o.detach()
            last["grad_input1"], last["grad_input2"] = torch.autograd.grad(o, (f1, f2), gO)
        step_how = "flownet2_b200.Correlation module forward + autograd backward (torch.autograd.grad), both input gradients"
    else:
        last = {"output": out, "grad_input1": g1, "grad_input2": g2}

        def step():
            fwd(f1, f2, out)
            bwd(f1, f2, gO, g1, g2)
        step_how = ("flownet2_b200.functional.correlation_forward + correlation_backward (workspace handed over)" if args.impl == "ours"
                    else "correlation_cuda.forward + correlation_cuda.backward of the reference extension")

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    K, Wm = args.steps, args.warmup
    l0 = launches()
    step()
    launches_timed = (launches() - l0) * K      # kernels launched per step x timed steps
    ms, t0, t1 = time_loop(step, K, Wm, sync, barrier if dist else None)
    clocks = sampler.window(t0, t1) if rank == 0 else None
    if args.dump_outputs and rank == 0:         # before the kernel timings below overwrite out / g1 / g2
        dump_outputs(args.dump_outputs, last)
    last.clear()

    # dominant-kernel timing (alone, same stream): forward kernel, backward kernels
    f1, f2 = f1.detach(), f2.detach()
    ms_f, _, _ = time_loop(lambda: fwd(f1, f2, out), K, 2, sync)
    ms_b, _, _ = time_loop(lambda: bwd(f1, f2, gO, g1, g2), K, 2, sync)

    # end-to-end through host buffers
    hf1, hf2, hgO = (torch.empty(t.shape, pin_memory=True).copy_(t) for t in (f1, f2, gO))
    hout, hg1, hg2 = (torch.empty(t.shape, pin_memory=True) for t in (out, g1, g2))
    h2d = sum(t.numel() * 4 for t in (hf1, hf2, hgO))
    d2h = sum(t.numel() * 4 for t in (hout, hg1, hg2))

    # Public entry point for host-resident data: flownet2_b200.hostpipe.HostPipeline (three streams, two sets of
    # device buffers): every step copies all three inputs H2D and all three results D2H; the D2H of step i and
    # the H2D of step i+1 share the full-duplex link.  Both arms go through the same pipeline.
    HostPipeline = load_host_pipeline(args.impl)
    pipe = HostPipeline([f1.shape, f2.shape, gO.shape], [out.shape, g1.shape, g2.shape], dev, depth=2)

    def e2e_compute(din, dout):
        fwd(din[0], din[1], dout[0])
        bwd(din[0], din[1], din[2], dout[1], dout[2])

    def e2e_step():
        pipe.submit(e2e_compute, (hf1, hf2, hgO), (hout, hg1, hg2))
    for _ in range(2):
        e2e_step()
    pipe.drain()
    if dist:
        barrier()
    sync()
    ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ee0.record()
    for _ in range(K):
        e2e_step()
    pipe.drain()
    ee1.record()
    sync()
    if dist:
        barrier()
    ms_e = ee0.elapsed_time(ee1)
    e2e_check = float((hg1 - g1.cpu()).abs().max()) if args.impl == "ours" else 0.0   # same inputs -> same result as the resident step

    stats = torch.tensor([ms, ms_e], device=dev, dtype=torch.float64)
    stats_min = stats.clone()
    if dist:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(stats_min, op=dist.ReduceOp.MIN)
    ms, ms_e = float(stats[0]), float(stats[1])
    ms_fastest_rank = float(stats_min[0])

    # second half of BASELINE.json's metric: FlowNet2 image-pairs/sec (every rank runs a replica)
    flow = {}
    if not args.no_extras:
        del pipe, hf1, hf2, hgO, hout, hg1, hg2, f1, f2, out, gO, g1, g2
        torch.cuda.empty_cache()
        mnames = ["FlowNet2C", "FlowNet2"] if world == 1 else ["FlowNet2"]
        ref_dir = None
        if args.impl == "ours" and rank == 0:
            # reference-kernel output flows for the agreement check, from a child process (rank 0 only)
            import tempfile
            ref_dir = tempfile.mkdtemp(prefix="fn2_flowref_")
            try:
                env = dict(os.environ, LOCAL_RANK=str(local))
                for k in ("RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID"):
                    env.pop(k, None)
                subprocess.run([sys.executable, os.path.abspath(__file__), "--flow-ref", ref_dir] + mnames, env=env, timeout=900,
                               stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, check=False)
            except Exception:
                pass
        if dist:
            barrier()
        for mname in mnames:
            try:
                r = flownet2_pairs_per_sec(args.impl, dev, mname, batch=8, steps=4 if args.impl == "reference" else 8, ref_dir=ref_dir)
            except Exception as e:
                r = {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:200])}
            if "ms_per_batch" in r:
                t = torch.tensor([r["ms_per_batch"]], device=dev, dtype=torch.float64)
                if dist:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                r["ms_per_batch_max_over_ranks"] = round(float(t[0]), 3)
                r["pairs_per_sec_total"] = round(8 * world / float(t[0]) * 1e3, 2)
            flow[mname] = r

    fwd_b, bwd_b, bwd_launch_b = alg_bytes(B)
    total_b = (fwd_b + bwd_b) * world
    value = total_b * K / (ms * 1e-3) / 1e9
    e2e_value = total_b * K / (ms_e * 1e-3) / 1e9
    peak, peak_src = measured_peak()

    if rank == 0:
        per_f, per_b = ms_f / K, ms_b / K
        dominant = "correlation_backward" if per_b >= per_f else "correlation_forward"
        kname = {"correlation_backward": "corr_bwd_tc_kernel (both input gradients in one launch)",
                 "correlation_forward": "corr_tc_split_kernel + corr_fwd_tc_kernel"}[dominant] if args.impl == "ours" else dominant
        if dominant == "correlation_backward":
            launch_ms = per_b          # ours: ONE launch computes both gradients; reference: all its launches
            ach = bwd_b / (launch_ms * 1e-3) / 1e9
        else:
            launch_ms = per_f
            ach = fwd_b / (per_f * 1e-3) / 1e9
        # DRAM traffic per launch: from the committed ncu capture IF it was taken on exactly these library sources
        # (profiles/ncu_traffic.json keyed by the source digest); never attached to the reference arm; null when stale.
        prof = profiled_traffic() if args.impl == "ours" else None
        traffic = traffic_fwd = None
        if prof:
            traffic = prof.get("corr_bwd_tc_kernel") if dominant == "correlation_backward" else (
                (prof.get("corr_fwd_tc_kernel") or 0) + (prof.get("corr_tc_split_kernel") or 0) or None)
            if prof.get("corr_fwd_tc_kernel") and prof.get("corr_tc_split_kernel"):
                traffic_fwd = prof["corr_fwd_tc_kernel"] + prof["corr_tc_split_kernel"]
        roofline = {"bound": "hbm", "kernel": kname, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                    "frac": round(ach / peak, 4), "traffic": traffic,
                    "traffic_source": ("dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full, %s (sources %s)"
                                       % (prof.get("source", "profiles/"), prof["digest"][:12])) if prof else
                                      "no committed ncu capture matches these library sources (profiles/ncu_traffic.json)",
                    "traffic_forward_incl_split_pass": traffic_fwd,
                    "algorithmic_bytes": bwd_b if dominant == "correlation_backward" else fwd_b,
                    "peak_source": peak_src, "launch_ms": round(launch_ms, 4),
                    "fp32_tflops": round((51.79e9 * 3) / ((per_f + per_b) * 1e-3) / 1e12, 2)}
        if prof and prof.get("note"):
            roofline["note"] = prof["note"]
        line = {
            "metric": "correlation_fwd_bwd_algorithmic_GBps", "value": round(value, 2), "unit": "GB/s",
            "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": round(ms / K, 4),
            "ms_per_step_fastest_rank": round(ms_fastest_rank / K, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "Correlation(pad=20,k=1,md=20,s1=1,s2=2) fwd+bwd on fp32 [8,256,112,256] per GPU "
                                   "(BASELINE configs[1])", "per_gpu_batch": B, "global_batch": B * world,
                       "l2": "inputs+outputs 1.75 GB per step >> 126 MB L2 (no flush needed)",
                       "parallelism": "replicas x%d (weak, no data-path collective)" % world, "impl": name,
                       "step": step_how},
            "frac_hbm_peak": round(value / world / peak, 4),
            "roofline": roofline,
            "kernels": {"forward_ms": round(per_f, 4), "backward_ms": round(per_b, 4),
                        "forward_GBps": round(fwd_b / per_f / 1e6, 1), "backward_GBps": round(bwd_b / per_b / 1e6, 1)},
            "e2e": {"value": round(e2e_value, 2), "unit": "GB/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": round(ms_e / K, 3), "steps": K,
                    "how": "flownet2_b200.hostpipe.HostPipeline: pinned host buffers, H2D / kernels / D2H of consecutive "
                           "steps on three streams, 2 device buffer sets", "max_abs_diff_vs_resident": e2e_check},
            "gpu_launches": int(launches_timed),
            "numa": numa_info,
            "clocks": clocks,
            "flownet2": flow,
        }
        if args.impl == "reference":
            line["impl"] = "reference"
            line["config"]["impl"] = "reference CUDA kernels rebuilt for sm_100a (oracle/_ref)"
        if world == 1:
            try:
                line["cpu_baseline"] = cpu_baseline_sample()
            except Exception as e:
                line["cpu_baseline"] = {"error": str(e)[:200]}
        if args.impl == "ours" and not args.no_extras and world == 1:
            try:
                line["ops"] = extras_ours(dev)
            except Exception as e:
                line["ops"] = {"error": str(e)[:300]}
        print(json.dumps(line))
    sampler.stop()
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
