#!/usr/bin/env python
"""bench.py - fake-quant fwd+bwd throughput on the ResNet-50 W4A4 QAT quantizer set.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one synthetic ImageNet-shaped batch: for each of the 54
quantised layers of torchvision ResNet-50 the activation fake-quant forward (A4 unsigned, per-tensor,
QBase form, dlmc/quantization/scalar/modules/base.py:96-102) and backward (dx + d in_scale), plus
the per-channel W4 weight fake-quant forward/backward of all 54 weight tensors (one grouped launch
each way).  Metric: algorithmic HBM GB/s = 20 B/element (fp32: read x, write y, read dy, read x,
write dx) * elements / time (SURVEY.md 8d, BASELINE.md 3).

  value        device-resident (inputs in HBM before the timed region), CUDA-graph replayed
  e2e          same workload through the host-buffer C-ABI entry (pinned host tensors in and out,
               H2D/D2H inside the timed region)
  roofline     the dominant kernel (fq_bwd_flat: 12 B/elem) timed live with CUDA events
  cpu_baseline the oracle port (the reference's eager torch chain) on the host cores, bounded sample

`--impl reference` times that CPU implementation alone (rank 0 only under torchrun).
"""
import argparse
import ctypes as C
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "fakequant_fwd_bwd_hbm_gbps"
UNIT = "GB/s"
BYTES_FWD, BYTES_BWD = 8, 12      # fp32, per element (SURVEY.md 8d)
A_BITS, W_BITS = 4, 4


# ------------------------------------------------------------------------------------------
def resnet50_layers():
    """(name, activation C,H,W per image, weight shape) of the 54 quantised layers of torchvision
    resnet50 at 224x224 (SURVEY.md App. B: 10 664 448 activation and 25 502 912 weight elements)."""
    layers = [("conv1", (3, 224, 224), (64, 3, 7, 7))]
    cin, hw = 64, 56
    for li, (planes, blocks, stride) in enumerate([(64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2)], 1):
        for b in range(blocks):
            s = stride if b == 0 else 1
            pre = f"layer{li}.{b}"
            layers.append((pre + ".conv1", (cin, hw, hw), (planes, cin, 1, 1)))
            layers.append((pre + ".conv2", (planes, hw, hw), (planes, planes, 3, 3)))
            layers.append((pre + ".conv3", (planes, hw // s, hw // s), (planes * 4, planes, 1, 1)))
            if b == 0:
                layers.append((pre + ".downsample.0", (cin, hw, hw), (planes * 4, cin, 1, 1)))
            cin, hw = planes * 4, hw // s
    layers.append(("fc", (2048,), (1000, 2048)))
    assert len(layers) == 54
    assert sum(math.prod(a) for _, a, _ in layers) == 10664448
    assert sum(math.prod(w) for _, _, w in layers) == 25502912
    return layers


def qrange(signed, bits):
    return (-(2 ** (bits - 1) - 1), 2 ** (bits - 1) - 1) if signed else (0, 2 ** bits - 1)


# ------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs (NVML)."""

    def __init__(self, device_index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.h = None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            try:
                uuid = torch.cuda.get_device_properties(device_index).uuid
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.h = None

    NAMES = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
             0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
             0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def run(self):
        if self.h is None:
            return
        while not self._halt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.NAMES.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def stop(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=1.0)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------
class Workload:
    """Device-resident tensors + prebuilt C-ABI argument lists + CUDA graphs for one rank."""

    def __init__(self, batch, device, seed):
        from dlmc_quant_b200 import _lib
        from dlmc_quant_b200 import functional as F
        self.lib, self.F, self.h = _lib, F, _lib.lib()
        self.device, self.batch = device, batch
        self.layers = resnet50_layers()
        gen = torch.Generator(device=device).manual_seed(seed)
        ilo, ihi = qrange(False, A_BITS)
        wlo, whi = qrange(True, W_BITS)
        self.acts, self.wts = [], []
        n_layers = len(self.layers)
        wch = sum(w[0] for _, _, w in self.layers)
        # every quantizer's scale gradient lands in ONE flat buffer: a single all-reduce per step
        self.dscale = torch.zeros(n_layers + wch, dtype=torch.float32, device=device)
        ch_off = n_layers
        for i, (name, ashape, wshape) in enumerate(self.layers):
            x = torch.randn((batch,) + ashape, generator=gen, device=device)
            if i > 0:
                x = torch.relu(x) * 2                 # post-ReLU-like, ~50 % zeros (SURVEY.md 8d)
            dy = torch.randn(x.shape, generator=gen, device=device)
            stats = F.obs_stats(x)
            scale, off = F.minmax_from_stats(stats, A_BITS, False)
            n = x.numel()
            lay = _lib.Layout(1, 1, n, _lib.F32)
            qp = _lib.QParams(_lib.FORM_AFFINE, ilo, ihi, 1 / math.sqrt(n * ihi), scale.data_ptr(), off.data_ptr())
            self.acts.append(dict(x=x, dy=dy, y=torch.empty_like(x), dx=torch.empty_like(x), scale=scale, off=off,
                                  lay=lay, qp=qp, n=n, ds=self.dscale[i:i + 1]))
            w = torch.randn(wshape, generator=gen, device=device) * 0.02
            dw = torch.randn(wshape, generator=gen, device=device)
            wstats = F.obs_stats(w, ch_axis=0)
            wscale, _ = F.minmax_from_stats(wstats, W_BITS, True)
            c, k = wshape[0], math.prod(wshape[1:])
            self.wts.append(dict(x=w, dy=dw, y=torch.empty_like(w), dx=torch.empty_like(w), scale=wscale, offset=None,
                                 dscale=self.dscale[ch_off:ch_off + c], channels=c, inner=k, form=_lib.FORM_AFFINE,
                                 lo=wlo, hi=whi, g=1 / math.sqrt(c * k * whi)))
            ch_off += c
        self.act_elems = sum(a["n"] for a in self.acts)
        self.wt_elems = sum(w["x"].numel() for w in self.wts)
        self.elems = self.act_elems + self.wt_elems
        self.ws = torch.zeros(self.h.dlmcq_workspace_bytes(None), dtype=torch.uint8, device=device)
        self.deferred = F.DeferredScaleGrads(device, len(self.acts))
        self.grp_f, self.grp_b = F.GroupedFakeQuant(device), F.GroupedFakeQuant(device)
        self.wf = [dict(w) for w in self.wts]
        self.wb = [dict(w, y=w["dx"]) for w in self.wts]
        self.launches_per_step = 2 * len(self.acts) + 1 + 1 + 2      # + finalize_many + grouped fwd/bwd/finalize

    # -- eager launches (also what gets captured) ------------------------------------------
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def fwd_acts(self):
        st, f = self._stream(), self.h.dlmcq_fq_forward
        for a in self.acts:
            self.lib.check(f(a["x"].data_ptr(), a["y"].data_ptr(), None, C.byref(a["lay"]), C.byref(a["qp"]), st))

    def bwd_acts(self):
        """54 backward launches leave their per-CTA partial sums behind; one batched launch reduces all 54
        scale gradients (dlmcq_fq_backward_partials + dlmcq_fq_finalize_many)."""
        st, f = self._stream(), self.h.dlmcq_fq_backward_partials
        for i, a in enumerate(self.acts):
            self.lib.check(f(a["x"].data_ptr(), a["dy"].data_ptr(), a["dx"].data_ptr(), C.byref(a["lay"]),
                             C.byref(a["qp"]), self.deferred.partials[i].data_ptr(), st))
        self.deferred.finalize([a["ds"] for a in self.acts])

    def weights(self):
        self.grp_f.forward(self.wf)
        self.grp_b.backward(self.wb)

    def capture(self):
        """Three CUDA graphs per step so that plain events between them can time the kernel groups."""
        self.fwd_acts(); self.bwd_acts(); self.weights()          # warm: tables, lazy module load
        torch.cuda.synchronize()
        self.g_fwd, self.g_bwd, self.g_wt = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.g_fwd):
            self.fwd_acts()
        with torch.cuda.graph(self.g_bwd):
            self.bwd_acts()
        with torch.cuda.graph(self.g_wt):
            self.weights()
        torch.cuda.synchronize()


def run_ours(args, rank, world, device):
    import torch.distributed as dist
    wl = Workload(args.batch, device, 2333 + rank)         # the reference's seed, per-rank offset
    wl.capture()

    pending = [None]

    def step(ev=None):
        wl.g_fwd.replay()
        if ev:
            ev[0].record()
        if pending[0] is not None:      # the previous step's all-reduce must be done before dscale is rewritten
            pending[0].wait()
        wl.g_bwd.replay()
        if ev:
            ev[1].record()
        wl.g_wt.replay()
        if world > 1 and not os.environ.get("DLMCQ_BENCH_NO_COLLECTIVE"):   # (diagnostic switch)
            # the path's one real exchange: scale gradients, one flat SUM all-reduce over NVLink,
            #             issued asynchronously so that it overlaps the next step's forward (as DDP overlaps backward)
            pending[0] = dist.all_reduce(wl.dscale, async_op=True)

    def fence():
        if pending[0] is not None:
            pending[0].wait()
            pending[0] = None
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # everything slow or rank-dependent (NVML init, event creation) happens BEFORE the fence, so that all
    # ranks enter the timed region together; otherwise early ranks just wait in the first all-reduce
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(device.index)
    for _ in range(args.warmup):
        step()
    fence()
    sampler.start()
    t0.record()
    for k in range(args.steps):
        step(evs[k])
    if pending[0] is not None:
        pending[0].wait()               # the last all-reduce is inside the timed region
    t1.record()
    fence()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(wl, args.dump_outputs)
    if os.environ.get("DLMCQ_BENCH_PER_RANK"):
        print(f"rank {rank}: {t0.elapsed_time(t1) / args.steps:.4f} ms/step", file=sys.stderr, flush=True)
    ms = torch.tensor([t0.elapsed_time(t1)], device=device)
    bwd_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in evs)], device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(bwd_ms, op=dist.ReduceOp.MAX)
    ms, bwd_ms = float(ms), float(bwd_ms)
    total_elems = wl.elems * world * args.steps
    value = total_elems * (BYTES_FWD + BYTES_BWD) / (ms * 1e-3) / 1e9

    # roofline of the dominant kernel: fq_bwd_flat<AFFINE,float>, 54 launches per step, 12 B/elem
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak, peak_kind = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")
    launches = len(wl.acts) * args.steps
    avg_launch_s = bwd_ms * 1e-3 / launches
    bytes_per_launch = BYTES_BWD * wl.act_elems / len(wl.acts)
    achieved = bytes_per_launch / avg_launch_s / 1e9
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = tj["fq_bwd_flat_dram_bytes_per_elem"] * wl.act_elems / len(wl.acts)
    except Exception:
        pass
    roofline = {"kernel": "fq_bwd_flat<AFFINE,f32>", "bound": "hbm", "achieved": round(achieved, 1), "peak": peak,
                "peak_kind": peak_kind, "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic,
                "bytes_per_launch": bytes_per_launch, "avg_launch_us": round(avg_launch_s * 1e6, 2),
                "frac_of_nominal_8TBps": round(achieved / 8000.0, 4)}

    e2e = run_e2e(args, wl, rank, world, device)
    launches_total = wl.launches_per_step * args.steps
    cfg_elems, cfg_act_elems, cfg_ds = wl.elems, wl.act_elems, wl.dscale.numel()
    del wl
    torch.cuda.empty_cache()
    qat = run_qat(args, rank, world, device)
    code_gemm = run_code_gemm(args, device) if (rank == 0 and world == 1) else None
    inference = run_inference(args, device) if (rank == 0 and world == 1) else None
    out = {"metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "resnet50_w4a4_qat_quantizers (54 layers: A4 per-tensor act + W4 per-channel weight, "
                                  "QBase form, fwd+bwd)", "per_gpu_batch": args.batch, "image": "3x224x224",
                      "elements_per_step_per_gpu": cfg_elems, "l2": "working set %.1f GB per GPU, far larger than the "
                      "126 MB L2; no flush needed" % (cfg_act_elems * 16 / 1e9), "cuda_graphs": True,
                      "collective": "all_reduce(SUM) of %d scale-grad floats per step" % cfg_ds if world > 1
                      else "none (1 GPU)"},
           "elements_per_s": round(total_elems / (ms * 1e-3), 1),
           "images_per_s_quantizer_path": round(args.batch * world * args.steps / (ms * 1e-3), 1),
           "gpu_launches": launches_total, "roofline": roofline, "clocks": clocks, "e2e": e2e,
           "qat_images_per_s": qat, "code_gemm": code_gemm,
           "inference_images_per_s": inference}
    if rank == 0:
        out["cpu_baseline"] = cpu_reference(sample_batch=1, passes=3) if world == 1 else None
        print(json.dumps(out), flush=True)


DUMP_SAMPLE = 1 << 16       # elements kept per array: 4 arrays x 54 layers x 64 Ki float32 stays under 64 MB


def dump_outputs(wl, out_dir):
    """What the timed path handed back in its last step, as float32 .npy files under out_dir: per layer the
    activation's and the weight's fake-quant forward (`<layer>.act_y`, `<layer>.wt_y`) and input gradient
    (`<layer>.act_dx`, `<layer>.wt_dx`), and `dscale`, the flat scale-gradient buffer (one entry per layer's
    activation, then the weights' per-channel entries in layer order).  An array longer than DUMP_SAMPLE is stored
    as DUMP_SAMPLE elements at sorted indices drawn from one fixed-seed generator in this fixed order, so two builds
    run with the same arguments are compared element for element.  Called on rank 0 only: with N > 1 ranks the y / dx
    arrays are rank 0's (inputs seeded 2333 + 0) and `dscale` holds the SUM over the N ranks, so a dump depends on N."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    gen = torch.Generator().manual_seed(2333)

    def save(name, t):
        flat = t.reshape(-1)
        if flat.numel() > DUMP_SAMPLE:
            idx = torch.randint(flat.numel(), (DUMP_SAMPLE,), generator=gen).sort().values
            flat = flat[idx.to(flat.device)]
        np.save(os.path.join(out_dir, name + ".npy"), flat.float().cpu().numpy())

    for (name, _, _), a, w in zip(wl.layers, wl.acts, wl.wts):
        save(name + ".act_y", a["y"])
        save(name + ".act_dx", a["dx"])
        save(name + ".wt_y", w["y"])
        save(name + ".wt_dx", w["dx"])
    np.save(os.path.join(out_dir, "dscale.npy"), wl.dscale.cpu().numpy())


def run_e2e(args, wl, rank, world, device):
    """Same workload through the host-buffer C-ABI calls (caller-owned dlmcq_host_ctx): pinned HOST x, dy in, results
    back in host memory, H2D / D2H inside the timed region.

    Headline (`value`): the compact LOSSLESS result format - packed 4-bit codes (y = code * s' + offset, bit-identical
    to the fp32 forward) and one keep bit per element (dx = keep ? dy : 0) - through dlmcq_host_ctx_fq_codes; inputs
    stay fp32, the arithmetic is the same fp32 arithmetic as `value` above.  `full_format` repeats the measurement with
    y and dx returned as fp32 tensors (dlmcq_host_ctx_fq_forward_backward, the round-1 format)."""
    import torch.distributed as dist
    if args.no_e2e:
        return None
    F, lib = wl.F, wl.lib
    steps = max(1, min(args.steps, args.e2e_steps))
    hq = F.HostFakeQuant(device, chunk_elems=1 << 22)
    # INPUTS: one pinned (x, dy) pair sized to the largest layer, read by all 54 layers - the bytes that cross PCIe per
    # step are exactly the workload's, while pinned memory stays at 2 x 411 MB per rank (8 ranks x 54 layers of fp32
    # inputs would not fit the box's RAM).  OUTPUTS: every layer owns its slice, so all results of a step are
    # consumable after the step.
    nmax = max(a["n"] for a in wl.acts)
    big = max(wl.acts, key=lambda a: a["n"])
    hx_all, hdy_all = big["x"].reshape(-1).cpu().pin_memory(), big["dy"].reshape(-1).cpu().pin_memory()
    codes_all = torch.empty(sum((a["n"] + 1) // 2 for a in wl.acts), dtype=torch.uint8).pin_memory()
    keep_all = torch.empty(sum((a["n"] + 7) // 8 for a in wl.acts), dtype=torch.uint8).pin_memory()
    host, c0, k0 = [], 0, 0
    for a in wl.acts:
        n = a["n"]
        host.append((hx_all[:n], hdy_all[:n], codes_all[c0:c0 + (n + 1) // 2], keep_all[k0:k0 + (n + 7) // 8],
                     float(a["scale"]), float(a["off"]), a["qp"].lo, a["qp"].hi, a["qp"].g))
        c0 += (n + 1) // 2
        k0 += (n + 7) // 8
    hw = [(w["x"].cpu().pin_memory(), w["dy"].cpu().pin_memory(), torch.empty_like(w["x"], device="cpu").pin_memory(),
           torch.empty_like(w["x"], device="cpu").pin_memory()) for w in wl.wts]
    hds = torch.empty(wl.dscale.numel(), dtype=torch.float32).pin_memory()
    hy_full = hdx_full = None

    def weights_roundtrip():
        for w, (hx, hdy, hy, hdx) in zip(wl.wts, hw):
            w["x"].copy_(hx, non_blocking=True)
            w["dy"].copy_(hdy, non_blocking=True)
        wl.weights()
        for w, (hx, hdy, hy, hdx) in zip(wl.wts, hw):
            hy.copy_(w["y"], non_blocking=True)
            hdx.copy_(w["dx"], non_blocking=True)
        hds[len(host):].copy_(wl.dscale[len(host):], non_blocking=True)

    def step_compact():
        for i, (hx, hdy, hc, hk, s, o, lo, hi, g) in enumerate(host):       # enqueue all layers, drain once
            hq.codes_async(hx, hdy, hc, hk, hds[i:i + 1], s, o, lo, hi, form=lib.FORM_AFFINE, g=g, pack4=True)
        weights_roundtrip()
        hq.synchronize()
        torch.cuda.synchronize()

    def step_full():
        for i, (hx, hdy, hc, hk, s, o, lo, hi, g) in enumerate(host):
            n = hx.numel()
            hq.forward_backward_async(hx, hdy, hy_full[:n], hdx_full[:n], hds[i:i + 1], s, o, lo, hi,
                                      form=lib.FORM_AFFINE, g=g)
        weights_roundtrip()
        hq.synchronize()
        torch.cuda.synchronize()

    def timed(step):
        step()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        if world > 1:
            dist.barrier()
        dt = torch.tensor([time.perf_counter() - t0], device=device)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return float(dt)

    dt = timed(step_compact)
    wbytes = 4 * wl.wt_elems
    h2d = 2 * 4 * wl.act_elems + 2 * wbytes
    d2h = codes_all.numel() + keep_all.numel() + 2 * wbytes + 4 * wl.dscale.numel()
    out = {"value": round(wl.elems * world * steps * (BYTES_FWD + BYTES_BWD) / dt / 1e9, 2), "unit": UNIT,
           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": steps, "ms_per_step": round(dt / steps * 1e3, 2),
           "result_format": "activations: packed 4-bit codes + 1 keep bit per element (lossless: y = code*s'+offset, "
                            "dx = keep ? dy : 0); weights: fp32 y, dx",
           "host_buffers": "pinned; inputs: one (x, dy) pair sized to the largest layer, read by all layers; outputs: "
                           "every layer has its own slice (all results of a step are consumable)",
           "api": "dlmcq_host_ctx_fq_codes per layer on a caller-owned dlmcq_host_ctx + one dlmcq_host_ctx_synchronize "
                  "(activations); H2D / grouped launch / D2H (weights)"}
    try:
        hy_full, hdx_full = torch.empty(nmax).pin_memory(), torch.empty(nmax).pin_memory()
        dtf = timed(step_full)
        out["full_format"] = {"value": round(wl.elems * world * steps * (BYTES_FWD + BYTES_BWD) / dtf / 1e9, 2),
                              "ms_per_step": round(dtf / steps * 1e3, 2), "h2d_bytes_per_step": h2d,
                              "d2h_bytes_per_step": 2 * 4 * wl.act_elems + 2 * wbytes + 4 * wl.dscale.numel(),
                              "result_format": "fp32 y and dx (outputs share one buffer pair: not consumable per layer)",
                              "api": "dlmcq_host_ctx_fq_forward_backward"}
    except Exception as e:
        out["full_format"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    hq.close()
    return out


# ------------------------------------------------------------------------------------------
# second half of BASELINE.json's metric: end-to-end ResNet-50 W4A4 QAT images/s
# ------------------------------------------------------------------------------------------
QAT_CFG = {"weight": {"enable": True, "type": "minmax_channel", "args": {"n_bits": W_BITS, "signed": True, "ch_axis": 0}},
           "input": {"enable": True, "type": "minmax_tensor", "args": {"n_bits": A_BITS, "signed": False}},
           "exclude_layers": [], "override_options": [], "momentum": 0.1}


def _eager_reference_modules(model):
    """The `eager` arm: every Conv2d / Linear wrapped so that its input and weight go through the reference's own
    eager op chain on the SAME GPU - a restatement, for timing only, of dlmc/quantization/scalar/modules/base.py:
    82-102,106-133 with utils.py:24-32 (grad_scale, round_pass) and the min/max observers of ops.py:20-34,121-140,
    including the reference's per-forward `if self.in_init_state == 0` device-to-host checks (base.py:82,107).
    Per-channel wt_scale is pre-shaped [C,1,1,1] (the only way the reference runs per-channel, SURVEY.md a6)."""
    import torch.nn as nn
    import torch.nn.functional as TF

    def grad_scale(x, scale):                  # utils.py:24-27
        y_grad = x * scale
        return (x - y_grad).detach() + y_grad

    def round_pass(x):                         # utils.py:29-32
        return (x.round() - x).detach() + x

    class EagerQ(nn.Module):
        def __init__(self, base):
            super().__init__()
            self.base = base
            dev = base.weight.device
            self.in_scale = nn.Parameter(torch.ones(1, device=dev))
            self.wt_scale = nn.Parameter(torch.ones([base.weight.shape[0]] + [1] * (base.weight.dim() - 1), device=dev))
            self.register_buffer("in_init_state", torch.zeros(1, device=dev))
            self.register_buffer("wt_init_state", torch.zeros(1, device=dev))
            self.in_max, self.wt_max = 2 ** A_BITS - 1, 2 ** (W_BITS - 1) - 1

        def forward(self, x):
            w = self.base.weight
            if self.in_init_state == 0:                                             # base.py:82 (D2H sync)
                mn, mx = x.detach().min(), x.detach().max()                         # ops.py:26-33
                self.in_scale.data.copy_((mx - mn) / self.in_max)
                self.in_offset = mn
                self.in_init_state.fill_(1)
            g_i = 1 / math.sqrt(x.numel() * self.in_max)                            # base.py:96
            s = grad_scale(self.in_scale, g_i)
            x = round_pass(((x - self.in_offset) / s).clamp(0, self.in_max)) * s + self.in_offset   # base.py:102
            if self.wt_init_state == 0:                                             # base.py:107 (D2H sync)
                absmax = w.detach().reshape(w.shape[0], -1).abs().max(dim=1)[0]     # ops.py:121-127
                self.wt_scale.data.copy_((absmax / self.wt_max).reshape(self.wt_scale.shape))
                self.wt_offset = torch.zeros_like(self.wt_scale)
                self.wt_init_state.fill_(1)
            g_w = 1 / math.sqrt(w.numel() * self.wt_max)                            # base.py:131
            ws = grad_scale(self.wt_scale, g_w)
            wq = round_pass(((w - self.wt_offset) / ws).clamp(-self.wt_max, self.wt_max)) * ws + self.wt_offset
            b = self.base
            if isinstance(b, nn.Conv2d):
                return TF.conv2d(x, wq, b.bias, b.stride, b.padding, b.dilation, b.groups)
            return TF.linear(x, wq, b.bias)

    for _, m in list(model.named_modules()):
        for cname, c in list(m.named_children()):
            if isinstance(c, (nn.Conv2d, nn.Linear)):
                setattr(m, cname, EagerQ(c))
    return model


def _qat_arm(arm, channels_last, batch, steps, rank, world, device, graphed=False):
    """One arm of the QAT benchmark, with the reference harness's methodology (example/benchmark/benchmark.py:168-197:
    SGD nesterov lr 0.01 wd 5e-4 momentum 0.9, cross-entropy, 2 warm-up steps, wall clock over the remaining steps,
    images = batch * n_gpu per step; benchmark.yaml:14 cudnn.benchmark on; DDP for N > 1)."""
    import copy
    import torch.distributed as dist
    import torch.nn as nn
    import torchvision
    torch.manual_seed(2333)
    model = torchvision.models.resnet50().to(device)
    if arm in ("ours", "ours_fused"):
        from dlmc_quant_b200 import quantize_model
        quantize_model(model, copy.deepcopy(QAT_CFG), None)
    elif arm == "eager":
        _eager_reference_modules(model)
    x = torch.randn(batch, 3, 224, 224, device=device)
    if channels_last:
        model = model.to(memory_format=torch.channels_last)
        x = x.contiguous(memory_format=torch.channels_last)
    t = torch.randint(0, 1000, (batch,), device=device)
    model.train()
    with torch.no_grad():
        model(x[:8])                    # lazy observer init (all arms: same warm state) before DDP / the optimizer
    fused_sites = None
    if arm in ("ours", "ours_fused"):
        from dlmc_quant_b200.quantize import group_weight_quantizers
        group_weight_quantizers(model)  # all 54 weight tensors: one launch per direction
    if arm == "ours_fused":
        from dlmc_quant_b200.fuse import fuse_bn_act_quant
        h = fuse_bn_act_quant(model)
        fused_sites = {"blocks": h.blocks, "sequentials": h.sequentials, "batchnorms": h.batchnorms}
    crit = nn.CrossEntropyLoss()
    if world > 1:
        if graphed:                     # DDP built on a side stream so that its all-reduces can be captured (graph.py)
            from dlmc_quant_b200.graph import wrap_ddp
            model = wrap_ddp(model, device_ids=[device.index])
        else:
            model = nn.parallel.DistributedDataParallel(model, device_ids=[device.index])
    opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9, nesterov=True, weight_decay=5e-4)

    def step():
        opt.zero_grad()
        loss = crit(model(x), t)
        loss.backward()
        opt.step()
        return loss

    if graphed:                         # whole step (forward, backward, gradient all-reduce, optimizer): one CUDA graph
        from dlmc_quant_b200.graph import graph_train_step
        gstep = graph_train_step(model, opt, crit, x, t)
        step = lambda: gstep(x, t)      # noqa: E731  (the per-step input copy into the static buffers is included)
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(device.index)
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(steps):
        loss = step()
    lv = float(loss.detach())
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    dt = torch.tensor([time.perf_counter() - t0], device=device, dtype=torch.float64)
    clocks = sampler.stop()
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    dt = float(dt)
    out = {"images_per_s": round(batch * world * steps / dt, 1), "ms_per_step": round(dt / steps * 1e3, 2),
           "loss_finite": math.isfinite(lv), "sm_mhz": clocks["sm_mhz"], "reasons": clocks["reasons"]}
    if fused_sites:
        out["fused_sites"] = fused_sites
    del model, opt
    torch.cuda.empty_cache()
    return out


# torchvision ResNet-50's stride-1 1x1 convolutions: (H = W, Cin, Cout, how many layers have this shape)
R50_POINTWISE = [(56, 64, 64, 1), (56, 64, 256, 4), (56, 256, 64, 2), (56, 256, 128, 1), (28, 128, 512, 4),
                 (28, 512, 128, 3), (28, 512, 256, 1), (14, 256, 1024, 6), (14, 1024, 256, 5), (14, 1024, 512, 1),
                 (7, 512, 2048, 3), (7, 2048, 512, 2)]


def _event_us(fn, iters=20, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters * 1e3


def run_code_gemm(args, device):
    """Consumer side of row f2 (dlmc_quant_b200.qgemm, csrc/qgemm_kernels.cu): the 1x1 convolutions of ResNet-50 as
    integer-code GEMMs on the tcgen05 tensor cores (W4A4 codes, one byte each, channels-last) beside the reference's
    path for the same layers - cuDNN convolution of the fake-quantised fp32 tensor (TF32, torch's default).
    Per shape: CUDA-event time of 20 calls after 5 warm-ups; totals weight each shape by its layer count."""
    if args.no_qat:
        return None
    from dlmc_quant_b200 import qgemm as Q
    res = {"workload": "torchvision resnet50 stride-1 1x1 convolutions, batch %d, channels_last, W4A4 codes" % args.batch,
           "kernel": "TMA -> tcgen05.mma kind::f8f6f4 on e4m3-encoded codes (bit-identical to kind::i8) -> TMEM -> "
                     "alpha[n]*acc + beta[n] epilogue", "shapes": [], "timing": "CUDA events, 20 calls after 5 warm-ups"}
    tot = {"ours_f32_us": 0.0, "ours_bf16_us": 0.0, "cudnn_tf32_us": 0.0, "ours_bytes_f32": 0, "cudnn_bytes": 0}
    worst = 0.0
    try:
        for hw, cin, cout, count in R50_POINTWISE:
            m, k, n = args.batch * hw * hw, cin, cout
            g = torch.Generator(device="cuda").manual_seed(hw * 1000 + cin)
            ca = torch.randint(0, 16, (m, k), device=device, generator=g, dtype=torch.uint8)
            cw = torch.randint(-7, 8, (n, k), device=device, generator=g, dtype=torch.int8)
            a_b = ca.float().to(torch.float8_e4m3fn).view(torch.uint8)
            w_b = cw.float().to(torch.float8_e4m3fn).view(torch.uint8)
            s_a, s_w = 0.11, torch.rand(n, device=device, generator=g) * 0.01 + 0.002
            alpha, beta = (s_a * s_w).float(), torch.zeros(n, device=device)
            o32 = torch.empty(m, n, device=device)
            o16 = torch.empty(m, n, device=device, dtype=torch.bfloat16)
            x = (ca.float() * s_a).view(args.batch, hw, hw, k).permute(0, 3, 1, 2)     # NCHW view, channels-last storage
            w = (cw.float() * s_w[:, None]).view(n, k, 1, 1).contiguous(memory_format=torch.channels_last)
            t32 = _event_us(lambda: Q.qgemm(a_b, w_b, alpha, beta, encoding=Q.QGEMM_E4M3, out=o32))
            t16 = _event_us(lambda: Q.qgemm(a_b, w_b, alpha, beta, encoding=Q.QGEMM_E4M3, out=o16,
                                            out_dtype=torch.bfloat16))
            torch.backends.cudnn.allow_tf32 = True
            tc = _event_us(lambda: torch.nn.functional.conv2d(x, w))
            torch.backends.cudnn.allow_tf32 = False
            ref = torch.nn.functional.conv2d(x, w).permute(0, 2, 3, 1).reshape(m, n)
            torch.backends.cudnn.allow_tf32 = True
            err = float(((o32 - ref).abs() / ((15 * s_a) * (7 * s_w) * k)).max())
            worst = max(worst, err)
            by = m * k + n * k + m * n * 4
            res["shapes"].append({"m": m, "k": k, "n": n, "layers": count, "ours_f32_us": round(t32, 2),
                                  "ours_bf16_us": round(t16, 2), "cudnn_tf32_us": round(tc, 2),
                                  "ours_f32_gbs": round(by / t32 * 1e-3, 1)})
            tot["ours_f32_us"] += count * t32
            tot["ours_bf16_us"] += count * t16
            tot["cudnn_tf32_us"] += count * tc
            tot["ours_bytes_f32"] += count * by
            tot["cudnn_bytes"] += count * (m * k * 4 + n * k * 4 + m * n * 4)
            del ca, cw, a_b, w_b, o32, o16, x, w, ref
            torch.cuda.empty_cache()
        res["total"] = {k_: (round(v, 1) if isinstance(v, float) else v) for k_, v in tot.items()}
        res["speedup_vs_cudnn_tf32"] = {"f32_out": round(tot["cudnn_tf32_us"] / tot["ours_f32_us"], 3),
                                        "bf16_out": round(tot["cudnn_tf32_us"] / tot["ours_bf16_us"], 3)}
        res["max_err_vs_strict_fp32_cudnn_over_sum_abs_bound"] = worst
        res["parity_ok"] = worst <= 1e-5
    except Exception as e:                              # must not take the headline metric down
        res["error"] = f"{type(e).__name__}: {e}"[:300]
    return res


def run_inference(args, device):
    """ResNet-50 W4A4 inference (eval, no autograd, channels_last, synthetic batch) through the public module API:
    un-quantised, quantize_model (fake-quant kernels + cuDNN on fp32), and the same model after
    qgemm.enable_code_gemm (every stride-1 1x1 convolution and the classifier as an integer-code GEMM)."""
    if args.no_qat:
        return None
    import copy
    import torchvision
    res = {"model": "torchvision resnet50 W4A4 (QBase, minmax observers), eval / no_grad, channels_last, batch %d, fp32 "
                    "tensors (cuDNN TF32 convolutions: torch default)" % args.qat_batch,
           "timing": "CUDA events, %d forwards after 3 warm-ups" % args.qat_steps}
    try:
        x = torch.randn(args.qat_batch, 3, 224, 224, device=device).contiguous(memory_format=torch.channels_last)
        outs = {}
        for arm in ("fp32", "ours", "ours_code_gemm"):
            torch.manual_seed(2333)
            model = torchvision.models.resnet50().to(device).to(memory_format=torch.channels_last)
            if arm != "fp32":
                from dlmc_quant_b200 import quantize_model
                quantize_model(model, copy.deepcopy(QAT_CFG), None)
            model.eval()
            switched = None
            with torch.no_grad():
                model(x[:8])                                 # lazy observer initialisation
                if arm == "ours_code_gemm":
                    from dlmc_quant_b200.qgemm import enable_code_gemm
                    switched = len(enable_code_gemm(model))
                for _ in range(3):
                    y = model(x)
                torch.cuda.synchronize()
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                for _ in range(args.qat_steps):
                    y = model(x)
                t1.record()
                torch.cuda.synchronize()
            ms = t0.elapsed_time(t1) / args.qat_steps
            outs[arm] = y.float()
            if arm != "fp32":                                # the same model with strict-fp32 library convolutions
                torch.backends.cudnn.allow_tf32 = False      # (ours_code_gemm: its 3x3 / strided layers)
                torch.backends.cuda.matmul.allow_tf32 = False
                with torch.no_grad():
                    outs[arm + "_strict_fp32"] = model(x).float()
                torch.backends.cudnn.allow_tf32 = True
            res[arm] = {"images_per_s": round(args.qat_batch / ms * 1e3, 1), "ms_per_forward": round(ms, 3)}
            if switched is not None:
                res[arm]["layers_on_code_gemm"] = switched
                used = sum(1 for m_ in model.modules() if getattr(m_.__dict__.get("_code_gemm"), "usable", False))
                res[arm]["layers_that_used_it"] = used
            del model
            torch.cuda.empty_cache()
        # 4-bit activations: a relative error of 1e-3 in a convolution (TF32) flips codes downstream, each flip is 1/15
        # of a layer's range, and an untrained 50-layer network amplifies that - so the yardstick is the model with
        # strict-fp32 library convolutions, and how far the TF32 default itself is from it.  Layer-by-layer parity of
        # the code path (same inputs, 2e-5) is a GPU test: tests/qgemm_cases.py::case_resnet_layers.
        ref = outs["ours_strict_fp32"]
        rel = lambda a: float((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30))  # noqa: E731
        top = lambda a: float((a.argmax(1) == ref.argmax(1)).float().mean())             # noqa: E731
        res["vs_strict_fp32_library_path"] = {
            "logits_max_diff_rel": {"code_gemm_with_strict_fp32_3x3_layers": rel(outs["ours_code_gemm_strict_fp32"]),
                                    "code_gemm_with_tf32_3x3_layers": rel(outs["ours_code_gemm"]),
                                    "library_path_with_tf32": rel(outs["ours"])},
            "top1_agreement": {"code_gemm_with_strict_fp32_3x3_layers": top(outs["ours_code_gemm_strict_fp32"]),
                               "code_gemm_with_tf32_3x3_layers": top(outs["ours_code_gemm"]),
                               "library_path_with_tf32": top(outs["ours"])}}
    except Exception as e:                              # must not take the headline metric down
        res["error"] = f"{type(e).__name__}: {e}"[:300]
        torch.cuda.empty_cache()
    return res


def run_qat(args, rank, world, device):
    """ResNet-50 W4A4 QAT images/s for four arms on the same GPU(s): un-quantised, the reference's eager quantizer
    chain, this package (fused quantizer kernels), this package with the quantizers fused into their producers."""
    if args.no_qat:
        return None
    torch.backends.cudnn.benchmark = True
    res = {"model": "torchvision resnet50, W4 per-channel (minmax_channel) / A4 per-tensor (minmax_tensor) QBase QAT, "
                    "fp32 tensors (cuDNN TF32 convolutions: torch default)",
           "methodology": "example/benchmark/benchmark.py:168-197 (SGD nesterov, 2 warm-up steps, wall clock, "
                          "images = batch * n_gpu * steps / s), synthetic 3x224x224",
           "per_gpu_batch": args.qat_batch, "n_gpus": world, "steps": args.qat_steps,
           "parallelism": "DistributedDataParallel (bucketed ncclAllReduce of 25.6 M weight gradients + scale "
                          "gradients per step)" if world > 1 else "single GPU",
           "arms": {"fp32": "un-quantised model", "eager": "reference eager op chain + autograd on this GPU",
                    "ours": "dlmc_quant_b200.quantize_model + group_weight_quantizers",
                    "ours_fused": "ours + fuse_bn_act_quant (BatchNorm+ReLU+next layer's input fake-quant in one "
                                  "kernel per direction; channels_last only)",
                    "*_graphed": "the same step (forward, backward, gradient all-reduce, optimizer) captured once as a "
                                 "CUDA graph and replayed: the eager DDP step is host-bound"}}
    only = set(args.qat_arms.split(",")) if args.qat_arms else None
    for fmt, cl, arms in (("nchw", False, ("fp32", "eager", "ours")),
                          ("channels_last", True, ("fp32", "eager", "ours", "ours_fused", "fp32_graphed",
                                                   "ours_fused_graphed"))):
        if only and fmt not in only and not (only & set(arms)):
            continue
        res[fmt] = {}
        for arm in arms:
            if only and arm not in only and fmt not in only:
                continue
            try:
                res[fmt][arm] = _qat_arm(arm.replace("_graphed", ""), cl, args.qat_batch, args.qat_steps, rank, world,
                                         device, graphed=arm.endswith("_graphed"))
            except Exception as e:                      # an arm that fails must not take the headline metric down
                res[fmt][arm] = {"error": f"{type(e).__name__}: {e}"[:300]}
                torch.cuda.empty_cache()
    # small per-GPU batch: the step is host-bound for the module path (~40 us of Python + ctypes per quantizer call);
    # the same step captured once and replayed as ONE CUDA graph (dlmc_quant_b200.graph) removes the host from it
    if world == 1 and (not only or "small_batch" in only):
        sb = res["channels_last_small_batch"] = {"per_gpu_batch": args.qat_small_batch}
        for arm, graphed in (("fp32", False), ("fp32", True), ("ours_fused", False), ("ours_fused", True)):
            key = arm + ("_graphed" if graphed else "")
            try:
                sb[key] = _qat_arm(arm, True, args.qat_small_batch, 2 * args.qat_steps, rank, world, device, graphed)
            except Exception as e:
                sb[key] = {"error": f"{type(e).__name__}: {e}"[:300]}
                torch.cuda.empty_cache()
    return res

# ------------------------------------------------------------------------------------------
def cpu_reference(sample_batch=1, passes=3):
    """The oracle port (= the reference's eager PyTorch chain, restated op for op) on the host
    cores: every layer's activation + per-channel weight fake-quant fwd+bwd at `sample_batch`."""
    from oracle import restate as R
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    gen = torch.Generator().manual_seed(2333)
    ilo, ihi = qrange(False, A_BITS)
    wlo, whi = qrange(True, W_BITS)
    data, elems = [], 0
    for i, (name, ashape, wshape) in enumerate(resnet50_layers()):
        x = torch.randn((sample_batch,) + ashape, generator=gen)
        if i > 0:
            x = torch.relu(x) * 2
        dy = torch.randn(x.shape, generator=gen)
        s, o = R.obs_minmax_tensor(x, A_BITS, False)
        w = torch.randn(wshape, generator=gen) * 0.02
        dw = torch.randn(wshape, generator=gen)
        ws, wo = R.obs_minmax_channel(w, W_BITS, True, ch_axis=0)
        data.append((x, dy, s.reshape(1), o.reshape(1), w, dw, ws, wo))
        elems += x.numel() + w.numel()
    best = float("inf")
    for _ in range(passes):
        t0 = time.perf_counter()
        for x, dy, s, o, w, dw, ws, wo in data:
            R.fq_affine_fwd_bwd(x, s, o, ilo, ihi, R.lsq_g(x.numel(), ihi), dy)
            R.fq_affine_fwd_bwd(w, ws, wo, wlo, whi, R.lsq_g(w.numel(), whi), dw)
        best = min(best, time.perf_counter() - t0)
    return {"value": round(elems * (BYTES_FWD + BYTES_BWD) / best / 1e9, 3), "unit": UNIT, "cores": cores,
            "threads": torch.get_num_threads(), "kind": "port",
            "sample": f"all 54 layers (act + per-channel weight) at batch {sample_batch}: {elems} elements, "
                      f"best of {passes} passes, torch {torch.__version__} CPU eager + autograd",
            "elements_per_s": round(elems / best, 1), "seconds_per_pass": round(best, 3)}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the reference
    itself is pure Python and /root/reference does not exist on the GPU box)."""
    if rank != 0:
        return
    from oracle import restate as R
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    gen = torch.Generator().manual_seed(2333)
    ilo, ihi = qrange(False, A_BITS)
    wlo, whi = qrange(True, W_BITS)
    sb = args.ref_batch
    data, elems = [], 0
    for i, (name, ashape, wshape) in enumerate(resnet50_layers()):
        x = torch.randn((sb,) + ashape, generator=gen)
        if i > 0:
            x = torch.relu(x) * 2
        s, o = R.obs_minmax_tensor(x, A_BITS, False)
        w = torch.randn(wshape, generator=gen) * 0.02
        ws, wo = R.obs_minmax_channel(w, W_BITS, True, ch_axis=0)
        data.append((x, torch.randn(x.shape, generator=gen), s.reshape(1), o.reshape(1), w,
                     torch.randn(wshape, generator=gen), ws, wo))
        elems += x.numel() + w.numel()

    def step():
        for x, dy, s, o, w, dw, ws, wo in data:
            R.fq_affine_fwd_bwd(x, s, o, ilo, ihi, R.lsq_g(x.numel(), ihi), dy)
            R.fq_affine_fwd_bwd(w, ws, wo, wlo, whi, R.lsq_g(w.numel(), whi), dw)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = round(elems * args.steps * (BYTES_FWD + BYTES_BWD) / dt / 1e9, 3)
    sample = (f"each step = all 54 layers (act + per-channel weight) at batch {sb} ({elems} elements), "
              f"{cores} host threads, torch {torch.__version__} CPU eager + autograd")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "resnet50_w4a4_qat_quantizers (54 layers: A4 per-tensor act + W4 per-channel weight, "
                               "QBase form, fwd+bwd)", "per_gpu_batch": args.batch, "image": "3x224x224",
                   "sample_batch_per_step": sb},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=128,
                    help="per-GPU batch of 3x224x224 images (the reference harness runs 256 on 2 GPUs: benchmark.yaml:8,38)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--ref-batch", type=int, default=1)
    ap.add_argument("--no-qat", action="store_true", help="skip the ResNet-50 QAT images/s arms")
    ap.add_argument("--qat-steps", type=int, default=10)
    ap.add_argument("--qat-arms", default="", help="comma list restricting the QAT arms / formats (diagnostic), e.g. "
                                                   "'channels_last' or 'fp32,ours_fused'")
    ap.add_argument("--qat-only", action="store_true", help="skip the kernel metric; print only the QAT arms (diagnostic)")
    ap.add_argument("--qat-batch", type=int, default=128, help="per-GPU batch of the QAT arms")
    ap.add_argument("--qat-small-batch", type=int, default=32, help="per-GPU batch of the host-bound / CUDA-graph arms")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's outputs to DIR/<name>.npy (float32, sampled "
                         "to at most 64 MB in all) for comparing two builds on identical seeded inputs; under torchrun "
                         "only rank 0 writes (its own y/dx, and the scale gradients summed over ranks), so compare "
                         "dumps taken with the same number of GPUs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.qat_only):
        ap.error("--dump-outputs writes the outputs of the timed kernel path: it needs --impl ours without --qat-only")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - this path has no CPU fallback (use --impl reference for the CPU arm)")
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")      # NCCL work inside CUDA graphs (graphed arms)
        dist.init_process_group("nccl", device_id=device)
    try:
        if args.qat_only:
            q = run_qat(args, rank, world, device)
            if rank == 0:
                print(json.dumps({"qat_images_per_s": q}), flush=True)
        else:
            run_ours(args, rank, world, device)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
