#!/usr/bin/env python
"""bench.py -- SpectralConv fwd+bwd samples/sec at (B,C,H,W)=(32,64,128,128), modes=(32,32)  (BASELINE.json).

    python bench.py --gpus 1 --steps 50 --warmup 10              # our sm_100a path, one JSON line
    python bench.py --impl reference --steps 5 --warmup 1        # the reference's CPU path (oracle port)
    python bench.py --steps 50 --dump-outputs DIR                 # ... and write the last timed step's outputs as DIR/<name>.npy
    torchrun --nproc-per-node N ... bench.py --gpus N ...        # batch-sharded, one NCCL gradient all-reduce/step

One "step" = y = conv(x); y.backward(g) producing dx, dweight, dbias for one batch of synthetic input
(weak scaling: every rank owns a full batch of 32).  `value` is measured with inputs resident in HBM;
`e2e` is the same step through the nn.Module with pinned HOST buffers, copies inside the timed region.
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

METRIC = "SpectralConv fwd+bwd samples/sec at (B,C,H,W)=(32,64,128,128) modes=(32,32)"
UNIT = "samples/s"
B, C, H, W = 32, 64, 128, 128
MODES = (32, 32)
WORKLOAD = "FNO2d Darcy dense SpectralConv fwd+bwd, (B,C,H,W)=(32,64,128,128) per GPU, n_modes=(32,32) [BASELINE configs[1]]"


def algorithmic_bytes_step(b=B, ci=C, co=C, grid=(H, W), kept=(32, 17)):
    """SURVEY.md section 8(d): 16*B*C*S + 24*Ci*Co*M + 16*B*C*M bytes per fwd+bwd step."""
    s = 1
    for g in grid:
        s *= g
    m = 1
    for k in kept:
        m *= k
    return 16 * b * ci * s + 24 * ci * co * m + 16 * b * ci * m


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(plan):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the fused analysis kernel, from the committed ncu launch
    list of this round's build (profiles/r02_launches.csv, `--cache-control none`, summarised in r02_launches_summary.json);
    None when that file or kernel is absent, or when csrc/sc_fast.cu / sc_umma.cuh no longer hash to what the capture was taken
    from (`_source_sha1` in the summary).  A citation of a committed capture, not a measurement of this run."""
    if not plan.uses_fast_path() & 1:
        return None
    path = os.path.join(ROOT, "profiles", "r02_launches_summary.json")
    try:
        with open(path) as f:
            d = json.load(f)
        # staleness guard: the capture is only cited while the kernel sources it was taken from are unchanged
        import hashlib
        for fname, sha in d.get("_source_sha1", {}).items():
            with open(os.path.join(ROOT, "neuraloperator_b200", "csrc", fname), "rb") as src:
                if hashlib.sha1(src.read()).hexdigest() != sha:
                    return None
        k = d.get("k_fused_analysis2") or d["k_fused_analysis"]
        return (k["dram_read_mb"] + k["dram_write_mb"]) * 1e6
    except Exception:
        return None


def torch_cufft_forward(x, w, bias, n_modes_stored):
    """The reference's op sequence for real data and default flags (neuralop/layers/spectral_convolution.py:429-568) on
    whatever device `x` lives on: on the GPU this is PyTorch eager + cuFFT + cuBLAS, the denominator of north_star's
    ">= 1.5x the reference's own PyTorch+cuFFT" target.  Restated here (not imported from oracle/): it is a timed baseline."""
    import torch
    d = x.ndim - 2
    dims = list(range(-d, 0))
    grid = list(x.shape[2:])
    xf = torch.fft.rfftn(x, norm="forward", dim=dims)                                     # :443
    if d > 1:
        xf = torch.fft.fftshift(xf, dim=dims[:-1])                                        # :448-449
    sizes = list(xf.shape[2:])
    sl = [slice(None), slice(None)]
    for j, (size, k) in enumerate(zip(sizes, n_modes_stored)):                            # :500-519 (n_modes == max_n_modes)
        k = min(size, k)
        if j == d - 1:
            sl.append(slice(None, k))
        else:
            c = size // 2
            sl.append(slice(c - k // 2, c + k // 2 + k % 2))
    sl = tuple(sl)
    out_fft = torch.zeros([x.shape[0], w.shape[1], *sizes], device=x.device, dtype=torch.cfloat)    # :459-462
    out_fft[sl] = torch.einsum("bi...,io...->bo...", xf[sl], w)                           # :520-522, _contract_dense :21-46
    if d > 1:
        out_fft = torch.fft.ifftshift(out_fft, dim=dims[:-1])                             # :531-532
        out_fft = torch.fft.ifftn(out_fft, s=grid[:-1], dim=dims[:-1], norm="forward")    # :548
    out_fft[..., 0].imag.zero_()                                                          # :552
    if grid[-1] % 2 == 0:
        out_fft[..., -1].imag.zero_()                                                     # :555-556
    y = torch.fft.irfft(out_fft, n=grid[-1], dim=dims[-1], norm="forward")                # :559
    return y + bias                                                                       # :567-568


def time_cuda(fn, warm, reps):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def time_cuda_rot(fn, warm, reps):
    import torch
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


# BASELINE.json configs other than the headline one: (name, batch, channels, grid, n_modes, kind)
OTHER_CONFIGS = [
    ("1 FNO1d Burgers", 16, 32, (1024,), (16,), "dense"),
    ("3 TFNO2d Darcy Tucker(36,36,18,10) factorized", 32, 64, (128, 128), (32, 32), "tucker"),
    ("4 FNO3d Navier-Stokes", 8, 32, (64, 64, 64), (16, 16, 16), "dense"),
    ("5a FNO2d 256^2", 16, 64, (256, 256), (64, 64), "dense"),
    ("5b FNO2d 512^2", 16, 64, (512, 512), (64, 64), "dense"),
    ("5c FNO2d 1024^2", 16, 64, (1024, 1024), (64, 64), "dense"),
]


def measure_config(nb, dev, peak, batch, ch, grid, modes, kind, with_torch=True):
    """One BASELINE config on one GPU: eager fwd+bwd through the nn.Module (ours) and the reference op sequence on
    PyTorch+cuFFT, same tensors, CUDA events.  Returns samples/s, roofline fraction of the step, and the ratio."""
    import torch
    torch.manual_seed(0)
    tucker_ranks = [36, 36, 18, 10]
    if kind == "tucker":
        conv = nb.SpectralConv(ch, ch, modes, factorization="tucker", rank=tucker_ranks, implementation="factorized").to(dev)
    else:
        conv = nb.SpectralConv(ch, ch, modes).to(dev)
    x = torch.randn(batch, ch, *grid, device=dev)
    g = torch.randn(batch, ch, *grid, device=dev)

    def ours():
        xx = x.detach().requires_grad_(True)
        for prm in conv.parameters():
            prm.grad = None
        conv(xx).backward(g)

    big = x.numel() * 4 > (1 << 30)
    reps = 5 if big else 20
    t_ours = time_cuda(ours, 3, reps)
    kept = nb.get_plan(dev, grid, grid, conv.n_modes, conv.max_n_modes).kept
    S = 1
    for n in grid:
        S *= n
    M = 1
    for k in kept:
        M *= k
    w_elems = sum(prm.numel() for prm in conv.weight.decomposition()) if kind == "tucker" else ch * ch * M
    step_bytes = 16 * batch * ch * S + 24 * w_elems + 16 * batch * ch * M          # SURVEY.md section 8(d)
    out = {"shape": [batch, ch, *grid], "n_modes": list(modes), "ms_per_step": t_ours, "samples_per_s": batch / t_ours * 1e3,
           "step_bytes": step_bytes, "roofline_frac": step_bytes / (t_ours * 1e-3) / 1e9 / peak, "timing": f"eager nn.Module, {reps} steps"}
    if with_torch:
        w = conv.weight.to_tensor().detach().clone().requires_grad_(True)       # Tucker: the eager reference reconstructs (see DESIGN.md)
        b = conv.bias.detach().clone().requires_grad_(True)

        def ref():
            xx = x.detach().requires_grad_(True)
            w.grad = None
            b.grad = None
            torch_cufft_forward(xx, w, b, conv.n_modes).backward(g)

        t_ref = time_cuda(ref, 2, max(3, reps // 2))
        out["torch_cufft_ms_per_step"] = t_ref
        out["speedup_vs_torch_cufft"] = t_ref / t_ours
    del conv, x, g
    torch.cuda.empty_cache()
    return out


def torch_layer_forward(x, prm, n_modes_stored, last=False):
    """One Fourier layer of the reference (fno_block.py:377-414: linear skip, ChannelMLP + soft gating, GELU) as plain PyTorch ops on
    the GPU -- the denominator for the fused layer epilogue.  prm: w, b (conv), w_skip, w1, b1, w2, b2, gate."""
    import torch
    import torch.nn.functional as F
    size = list(x.shape)
    flat = lambda t: t.reshape(size[0], t.shape[1], -1)                                   # noqa: E731
    x_skip = F.conv1d(flat(x), prm["w_skip"]).view(size)
    x_skip_mlp = prm["gate"] * x
    y = torch_cufft_forward(x, prm["w"], prm["b"], n_modes_stored) + x_skip
    if not last:
        y = F.gelu(y)
    h = F.gelu(F.conv1d(flat(y), prm["w1"], prm["b1"]))
    y = F.conv1d(h, prm["w2"], prm["b2"]).view(size) + x_skip_mlp
    return y if last else F.gelu(y)


def run_layer(args):
    """`--layer-only` (own process, called from the main run): the Fourier layer around the conv (SURVEY section 8 f1 / f2) at the
    headline shape -- nb.FNOBlocks (CUDA conv + fused epilogue kernels) next to the same layer on PyTorch eager + cuFFT/cuBLAS/cuDNN,
    plus the epilogue alone and a parity figure of ours against PyTorch (TF32 off for that comparison)."""
    import torch
    import torch.nn.functional as F
    import neuraloperator_b200 as nb
    from neuraloperator_b200 import _lib
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    torch.manual_seed(0)
    blk = nb.FNOBlocks(C, C, MODES, n_layers=2, implementation="reconstructed").to(dev)
    with torch.no_grad():
        blk.channel_mlp_skips[0].weight.add_(0.2 * torch.randn_like(blk.channel_mlp_skips[0].weight))
    conv = blk.convs[0]
    x = torch.randn(B, C, H, W, device=dev)
    g = torch.randn(B, C, H, W, device=dev)
    prm = {"w": conv.weight.tensor, "b": conv.bias, "w_skip": blk.fno_skips[0].conv.weight, "w1": blk.channel_mlp[0].fcs[0].weight,
           "b1": blk.channel_mlp[0].fcs[0].bias, "w2": blk.channel_mlp[0].fcs[1].weight, "b2": blk.channel_mlp[0].fcs[1].bias,
           "gate": blk.channel_mlp_skips[0].weight}
    prm_t = {k: v.detach().clone().requires_grad_(True) for k, v in prm.items()}

    def zero(ps):
        for p_ in ps:
            p_.grad = None

    def ours_layer():
        zero(blk.parameters())
        xx = x.detach().requires_grad_(True)
        blk(xx, 0).backward(g)
        return xx

    def torch_layer():
        zero(prm_t.values())
        xx = x.detach().requires_grad_(True)
        torch_layer_forward(xx, prm_t, conv.n_modes).backward(g)
        return xx

    c0 = _lib.launch_count()
    ours_layer()
    torch.cuda.synchronize(dev)
    launches = _lib.launch_count() - c0
    # parity of the whole layer against PyTorch on the same GPU (fp32 everywhere: TF32 off for this comparison only)
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    xo, xt = ours_layer(), torch_layer()
    with torch.no_grad():
        yo, yt = blk(x, 0), torch_layer_forward(x, prm_t, conv.n_modes)
    rel = lambda a, b_: float((a - b_).abs().max() / b_.abs().max())                         # noqa: E731
    parity = {"y": rel(yo, yt), "dx": rel(xo.grad, xt.grad), "dw_skip": rel(prm["w_skip"].grad, prm_t["w_skip"].grad),
              "dw1": rel(prm["w1"].grad, prm_t["w1"].grad), "dw2": rel(prm["w2"].grad, prm_t["w2"].grad),
              "dgate": rel(prm["gate"].grad, prm_t["gate"].grad), "dW_conv": rel(prm["w"].grad, prm_t["w"].grad)}
    del xo, xt, yo, yt
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    t_ours = time_cuda(ours_layer, 3, 20)
    t_torch = time_cuda(torch_layer, 3, 20)
    # the epilogue alone, forward + backward, the conv output given
    x_fno = torch.randn(B, C, H, W, device=dev)

    def ours_epilogue():
        zero(blk.parameters())
        xx, xf = x.detach().requires_grad_(True), x_fno.detach().requires_grad_(True)
        x1 = nb.channel_mix(xx, prm["w_skip"], add=xf, act=_lib.ACT_GELU)
        blk.channel_mlp[0]._forward_fused(x1, gate=prm["gate"], gated=xx, final_act=_lib.ACT_GELU).backward(g)

    def torch_epilogue():
        zero(prm_t.values())
        xx, xf = x.detach().requires_grad_(True), x_fno.detach().requires_grad_(True)
        size = list(xx.shape)
        flat = lambda t: t.reshape(size[0], t.shape[1], -1)                                # noqa: E731
        x1 = F.gelu(xf + F.conv1d(flat(xx), prm_t["w_skip"]).view(size))
        h = F.gelu(F.conv1d(flat(x1), prm_t["w1"], prm_t["b1"]))
        F.gelu(F.conv1d(h, prm_t["w2"], prm_t["b2"]).view(size) + prm_t["gate"] * xx).backward(g)

    t_ours_ep = time_cuda(ours_epilogue, 3, 20)
    t_torch_ep = time_cuda(torch_epilogue, 3, 20)
    with torch.no_grad():
        def ours_ep_fwd():
            x1 = nb.channel_mix(x, prm["w_skip"], add=x_fno, act=_lib.ACT_GELU)
            blk.channel_mlp[0]._forward_fused(x1, gate=prm["gate"], gated=x, final_act=_lib.ACT_GELU)
        t_ours_ep_fwd = time_cuda(ours_ep_fwd, 3, 20)
    # the same layer step replayed from a CUDA graph (as the headline step is): what is left when the Python / autograd issue time is gone
    t_graph, graph_err = None, None
    try:
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(3):
                ours_layer()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        layer_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(layer_graph):
            ours_layer()
        t_graph = time_cuda(layer_graph.replay, 3, 20)
    except Exception as exc:   # noqa: BLE001 -- reported, the eager numbers stand
        graph_err = repr(exc)[:200]
        try:
            torch.cuda.synchronize(dev)
        except Exception:   # noqa: BLE001
            pass

    # ---- the layer kernels one by one (standalone launches through the C ABI / the functional op, same tensors) ----
    kernels = {}
    try:
        import ctypes
        lib = _lib.load()
        ptr = lambda t_: ctypes.c_void_p(t_.data_ptr()) if t_ is not None else None                     # noqa: E731
        st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        n_pass = 4 * B * C * H * W                                                                       # bytes of one (B, C, H, W) pass
        hid = prm["w1"].shape[0]
        Pn = H * W
        with torch.no_grad():
            h_act = nb.channel_mix(x, prm["w1"], prm["b1"], act=_lib.ACT_GELU)
            gpre = torch.randn(B, C, H, W, device=dev)
            pre = torch.randn(B, C, H, W, device=dev)
            gout, dgated = torch.empty_like(gpre), torch.empty_like(gpre)
            dbias, dgate = torch.empty(C, device=dev), torch.empty(C, device=dev)
            dx_buf = torch.empty_like(x)
            dw_buf = torch.empty(C, C, device=dev)
            gate_flat = prm["gate"].detach().reshape(-1).contiguous()
            w_skip2 = prm["w_skip"].detach().reshape(C, C).contiguous()
            cases = {
                "mix_f1 (x, conv out -> x1: skip GEMM + add + GELU)": (lambda: nb.channel_mix(x, prm["w_skip"], add=x_fno, act=_lib.ACT_GELU), 3.0, 2 * C * C),
                "mix_fc1 (x1 -> h: GEMM + bias + GELU)": (lambda: nb.channel_mix(x, prm["w1"], prm["b1"], act=_lib.ACT_GELU), 1.0 + hid / C, 2 * C * hid),
                "mix_fc2 (h, x -> out: GEMM + bias + gate * x + GELU)": (lambda: nb.channel_mix(h_act, prm["w2"], prm["b2"], gate=prm["gate"], gated=x, act=_lib.ACT_GELU), hid / C + 2.0, 2 * C * hid),
                "act_backward (GELU' + dbias + dgate + d gated)": (lambda: lib.sc_channel_mix_act_backward(ptr(gpre), ptr(pre), _lib.ACT_GELU, ptr(gate_flat), ptr(x), ptr(gout), ptr(dgated), ptr(dbias), ptr(dgate), B, C, Pn, st), 5.0, 0),
                "input_gradient (W^T gpre)": (lambda: lib.sc_channel_mix(ptr(gpre), ptr(w_skip2), 1, C, None, None, None, None, _lib.ACT_IDENTITY, ptr(dx_buf), None, B, C, C, Pn, st), 2.0, 2 * C * C),
                "weight_gradient (sum over points of gpre x^T)": (lambda: lib.sc_channel_mix_weight_grad(ptr(gpre), ptr(x), ptr(dw_buf), B, C, C, Pn, st), 2.0, 2 * C * C),
            }
            for name, (fn, passes, flops_per_point) in cases.items():
                ms_k = time_cuda(fn, 3, 20)
                kb = passes * n_pass
                kernels[name] = {"ms": ms_k, "algorithmic_bytes": kb, "gbs": kb / ms_k / 1e6, "hbm_frac": kb / ms_k / 1e6 / measured_peaks()[0],
                                 "tflops": flops_per_point * B * Pn / ms_k / 1e9}
    except Exception as exc:   # noqa: BLE001
        kernels["error"] = repr(exc)[:200]
    n_bytes = 4 * B * C * H * W
    fwd_bytes = 7 * n_bytes            # f1: x, conv output -> x1 (3); f2: x1 -> h (1.5), h, x -> out (2.5), in units of one (B,C,H,W) pass
    peak, _ = measured_peaks()
    out = {"what": "one Fourier layer (fno_block.py:377-414: SpectralConv + linear skip + GELU + ChannelMLP(0.5) + soft-gating skip + GELU) "
                   "fwd+bwd, eager nn.Module, same shape as the headline step; PyTorch = the same ops on eager + cuFFT/cuBLAS/cuDNN",
           "shape": [B, C, H, W], "ours_ms_per_step": t_ours, "torch_ms_per_step": t_torch, "speedup_vs_torch": t_torch / t_ours,
           "ours_cuda_graph_ms_per_step": t_graph, "cuda_graph_error": graph_err,
           "ours_launches_per_step": launches, "mixing_kernel": "k_channel_mix_tc (tcgen05 bf16x3, opt-in)" if nb.uses_tensor_core_mixing()
           else "k_channel_mix (SIMT fp32, default)",
           "epilogue_only": {"ours_fwd_bwd_ms": t_ours_ep, "torch_fwd_bwd_ms": t_torch_ep, "speedup": t_torch_ep / t_ours_ep,
                             "ours_fwd_ms": t_ours_ep_fwd, "fwd_algorithmic_bytes": fwd_bytes,
                             "fwd_gbs": fwd_bytes / t_ours_ep_fwd / 1e6, "fwd_roofline_frac": fwd_bytes / t_ours_ep_fwd / 1e6 / peak,
                             "kernels": "k_channel_mix (SIMT fp32), k_channel_act_backward, k_channel_weight_grad: first hardware run of "
                                        "these kernels is this driver run (written after the round's GPU minutes were spent)"},
           "kernels": kernels, "max_rel_err_vs_torch_fp32": parity}
    print("LAYER_JSON " + json.dumps(out), flush=True)
    return 0


def layer_block_subprocess(timeout_s=240, tensor_cores=False):
    """Runs `bench.py --layer-only` in its own process: a fault in the (new) layer kernels cannot touch the headline line.
    tensor_cores: the opt-in tcgen05 variant of the mixing kernel (SC_MIX_TC=1) instead of the default exact-fp32 SIMT kernel."""
    try:
        env = dict(os.environ, SC_MIX_TC="1" if tensor_cores else "0")
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--layer-only"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                           text=True, timeout=timeout_s, env=env)
        for ln in r.stdout.splitlines():
            if ln.startswith("LAYER_JSON "):
                return json.loads(ln[len("LAYER_JSON "):])
        return {"error": f"exit code {r.returncode}: {r.stderr.strip()[-400:]}"}
    except Exception as exc:   # noqa: BLE001
        return {"error": repr(exc)[:300]}


class ClockSampler:
    """Samples SM clocks / throttle reasons WHILE the timed region runs.  The timed region is only ~10 ms (50 steps of
    0.2 ms), far below nvidia-smi's sampling period, so NVML is polled directly from a thread (about every millisecond)."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self.mask = 0
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None
            return
        self._thread = threading.Thread(target=self._poll, daemon=True)
        self._thread.start()

    def _poll(self):
        nv = self._nvml
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._handle, nv.NVML_CLOCK_SM)))
                self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._handle))
            except Exception:
                break
            time.sleep(0.0005)

    def stop(self):
        if self._nvml is None or self._thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvml unavailable"]}
        self._stop.set()
        self._thread.join(timeout=2)
        sm = sorted(self.samples)
        reasons = sorted(name for bit, name in self.REASONS.items() if self.mask & bit)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "samples": len(sm), "reasons": reasons}


def cpu_oracle_step_time(steps, warmup, max_seconds=None, budget_seconds=150.0):
    """The reference's CPU path (oracle port: the same torch.fft / einsum calls) on the host cores.

    Thread count: PyTorch's default is every core; on many-core hosts the FFTs of this size run faster on fewer threads, so
    a few candidates are tried once and the fastest is used (reported as `cores`).  Sample: the full batch of 32 when
    `steps + warmup` such steps fit the budget, else the largest leading slice of the batch that does (reported)."""
    import torch
    from oracle import spectral_conv_oracle as O
    cores = os.cpu_count() or 1
    x, w, bias, gy = O.make_inputs(B, C, C, (H, W), MODES, seed=0)

    def one(b):
        t0 = time.perf_counter()
        O.spectral_conv_fwd_bwd(x[:b], w, bias, gy[:b], MODES)
        return time.perf_counter() - t0

    probe = 4
    cands = sorted({c for c in (cores, cores // 2, cores // 4, 32, 16, 8) if 1 <= c <= cores}, reverse=True)
    best_t, best_threads = None, cores
    torch.set_num_threads(cores)
    one(probe)                                       # first-call overheads (plans, allocator)
    for c in cands:
        torch.set_num_threads(c)
        t = one(probe)
        if best_t is None or t < best_t:
            best_t, best_threads = t, c
    torch.set_num_threads(best_threads)
    per_sample = best_t / probe
    budget = budget_seconds if max_seconds is None else max_seconds
    b = int(max(1, min(B, budget / (per_sample * (steps + warmup)))))
    times = []
    t_start = time.perf_counter()
    for i in range(warmup + steps):
        dt = one(b)
        if i >= warmup:
            times.append(dt)
        if max_seconds is not None and i >= warmup and time.perf_counter() - t_start > max_seconds:
            break
    return times, best_threads, b


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    times, cores, sample_b = cpu_oracle_step_time(args.steps, args.warmup,
                                                  budget_seconds=float(os.environ.get("SC_BENCH_CPU_BUDGET_S", "150")))
    total = sum(times)
    value = sample_b * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times) * (B / sample_b), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "arm": "reference CPU path (torch.fft + einsum, oracle port of "
                   "neuralop/layers/spectral_convolution.py:417-570 + autograd backward)", "host_threads": cores},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{len(times)} steps on the first {sample_b} of the {B} samples of the batch, {cores} of "
                                   f"{os.cpu_count()} host threads (fastest of the thread counts tried)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


DUMP_WHOLE_BYTES = 32 << 20    # an output larger than this is written as a fixed sample of DUMP_SAMPLE of its entries
DUMP_SAMPLE = 1 << 21


def dump_outputs(out_dir, outputs):
    """Writes what the timed step returned to its caller as out_dir/<name>.npy in float32 (complex: a trailing (real, imag) axis).
    An output of more than DUMP_WHOLE_BYTES is written flat, as its entries at DUMP_SAMPLE positions drawn once with seed 0 and kept
    in ascending order, so that two runs write the same positions.  At the headline shape y and dx are sampled (8 MB each), dweight
    (18 MB) and dbias are whole."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        t = t.detach()
        a = torch.view_as_real(t) if t.is_complex() else t
        if a.numel() * 4 > DUMP_WHOLE_BYTES:
            rows = a.reshape(-1, 2) if t.is_complex() else a.reshape(-1)
            index = np.sort(np.random.default_rng(0).choice(rows.shape[0], size=DUMP_SAMPLE, replace=False))
            a = rows[torch.from_numpy(index).to(rows.device)]
        np.save(os.path.join(out_dir, name + ".npy"), a.float().cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    import neuraloperator_b200 as nb
    from neuraloperator_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.gpus != world:
        args.gpus = world

    torch.manual_seed(rank)
    conv = nb.SpectralConv(C, C, MODES).to(dev)
    x = torch.randn(B, C, H, W, device=dev, requires_grad=True)
    g = torch.randn(B, C, H, W, device=dev)
    # SC_ALLREDUCE=nccl: NCCL all-reduce; default: the library's own two-shot kernel over NVLink peer memory (sc_allreduce_p2p)
    collective = os.environ.get("SC_ALLREDUCE", "p2p")
    reducer = None
    if world > 1:
        reducer = (nb.PeerGradientAllReducer(conv.parameters(), n_ctas=int(os.environ.get("SC_ALLREDUCE_CTAS", "12")))
                   if collective == "p2p" else nb.GradientAllReducer(conv.parameters()))
    reserved_sms = 0
    if reducer is not None:
        # backward all-reduces dweight / dbias itself: the collective starts on the library's grads_ready event (right after the
        # dweight kernel) on the reducer's stream and runs underneath the dxm contraction and the dx synthesis kernel; the
        # persistent transform launches leave a few SMs free so that NCCL's CTAs find room next to them
        conv.gradient_reducer = reducer
        reserved_sms = int(os.environ.get("SC_RESERVED_SMS", "12"))
        nb.get_plan(dev, (H, W), (H, W), conv.n_modes, conv.max_n_modes).set_reserved_sms(reserved_sms)

    last = {}

    def step_body():
        conv.weight.tensor.grad = None
        conv.bias.grad = None
        x.grad = None
        y = conv(x)
        y.backward(g)
        if args.dump_outputs:
            # the output's storage (a graph replay rewrites it); detached, so that this step's autograd graph is still freed here and
            # not while the next step is being captured
            last["y"] = y.detach()
        if reducer is not None:
            reducer.finish()               # nothing pending (backward already ordered the stream after the collective): ends the step's bookkeeping

    # The step is 6 kernel launches of 10-40 us each (+ one NCCL all-reduce on N > 1): capture it once in a CUDA graph so that the
    # timed loop is not bound by Python / autograd / NCCL enqueue (the eager path is what `e2e` measures).
    graph = None
    graph_error = None
    c0 = _lib.launch_count()
    try:
        step_body()
    except Exception as exc:   # noqa: BLE001 -- e.g. no CUDA symmetric memory on this box: fall back to the NCCL collective
        if reducer is None or collective != "p2p":
            raise
        print(f"bench.py: peer-memory all-reduce unavailable ({exc!r}); using NCCL", file=sys.stderr, flush=True)
        collective = "nccl"
        reducer = nb.GradientAllReducer(conv.parameters())
        conv.gradient_reducer = reducer
        c0 = _lib.launch_count()
        step_body()
    launches_per_step = _lib.launch_count() - c0       # kernels this library launches for one fwd+bwd
    torch.cuda.synchronize(dev)
    if not args.no_graph:
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(3):
                    step_body()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
            graph = torch.cuda.CUDAGraph()
            # thread_local: NCCL's watchdog thread queries events while this thread captures
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                step_body()
        except Exception as exc:  # pragma: no cover - reported in the JSON line
            graph = None
            graph_error = repr(exc)[:300]
            torch.cuda.synchronize(dev)

    def step():
        if graph is not None:
            graph.replay()                 # N > 1: the all-reduce is a node of the graph, forked after the dweight kernel
        else:
            step_body()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"y": last["y"], "dx": x.grad, "dweight": conv.weight.tensor.grad, "dbias": conv.bias.grad})
    launches = _lib.launch_count() - launches0
    if graph is not None:
        launches = launches_per_step * args.steps      # replayed by the graph: the library's own counter does not see them
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = t.item()
    ms_per_step = ms_max / args.steps
    value = world * B / (ms_per_step * 1e-3)

    # ---- roofline of the dominant kernel: the forward analysis transform chain (x -> kept modes) ------------
    plan = nb.get_plan(dev, (H, W), (H, W), conv.n_modes, conv.max_n_modes)
    # three distinct 134 MB inputs in rotation (402 MB > 126 MB L2): no launch finds any of its input in L2
    xs = [x.detach(), g, torch.randn(B, C, H, W, device=dev)]
    for i in range(3):
        nb.analyze(plan, xs[i])
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    reps = 21
    k0.record()
    for i in range(reps):
        nb.analyze(plan, xs[i % 3])
    k1.record()
    torch.cuda.synchronize(dev)
    analyze_ms = k0.elapsed_time(k1) / reps
    del xs
    kept = plan.kept
    m_tot = kept[0] * kept[1]
    # the other two kernels of the step, timed the same way (CUDA events, back to back, rotating buffers > L2 for the images)
    kernels = None
    if rank == 0:
        ys = [torch.empty(B, C, H, W, device=dev) for _ in range(3)]
        ym = torch.randn(B, C, *kept, dtype=torch.complex64, device=dev)
        bias_v = conv.bias.detach().reshape(-1)
        syn_ms = time_cuda_rot(lambda i: nb.synthesize(plan, ym, bias_v), 3, 21)
        xm = torch.randn(B, C, *kept, dtype=torch.complex64, device=dev)
        gm = torch.randn(B, C, *kept, dtype=torch.complex64, device=dev)
        wt = conv.weight.tensor.detach()
        cf_ms = time_cuda_rot(lambda i: nb.contract_dense(plan, xm, wt), 3, 21)
        cb_ms = time_cuda_rot(lambda i: nb.contract_dense_backward(plan, xm, gm, wt), 3, 21)
        syn_bytes = 4 * B * C * H * W + 8 * B * C * m_tot
        con_bytes = 8 * (2 * B * C * m_tot + C * C * m_tot)
        kernels = {"note": "standalone launches through the C ABI, standard mode layout, operands of the contractions L2-resident",
                   "synthesis": {"ms": syn_ms, "bytes": syn_bytes, "gbs": syn_bytes / syn_ms / 1e6},
                   "contract_fwd": {"ms": cf_ms, "bytes": con_bytes, "gbs": con_bytes / cf_ms / 1e6},
                   "contract_bwd_dw_plus_dxm": {"ms": cb_ms, "bytes": 2 * con_bytes, "gbs": 2 * con_bytes / cb_ms / 1e6}}
        del ys, ym, xm, gm
    analyze_bytes = 4 * B * C * H * W + 8 * B * C * m_tot
    peak, peak_src = measured_peaks()
    achieved = analyze_bytes / (analyze_ms * 1e-3) / 1e9
    step_bytes = algorithmic_bytes_step(kept=kept)
    step_gbs = step_bytes / (ms_per_step * 1e-3) / 1e9

    # ---- e2e: same step through the nn.Module with pinned host buffers -------------------------------------
    e2e = None
    cpu_base = None
    if True:
        xh = torch.randn(B, C, H, W).pin_memory()
        gh = torch.randn(B, C, H, W).pin_memory()
        yh = torch.empty(B, C, H, W).pin_memory()
        dxh = torch.empty(B, C, H, W).pin_memory()
        dwh = torch.empty(conv.weight.tensor.shape, dtype=torch.complex64).pin_memory()
        dbh = torch.empty(conv.bias.shape).pin_memory()

        # Host buffers in, host buffers out, every step.  The three legs run on their own streams (H2D of step i+1 and D2H
        # of step i-1 overlap the kernels of step i; PCIe is full duplex), double-buffered on the device side.
        s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream(dev)
        xd_buf = [torch.empty(B, C, H, W, device=dev) for _ in range(2)]
        gd_buf = [torch.empty(B, C, H, W, device=dev) for _ in range(2)]
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_free = [torch.cuda.Event() for _ in range(2)]
        for e in ev_free:
            e.record(main)
        state = {"i": 0}

        def e2e_step():
            i = state["i"]; state["i"] += 1
            sb = i & 1
            with torch.cuda.stream(s_in):
                s_in.wait_event(ev_free[sb])                       # the kernels that last read this buffer pair are done
                xd_buf[sb].copy_(xh, non_blocking=True)
                gd_buf[sb].copy_(gh, non_blocking=True)
                ev_in[sb].record(s_in)
            main.wait_event(ev_in[sb])
            conv.weight.tensor.grad = None
            conv.bias.grad = None
            xd2 = xd_buf[sb].detach().requires_grad_(True)    # fresh leaf over the same storage
            y = conv(xd2)
            y.backward(gd_buf[sb])
            if reducer is not None:
                reducer.finish()
            ev_free[sb].record(main)
            outs = (y.detach(), xd2.grad, conv.weight.tensor.grad, conv.bias.grad)
            s_out.wait_stream(main)
            with torch.cuda.stream(s_out):
                for t in outs:
                    t.record_stream(s_out)
                yh.copy_(outs[0], non_blocking=True)
                dxh.copy_(outs[1], non_blocking=True)
                dwh.copy_(outs[2], non_blocking=True)
                dbh.copy_(outs[3], non_blocking=True)

        def e2e_join():
            main.wait_stream(s_in)
            main.wait_stream(s_out)

        for _ in range(3):
            e2e_step()
        e2e_join()
        barrier()
        n_e2e = max(5, min(args.steps, 20))
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(n_e2e):
            e2e_step()
        e2e_join()
        a1.record()
        barrier()
        t2 = torch.tensor([a0.elapsed_time(a1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        e2e_ms = t2.item() / n_e2e
        h2d = xh.numel() * 4 + gh.numel() * 4
        d2h = yh.numel() * 4 + dxh.numel() * 4 + dwh.numel() * 8 + dbh.numel() * 4
        e2e = {"value": world * B / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": e2e_ms, "steps": n_e2e}

    torch_gpu = None
    configs = None
    fourier_layer = None
    fourier_layer_tc = None
    if rank == 0 and world == 1 and not args.no_configs:
        # the reference op sequence on PyTorch + cuFFT/cuBLAS on this GPU, same shapes, eager -- the ">= 1.5x" denominator;
        # ours eager (nn.Module) next to it, and the graph-replayed headline step
        w_ref = conv.weight.tensor.detach().clone().requires_grad_(True)
        b_ref = conv.bias.detach().clone().requires_grad_(True)

        def ref_step():
            xx = x.detach().requires_grad_(True)
            w_ref.grad = None
            b_ref.grad = None
            torch_cufft_forward(xx, w_ref, b_ref, conv.n_modes).backward(g)

        def ours_eager():
            conv.weight.tensor.grad = None
            conv.bias.grad = None
            x.grad = None
            conv(x).backward(g)

        t_ref = time_cuda(ref_step, 3, 20)
        t_eager = time_cuda(ours_eager, 3, 20)
        torch_gpu = {"what": "reference op sequence (torch.fft rfftn/fftshift/einsum/ifftn/irfft, spectral_convolution.py:429-568) "
                             "fwd+bwd on PyTorch eager + cuFFT/cuBLAS, same GPU, same shapes, CUDA events, 20 steps",
                     "ms_per_step": t_ref, "value": B / t_ref * 1e3, "unit": UNIT,
                     "ours_eager_ms_per_step": t_eager, "speedup_eager": t_ref / t_eager, "speedup_graph": t_ref / ms_per_step}
        del w_ref, b_ref
        configs = {}
        for name, cb, cc, cgrid, cmodes, ckind in OTHER_CONFIGS:
            try:
                configs[name] = measure_config(nb, dev, measured_peaks()[0], cb, cc, cgrid, cmodes, ckind)
            except Exception as exc:   # noqa: BLE001 -- reported in the line, the headline number stands
                configs[name] = {"error": repr(exc)[:300]}
                torch.cuda.synchronize(dev)
        torch.cuda.empty_cache()
        fourier_layer = layer_block_subprocess()
        # the same block with the mixing launches on the opt-in tcgen05 kernel (never run on hardware before this driver run)
        fourier_layer_tc = layer_block_subprocess(tensor_cores=True)

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        times, cores, sample_b = cpu_oracle_step_time(steps=5, warmup=1, max_seconds=15.0)
        cpu_v = sample_b * len(times) / sum(times)
        cpu_base = {"value": cpu_v, "unit": UNIT, "cores": cores, "kind": "port",
                    "sample": f"{len(times)} steps on the first {sample_b} of the {B} samples after 1 warm-up, {cores} of "
                              f"{os.cpu_count()} host threads (oracle port of the reference's torch.fft/einsum CPU path)"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": world * B, "parallelism": f"dp{world}",
                       "l2": "no flush: x, g, y, dx are 134 MB each (537 MB touched per step) > 126 MB L2",
                       "fast_path_mask": plan.uses_fast_path(), "cuda_graph": graph is not None, "cuda_graph_error": graph_error,
                       "allreduce": None if world == 1 else (("one two-shot all-reduce kernel of this library over NVLink peer memory "
                                    "(sc_allreduce_p2p, symmetric memory) " if collective == "p2p" else "one NCCL all-reduce (AVG) ")
                                    + "of dweight+dbias per step, started on the "
                                    "grads_ready event after the dweight kernel, overlapping dxm + dx synthesis"
                                    + (", captured in the CUDA graph" if graph is not None else ", eager")),
                       "reserved_sms": reserved_sms},
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "forward analysis chain (x -> kept modes): " +
                         ("fused tcgen05 kernel" if plan.uses_fast_path() & 1 else "k_real_table_gemm + k_complex_table_gemm"),
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                         "bytes_per_launch": analyze_bytes, "ms_per_launch": analyze_ms, "traffic": ncu_traffic(plan),
                         "step": {"bytes": step_bytes, "achieved": step_gbs, "frac": step_gbs / peak}},
            "kernels": kernels,
            "cpu_baseline": cpu_base,
            "torch_gpu_baseline": torch_gpu,
            "configs": configs,
            "fourier_layer": fourier_layer,
            "fourier_layer_tensor_cores": fourier_layer_tc,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # The captured graph holds NCCL work: tearing the process group down under it has been seen to hang (2-GPU run, round 2).
        # The line is out; leave without the collective teardown.
        sys.stdout.flush()
        sys.stderr.flush()
        torch.cuda.synchronize(dev)
        os._exit(0)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the PyTorch+cuFFT denominator and the other BASELINE configs")
    ap.add_argument("--layer-only", action="store_true", help="internal: measure the Fourier layer (f1 / f2) and print LAYER_JSON")
    ap.add_argument("--no-graph", action="store_true", help="time the eager autograd path instead of a captured CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write y, dx, dweight, dbias of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.layer_only):
        ap.error("--dump-outputs writes the outputs of the timed step of --impl ours")
    if args.layer_only:
        return run_layer(args)
    if args.impl == "reference":
        args.steps = 5 if args.steps is None else args.steps
        args.warmup = 1 if args.warmup is None else args.warmup
        return run_reference(args)
    args.steps = 50 if args.steps is None else args.steps
    args.warmup = 10 if args.warmup is None else args.warmup
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
