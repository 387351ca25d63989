#!/usr/bin/env python
"""bench.py — denoise-steps/s of STDiT3-XL/2 (bf16) on a 64x32x32 latent, BASELINE.json's metric.

One "step" = one denoiser forward on one synthetic latent [1,4,64,32,32] with T5 embeddings
[1,1,300,4096] (36.13 algorithmic TFLOP, BASELINE.md §3 config 2) through the osb200 sm_100a path.

    python bench.py --gpus N --steps K --warmup W          # our arm (N>1 under torchrun)
    python bench.py --impl reference ...                   # the reference's CPU arithmetic (oracle port)
    python bench.py ... --dump-outputs DIR                 # also write the last timed step's output as DIR/*.npy

JSON line keys follow the driver's contract: `value` is device-resident throughput, `e2e` is the same
metric through the public model API with pinned-host inputs copied in and the result copied out
inside the timed region, `roofline` is the dominant kernel family (tcgen05 GEMM) measured live with
CUDA events on the launching stream, `cpu_baseline` is the oracle timed on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "open-sora_b200"))

import torch  # noqa: E402

METRIC = "denoise-steps/sec STDiT3-XL/2 64x32x32 bf16"
WORKLOAD = ("STDiT3-XL/2 (depth 28x2, C=1152, 16x72 heads) one denoise forward, latent 1x4x64x32x32 "
            "(T=64,S=256), text 300x4096 (260 valid)")
UNIT = "steps/s"
T_LAT, H_LAT, W_LAT = 64, 32, 32
FLOP_PER_STEP = 36.13e12  # BASELINE.md §3 / SURVEY.md §8d, per sample per forward


def algorithmic_flops(depth=28, C=1152, T=64, S=256, Ly=300):
    N = T * S
    return depth * (2 * (28 * N * C * C + 4 * Ly * C * C) + 4 * N * C * (S + T + 2 * Ly))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(burst=d.get("bf16_tflops"), sustained=d.get("bf16_tflops_sustained"), hbm=d.get("hbm_gbs"), src="measured")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (restatement of the reference arithmetic) on the host cores
# ------------------------------------------------------------------------------------------------
class CpuReference:
    """The reference arithmetic of the path on the host cores: the fp32 oracle (a restatement - STDiT3 is absent from the
    reference checkout, SURVEY.md 0).  One spatial+temporal block PAIR at the full 16 384 tokens is the timed sample
    (~10 s on 128 cores); a step is 28 such pairs + the embedders / final layer, which are timed once (exact
    extrapolation: the pairs are shape-identical)."""

    def __init__(self):
        from oracle import stdit3_oracle as O

        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        cfg = O.STDiT3_XL_2_config()
        cfg.depth = 1
        self.m = O.STDiT3(cfg).eval()
        O.init_synthetic_weights(self.m)
        self.inp = O.synthetic_inputs(cfg, 1, T_LAT, H_LAT, W_LAT)
        self.T, self.S, C = T_LAT, (H_LAT // 2) * (W_LAT // 2), cfg.hidden_size
        with torch.no_grad():
            self.y, self.y_lens = self.m.encode_text(self.inp["y"], self.inp["mask"])
        self.x0 = torch.randn(1, self.T * self.S, C)
        self.t_mlp = torch.randn(1, 6 * C)
        self.pair()                       # warm-up, untimed: thread pool, allocator, page faults
        t0 = time.perf_counter()
        with torch.no_grad():
            self.m(**self.inp)            # depth-1 model: embedders + 1 pair + final layer (warm by now)
        self.t_full1 = time.perf_counter() - t0

    def pair(self) -> float:
        with torch.no_grad():
            t0 = time.perf_counter()
            x = self.m.spatial_blocks[0](self.x0, self.y, self.t_mlp, self.y_lens, None, None, self.T, self.S)
            self.m.temporal_blocks[0](x, self.y, self.t_mlp, self.y_lens, None, None, self.T, self.S)
            return time.perf_counter() - t0

    def steps_per_s(self, t_pair: float) -> float:
        return 1.0 / (28 * t_pair + max(self.t_full1 - t_pair, 0.0))


def cpu_reference_step(sample_seconds_budget: float = 25.0, repeats: int = 3):
    """(steps_per_s, cores, sample description): median of up to `repeats` warmed pair timings within the budget."""
    ref = CpuReference()
    t_start = time.perf_counter()
    ts = []
    for _ in range(repeats):
        ts.append(ref.pair())
        if time.perf_counter() - t_start > sample_seconds_budget:
            break
    ts.sort()
    t_pair = ts[len(ts) // 2]
    return ref.steps_per_s(t_pair), ref.cores, (
        f"1 of 28 spatial+temporal block pairs of the fp32 oracle at the full 16384 tokens: median of {len(ts)} after a warm-up "
        f"({t_pair:.2f}s, spread {ts[0]:.2f}-{ts[-1]:.2f}s) + embedders/final ({max(ref.t_full1 - t_pair, 0.0):.2f}s), x28 extrapolated")


def library_baseline_step(dev, steps: int = 3):
    """Same-box reference point other than a CPU (BASELINE.md §4): the oracle's plain-PyTorch STDiT3 in bf16 on the GPU -
    cuBLAS GEMMs + torch SDPA + eager elementwise kernels, i.e. what the reference's own stack does without osb200.
    One block PAIR at the full 16384 tokens is timed with CUDA events and extrapolated x28 like the CPU arm (a full
    1.1 B-parameter second model next to the product would not change the number, only the memory footprint)."""
    from oracle import stdit3_oracle as O

    cfg = O.STDiT3_XL_2_config()
    cfg.depth = 1
    with torch.device(dev):
        m = O.STDiT3(cfg).eval()
    O.init_synthetic_weights(m)
    m = m.to(device=dev, dtype=torch.bfloat16)
    inp = O.synthetic_inputs(cfg, 1, T_LAT, H_LAT, W_LAT)
    inp = {k: (v.to(torch.bfloat16) if v.is_floating_point() else v).to(dev) for k, v in inp.items()}
    B, T, S, C = 1, T_LAT, (H_LAT // 2) * (W_LAT // 2), cfg.hidden_size
    with torch.no_grad():
        y, y_lens = m.encode_text(inp["y"], inp["mask"])
        x0 = torch.randn(B, T * S, C, device=dev, dtype=torch.bfloat16)
        t_mlp = torch.randn(B, 6 * C, device=dev, dtype=torch.bfloat16)

        def pair():
            x = m.spatial_blocks[0](x0, y, t_mlp, y_lens, None, None, T, S)
            return m.temporal_blocks[0](x, y, t_mlp, y_lens, None, None, T, S)

        for _ in range(3):
            pair()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            pair()
        e.record()
        torch.cuda.synchronize()
        ms_pair = s.elapsed_time(e) / steps
    del m
    torch.cuda.empty_cache()
    return {"value": 1e3 / (28 * ms_pair), "unit": UNIT, "ms_per_step": 28 * ms_pair,
            "kind": "plain PyTorch bf16 on the same GPU (cuBLAS + SDPA + eager elementwise), the oracle's module code",
            "sample": f"1 of 28 block pairs at 16384 tokens ({ms_pair:.2f} ms, CUDA events, 3 warm-ups), x28; embedders excluded"}


def run_reference(args, rank, budget_s: float = 170.0):
    """`--impl reference`: every step is ONE timed block pair (the bounded sample), W warm-up pairs are discarded, K are kept;
    a time budget caps the run at a few minutes whatever K is (later steps then reuse the median of the measured ones)."""
    if rank != 0:
        return
    t0 = time.perf_counter()
    ref = CpuReference()
    pairs = []
    for i in range(args.warmup + args.steps):
        if time.perf_counter() - t0 > budget_s and len(pairs) >= 3:
            break
        t = ref.pair()
        if i >= args.warmup:
            pairs.append(t)
    if not pairs:
        pairs.append(ref.pair())
    pairs.sort()
    t_pair = pairs[len(pairs) // 2]
    v = ref.steps_per_s(t_pair)
    sample = (f"each step = 1 of 28 block pairs of the fp32 oracle at the full 16384 tokens (x28 + embedders/final "
              f"{max(ref.t_full1 - t_pair, 0.0):.2f}s): median pair {t_pair:.2f}s over {len(pairs)} timed steps "
              f"(spread {pairs[0]:.2f}-{pairs[-1]:.2f}s) after {args.warmup} warm-up pairs; budget {budget_s:.0f}s")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 / v, "higher_is_better": True,
        "scaling": "weak" if args.parallel == "dp" else "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "implementation": "CPU oracle port of the path (STDiT3 is absent from the reference "
                                                           "checkout, SURVEY.md §0), all host threads"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": ref.cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def build_model(device):
    """Random-init STDiT3-XL/2 built and initialised ON the device (1.1 B parameters: CPU init would take minutes
    per rank; there are no checkpoints offline)."""
    from opensora.registry import MODELS, build_module

    torch.manual_seed(1234)   # module constructors draw from the default generators: identical on every rank
    with torch.device(device):
        m = build_module(dict(type="STDiT3-XL/2"), MODELS).eval()
    # every parameter and buffer comes from ONE explicitly seeded stream, so all ranks of a multi-GPU run hold the same
    # model whatever the per-device default generators did (a sequence-parallel run with rank-dependent adaLN tables
    # cannot match the single-GPU forward)
    g = torch.Generator(device=device).manual_seed(1234)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if "scale_shift_table" in n:
                p.copy_(torch.randn(p.shape, generator=g, device=device) / (p.shape[-1] ** 0.5))
            elif p.dim() >= 2:
                p.copy_(torch.randn(p.shape, generator=g, device=device) * (0.7 / (p[0].numel() ** 0.5)))
            elif n.endswith("bias"):
                p.copy_(0.02 * torch.randn(p.shape, generator=g, device=device))
            else:   # norm weights
                p.copy_(1.0 + 0.1 * torch.randn(p.shape, generator=g, device=device))
        for n, b in m.named_buffers():
            if b.is_floating_point():
                b.copy_(torch.randn(b.shape, generator=g, device=device) / (b.shape[-1] ** 0.5))
    return m.to(device=device, dtype=torch.bfloat16)


def host_inputs(seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(1, 4, T_LAT, H_LAT, W_LAT, generator=g).pin_memory()
    y = torch.randn(1, 1, 300, 4096, generator=g).to(torch.bfloat16).pin_memory()
    mask = torch.ones(1, 300, dtype=torch.int64)
    mask[0, 260:] = 0
    return dict(x=x, timestep=torch.tensor([500.0]).pin_memory(), y=y, mask=mask.pin_memory(), fps=torch.tensor([24.0]),
                height=torch.tensor([256.0]), width=torch.tensor([256.0]))


def vae_leg():
    """Second half of BASELINE.json's metric: causal 3D VAE encode / decode fps on a synthetic 65x720x1280 video
    (configs[2]), untiled, bf16, one B200; per-family device times from the same CUDA-event hook as the roofline."""
    import osb200
    from tests.vae_bench import DEC_TF, ENC_TF, run

    del_model = torch.cuda.empty_cache
    del_model()
    try:
        res = run(65, 720, 1280, iters=2)
        osb200.start_profile()
        from opensora.registry import MODELS, build_module

        torch.manual_seed(0)
        with torch.device("cuda"):
            m = build_module(dict(type="hunyuan_vae"), MODELS, device_map="cuda").eval()
        with torch.no_grad():
            z = torch.randn(1, 16, 17, 90, 160, device="cuda").to(torch.bfloat16)
            m.decode(z)
            osb200.stop_profile()
            osb200.start_profile()
            m.decode(z)
        fam = {}
        for name, work, t in osb200.stop_profile():
            f = fam.setdefault(name, [0, 0.0])
            f[0] += 1
            f[1] += t
        res["decode_families_ms"] = {k: {"launches": v[0], "ms": round(v[1], 2)} for k, v in fam.items()}
        conv_ms = fam.get("conv3d", [0, 1.0])[1]
        pk = peaks()
        res["conv_roofline"] = {"bound": "tensor", "kernel": "gemm_bf16_kernel<conv> (all conv3d launches of one decode)",
                                "achieved": DEC_TF / (conv_ms * 1e-3), "peak": pk["sustained"], "unit": "TFLOP/s",
                                "frac": DEC_TF / (conv_ms * 1e-3) / pk["sustained"],
                                "note": "algorithmic conv FLOPs (1017.9 TF, SURVEY.md 8d) / summed conv3d device time"}
        res["config"] = {"workload": "hunyuan causal 3D VAE, video 1x3x65x720x1280 <-> latent 1x16x17x90x160, untiled, bf16",
                         "algorithmic_conv_tflop": {"encode": ENC_TF, "decode": DEC_TF},
                         "mid_block_attention": "torch SDPA per frame prefix (library kernel; osb200 D=512 kernel pending)"}
        res["e2e"] = _vae_e2e(m, z, tuple(res["out_shape"]))
        res["tiled"] = _vae_tiled(m, z)
        del m
        torch.cuda.empty_cache()
        res["cpu_baseline"] = _vae_cpu_baseline()
        return res
    except Exception as e:  # the headline metric above must survive a VAE-leg failure
        return {"error": repr(e)[:300]}


def _vae_e2e(m, z, shape):
    """Decode through the public API with HOST buffers: the latent comes from pinned host memory and the video goes back to
    pinned host memory inside the timed region (CUDA events).  Own try/except: the device-timed numbers above survive."""
    try:
        zh = z.cpu().pin_memory()
        with torch.no_grad():
            out_h = torch.empty(shape, dtype=torch.bfloat16).pin_memory()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            v = m.decode(zh.to("cuda", non_blocking=True))
            out_h.copy_(v, non_blocking=True)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        return {"value": shape[2] / (ms * 1e-3), "unit": "frames/s", "ms": ms, "h2d_bytes": zh.numel() * zh.element_size(),
                "d2h_bytes": out_h.numel() * out_h.element_size()}
    except Exception as e:
        return {"error": repr(e)[:200]}


def _vae_tiled(m, z):
    """The same decode in the tiling mode the reference's VAE config ships (`configs/vae/inference/hunyuanvideo_vae.py`:
    use_spatial_tiling + use_temporal_tiling: 256-px / 64-frame tiles, 25 % overlap, linear blends - SURVEY.md 8d asks for both
    modes).  Tiles recompute their overlaps (~1.65x the convolution work at 720 x 1280) and normalise per tile, so this is a
    different computation from the untiled decode, timed for reference.  Own try/except."""
    try:
        m.enable_tiling(True)
        with torch.no_grad():
            v = m.decode(z)                       # warm-up at the tile shapes
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            v = m.decode(z)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        return {"decode_ms": ms, "decode_fps": v.shape[2] / (ms * 1e-3), "out_shape": list(v.shape),
                "mode": "spatial 256 px + temporal 64 frames, overlap 0.25 (the reference config's default)"}
    except Exception as e:
        return {"error": repr(e)[:200]}
    finally:
        m.enable_tiling(False)


def _vae_cpu_baseline():
    """The oracle's CausalConv3d (replicate pad + conv3d, fp32, all host threads) on a bounded sample - one 128 -> 128 3x3x3
    layer of the decoder's last stage at 5 x 180 x 320 positions - scaled by algorithmic FLOPs to the whole 1017.9 TF decode."""
    try:
        from oracle import vae_oracle as V
        from tests.vae_bench import DEC_TF

        torch.set_num_threads(os.cpu_count() or 1)
        g = torch.Generator().manual_seed(2)
        x = torch.randn(1, 128, 5, 180, 320, generator=g)
        w = torch.randn(128, 128, 3, 3, 3, generator=g) * 0.02
        b = torch.zeros(128)
        flop = 2.0 * 27 * 128 * 128 * 5 * 180 * 320
        with torch.no_grad():
            V.causal_conv3d(x, w, b)                      # warm-up
            ts = []
            t_end = time.perf_counter() + 20.0
            while len(ts) < 3 and (not ts or time.perf_counter() < t_end):
                t0 = time.perf_counter()
                V.causal_conv3d(x, w, b)
                ts.append(time.perf_counter() - t0)
        t = sorted(ts)[len(ts) // 2]
        decode_s = DEC_TF * 1e12 / (flop / t)
        return {"value": 65 / decode_s, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port",
                "sample": f"oracle CausalConv3d 128->128 on 5x180x320 positions ({flop / 1e9:.0f} GFLOP, median of {len(ts)}: {t:.2f} s = "
                          f"{flop / t / 1e12:.2f} TF/s), scaled to the decode's {DEC_TF} algorithmic conv TFLOP"}
    except Exception as e:
        return {"error": repr(e)[:200]}


# ---- MMDiT leg (SURVEY.md 8d Cfg5 at the 256px shape): its own process, so nothing it does can reach the headline -------------
MMDIT_256PX = dict(in_channels=64, vec_in_dim=768, context_in_dim=4096, hidden_size=3072, mlp_ratio=4.0, num_heads=24, depth=19,
                   depth_single_blocks=38, axes_dim=[16, 56, 56], theta=10_000, qkv_bias=True, guidance_embed=False, cond_embed=True,
                   fused_qkv=False, use_liger_rope=True)   # configs/diffusion/inference/256px.py:36-55


def mmdit_leg_main():
    """`bench.py --leg mmdit`: one denoiser forward of the in-tree MMDiT at the reference's 256px inference shape (B = 3 CFG
    branches, 33 x 12 x 21 = 8 316 image tokens + 512 text tokens, C = 3072, 24 x 128 heads, 19 + 38 blocks, the shipped
    `fused_qkv=False` / Liger-RoPE layout), random-init bf16 weights created on the device, inputs resident.  Prints one JSON
    object.  First written after the round-2 GPU budget was spent: it has never run before the driver runs it."""
    import osb200
    from opensora.models.mmdit.model import MMDiTConfig, MMDiTModel

    torch.cuda.set_device(0)
    osb200.init(0)
    cfg = MMDIT_256PX
    B, T, H, W, Lt = 3, 33, 12, 21, 512
    Li = T * H * W
    L, C = Li + Lt, cfg["hidden_size"]
    tflop = B * (cfg["depth"] + cfg["depth_single_blocks"]) * (24.0 * C * C * L + 4.0 * L * L * C) / 1e12   # SURVEY.md 8d
    torch.manual_seed(0)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.bfloat16)
    try:
        with torch.device("cuda"):
            model = MMDiTModel(MMDiTConfig(from_pretrained=None, cache_dir=None, **cfg)).eval()
    finally:
        torch.set_default_dtype(prev)
    with torch.no_grad():
        torch.nn.init.normal_(model.cond_in.weight, std=0.02)    # zero-init upstream: every path must carry signal (SURVEY 8d)
    g = torch.Generator(device="cuda").manual_seed(5)
    rb = lambda *s: torch.randn(*s, device="cuda", generator=g).to(torch.bfloat16)   # noqa: E731
    ids = torch.stack(torch.meshgrid(torch.arange(T), torch.arange(H), torch.arange(W), indexing="ij"), -1).reshape(1, Li, 3)
    inp = dict(img=rb(B, Li, 64), img_ids=ids.float().repeat(B, 1, 1).cuda().to(torch.bfloat16), txt=rb(B, Lt, 4096),
               txt_ids=torch.zeros(B, Lt, 3, device="cuda", dtype=torch.bfloat16), timesteps=torch.full((B,), 0.7, device="cuda", dtype=torch.bfloat16),
               y_vec=rb(B, 768), cond=rb(B, Li, 68), guidance=None)
    res = {"workload": f"MMDiT (flux) 256px inference shape: B={B}, L={Lt}+{Li}, C={C}, 24x128 heads, 19+38 blocks, fused_qkv=False, liger rope, bf16",
           "algorithmic_tflop_per_step": tflop, "params_b": sum(p.numel() for p in model.parameters()) / 1e9}
    with torch.no_grad():
        out = model(**inp)                      # warm-up: packs weights, caches pe / RoPE tables
        torch.cuda.synchronize()
        res["finite"] = bool(torch.isfinite(out.float()).all())
        res["out_shape"] = list(out.shape)
        steps = 2
        l0 = osb200.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = model(**inp)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        pk = peaks()
        res.update(metric="denoise-steps/sec MMDiT 256px (B=3 CFG batch) bf16", value=1e3 / ms, unit="steps/s", ms_per_step=ms,
                   tflops=tflop / (ms * 1e-3), frac_of_sustained_peak=tflop / (ms * 1e-3) / pk["sustained"],
                   gpu_launches_per_step=(osb200.launch_count() - l0) // steps, peak_gb=torch.cuda.max_memory_allocated() / 2**30)
        osb200.start_profile()
        model(**inp)
        fam = {}
        for name, work, t in osb200.stop_profile():
            f = fam.setdefault(name, [0, 0.0])
            f[0] += 1
            f[1] += t
        res["families_ms"] = {k: {"launches": v[0], "ms": round(v[1], 2)} for k, v in fam.items()}
    print(json.dumps(res), flush=True)


def mmdit_leg(timeout_s: float = 180.0):
    """Run the MMDiT leg in a child process (own CUDA context, hard time limit) and return its JSON object, or the reason it
    produced none.  The parent has finished all of its own device work before this is called."""
    try:
        torch.cuda.empty_cache()
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--leg", "mmdit"], capture_output=True, text=True,
                           timeout=timeout_s, cwd=ROOT)
        for ln in reversed(p.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"error": f"no result (rc {p.returncode}): " + (p.stderr or p.stdout)[-400:]}
    except subprocess.TimeoutExpired:
        return {"error": f"timed out after {timeout_s:.0f} s"}
    except Exception as e:
        return {"error": repr(e)[:300]}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each tensor as `out_dir/<name>.npy` in float32 (whole: the denoiser output of one step is 2 MB)."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    host = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    assert sum(a.nbytes for a in host.values()) <= DUMP_LIMIT_BYTES
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="osb200", choices=["osb200", "reference"])
    ap.add_argument("--parallel", default="sp", choices=["sp", "dp"],
                    help="N>1: sp (default) = ONE sample sequence-sharded over the ranks, exchange at the spatial<->temporal "
                         "boundary (north_star's partition; strong scaling; the dp replica rate is reported beside it as "
                         "`dp_replicas`); dp = one independent sample per rank, no data-path collective (weak scaling)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--graph", dest="graph", action="store_true", default=None,
                    help="replay the step as one CUDA graph (model.capture); default: on for sp, off otherwise")
    ap.add_argument("--no-graph", dest="graph", action="store_false")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--leg", default=None, choices=["mmdit"], help="run ONE auxiliary leg in this process and print its JSON")
    ap.add_argument("--no-mmdit", action="store_true", help="skip the MMDiT 256px leg (a child process of the N = 1 run)")
    ap.add_argument("--no-vae", action="store_true", help="skip the VAE leg (encode/decode fps of BASELINE.json's metric)")
    ap.add_argument("--profile-step", action="store_true",
                    help="after warm-up, bracket ONE step with cudaProfilerStart/Stop and exit (for `ncu --profile-from-start off`: "
                         "the launch list of exactly one step; prints no bench line)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (the denoiser output, float32) as DIR/<name>.npy; the inputs "
                         "and weights are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "osb200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.leg == "mmdit":
        mmdit_leg_main()
        return
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch.distributed as dist

    import osb200

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    osb200.init(local_rank)
    model = build_model(dev)
    mode = args.parallel if world > 1 else "single"
    if args.graph is None:
        args.graph = mode == "sp"   # 2 048 tokens per rank at N = 8: the step is launch-bound without a graph
    hin = host_inputs(4321 + (rank if mode == "dp" else 0))
    # height / width are host scalars (they select the cached positional table; STDiT3.capture documents them as host
    # values): a device copy would cost one device synchronisation per forward
    din = {k: (v if k in ("height", "width") else v.to(dev, non_blocking=True)) for k, v in hin.items()}
    sp_check = None
    if mode == "sp":
        # in-run parity of the partition: the sequence-parallel forward against the SAME model's single-GPU forward
        with torch.no_grad():
            single = model(**din).clone()
            model.enable_sequence_parallel(dist.group.WORLD)
            spo = model(**din)
        torch.cuda.synchronize()
        diff = (spo.double() - single.double())
        sp_check = {"sp_matches_single_gpu": bool(torch.equal(spo, single)),
                    "max_abs": float(diff.abs().max()), "rel_l2": float(diff.norm() / single.double().norm()),
                    "ref_absmax": float(single.abs().max())}
        flag = torch.tensor([1.0 if sp_check["rel_l2"] < 2e-3 else 0.0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        sp_check["all_ranks_ok"] = bool(flag.item() == 1.0)
        sp_check["exchange"] = model.sp_exchange_kind
        del single, spo

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            fn()
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    out_holder = {}
    replay = None
    graph_launches = 0
    if args.graph:
        replay = model.capture(**{**din, "height": hin["height"], "width": hin["width"]})
        graph_launches = replay.kernel_launches   # osb200 kernels recorded into the graph

    def step_resident():
        with torch.no_grad():
            out_holder["o"] = replay(**din) if replay is not None else model(**din)

    h2d = sum(v.numel() * v.element_size() for k, v in hin.items() if k in ("x", "timestep", "y", "mask"))
    host_out = torch.empty(1, 8, T_LAT, H_LAT, W_LAT, dtype=torch.float32).pin_memory()

    def step_e2e():  # the call a user makes: host tensors in, host tensor out
        with torch.no_grad():
            if replay is not None:   # host tensors are copied straight into the graph's static inputs
                o = replay(**hin)
            else:
                o = model(**{k: (v if k in ("height", "width") else v.to(dev, non_blocking=True)) for k, v in hin.items()})
            host_out.copy_(o, non_blocking=True)

    for _ in range(args.warmup):
        step_resident()
    if args.profile_step:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step_resident()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    l0 = osb200.launch_count()
    ms = timed(step_resident, args.steps)
    # a graph replay returns its static output buffer, which the e2e steps below overwrite: keep a copy of this one
    last_out = out_holder["o"].clone() if args.dump_outputs else None
    launches = osb200.launch_count() - l0
    if replay is not None:   # a replay re-issues the captured kernels without passing through the C ABI counter
        launches = graph_launches * args.steps
    clk = clocks.stop() if rank == 0 else None
    for _ in range(2):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps)

    # ---- roofline leg: per-launch CUDA-event timing of every kernel family over one more pass ------
    osb200.start_profile()
    for _ in range(2):   # always the eager path: per-launch events cannot bracket kernels inside a graph replay
        with torch.no_grad():
            model(**din)
    rec = osb200.stop_profile()
    fam = {}
    for name, work, t in rec:
        f = fam.setdefault(name, [0.0, 0.0, 0])
        f[0] += work
        f[1] += t
        f[2] += 1

    units = args.steps * (world if mode == "dp" else 1)
    value = units / (ms / 1e3)
    e2e = units / (ms_e2e / 1e3)

    # sp runs also report the replica rate (one independent sample per rank, no collective): the weak-scaling number
    dp_extra = None
    if mode == "sp":
        model.enable_sequence_parallel(None)
        hin_dp = host_inputs(4321 + rank)
        din_dp = {k: (v if k in ("height", "width") else v.to(dev, non_blocking=True)) for k, v in hin_dp.items()}

        def step_dp():
            with torch.no_grad():
                out_holder["o"] = model(**din_dp)

        for _ in range(3):
            step_dp()
        ms_dp = timed(step_dp, args.steps)
        dp_extra = {"value": args.steps * world / (ms_dp / 1e3), "unit": "samples/s", "ms_per_step": ms_dp / args.steps,
                    "scaling": "weak", "note": "one independent sample per rank, no data-path collective"}
    if rank != 0:
        if world > 1:
            _finish(dist)
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"stdit3_out": last_out})
    pk = peaks()
    g = fam.get("gemm", [0.0, 1.0, 1])
    gemm_tflops = g[0] / (g[1] * 1e-3) / 1e12
    traffic = None
    tp = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("dram_bytes_per_launch")
    roof = {"bound": "tensor", "kernel": "gemm_bf16_kernel (all %d launches of a step, FLOP-weighted)" % (g[2] // 2),
            "achieved": gemm_tflops, "peak": pk["sustained"], "unit": "TFLOP/s", "frac": gemm_tflops / pk["sustained"],
            "peak_kind": f"bf16_tflops_sustained of {pk['src']} (burst {pk['burst']})", "traffic": traffic,
            "step_frac_of_peak": (FLOP_PER_STEP * value / (world if mode == 'dp' else 1) / 1e12) / pk["sustained"] / (world if mode == 'sp' else 1),
            "families": {k: {"launches_per_step": v[2] // 2, "ms_per_step": v[1] / 2,
                             ("tflops" if k != "ln_modulate" else "gbs"): (v[0] / (v[1] * 1e-3) / (1e12 if k != "ln_modulate" else 1e9))}
                         for k, v in fam.items()}}
    vae = None
    if not args.no_vae and world == 1:
        vae = vae_leg()
    lib = None
    if not args.no_library_baseline and world == 1:
        try:
            lib = library_baseline_step(dev)
        except Exception as e:   # a reported baseline must not take the headline down with it
            lib = {"error": repr(e)[:300]}
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        v, cores, sample = cpu_reference_step()
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
    mmdit = None
    if not args.no_mmdit and world == 1:
        torch.cuda.synchronize()     # every number of this line is final before the child process touches the GPU
        mmdit = mmdit_leg()
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak" if args.parallel == "dp" else "strong",   # the --parallel mode the N > 1 runs of this line use (default sp: total work fixed)
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic (seeded N(0,1) latents / T5 embeddings, random-init weights)",
        "config": {"workload": WORKLOAD, "parallelism": mode + str(world), "cuda_graph": bool(args.graph),
                   "l2": "weights 2.2 GB + activations stream through every step (>> 126 MB L2): inputs larger than L2",
                   "algorithmic_tflop_per_step": FLOP_PER_STEP / 1e12},
        "clocks": clk, "gpu_launches": launches,
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": host_out.numel() * 4,
                "ms_per_step": ms_e2e / args.steps},
        "roofline": roof, "cpu_baseline": cpu, "library_baseline": lib, "vae": vae, "mmdit": mmdit,
    }
    if sp_check is not None:
        line["sp_check"] = sp_check
        line["config"]["exchange"] = sp_check.get("exchange")
    if dp_extra is not None:
        line["dp_replicas"] = dp_extra
    print(json.dumps(line), flush=True)
    if world > 1:
        _finish(dist)


def _finish(dist):
    """Multi-rank teardown: all work is done and the line is printed; symmetric-memory handles and captured graphs make an
    orderly interpreter shutdown slow (and it has hung a box) - synchronise, then leave."""
    torch.cuda.synchronize()
    try:
        dist.barrier()
    except Exception:
        pass
    sys.stdout.flush()
    os._exit(0)


if __name__ == "__main__":
    main()
