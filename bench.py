#!/usr/bin/env python
"""bench.py — VQ-IMG 256x256 images/sec (Encoder -> VectorQuantizer -> Decoder forward+backward), batch 32 per GPU.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line from rank 0.
  value  : whole-job images/s with the batch already resident in HBM (CUDA-event timed, max over ranks)
  e2e    : the same metric through the public module API with HOST (pinned) input buffers: H2D copy of the batch
           and a D2H read of the loss inside every timed step
  roofline     : dominant kernel (conv3x3 128->128 @256^2, batch 32) timed live with CUDA events
  vq           : the second headline metric (VQ argmin GB/s, algorithmic bytes) measured live
  cpu_baseline : the CPU oracle (a restatement of the reference; kind "port") timed on this box's host cores
`--impl reference` times that same CPU implementation alone and prints the line with "impl": "reference".
`--dump-outputs DIR` writes what the last timed step computed (dump_outputs) so that two builds can be compared output for
output: model, weights and batch come from fixed seeds, so the same arguments give the same inputs on every run.
Workload = BASELINE.json configs[1]; synthetic data (torch.rand images, seeded default-init weights, N(0,1) codebook,
q_counter past the re-init window so the real VQ branch runs — SURVEY.md 8d). Proxy loss: L1 + codebook term.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "make-a-scene_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

IMG_CFG = dict(z_channels=256, in_channels=3, out_channels=3, channels=[128, 128, 128, 256, 512, 512], num_res_blocks=2,
               resolution=512, attn_resolutions=[32], dropout=0.0)
N_EMBED, EMBED_DIM, BATCH, RES = 8192, 256, 32, 256
METRIC = "VQ-IMG 256^2 images/sec (enc+VQ+dec fwd+bwd)"
FLOP_PER_IMG_FWD_BWD = 1.336e12     # BASELINE.md section 2


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


SEG_CFG = dict(z_channels=256, in_channels=159, out_channels=159, channels=[128, 128, 128, 256, 512, 512], num_res_blocks=2,
               resolution=256, attn_resolutions=[16], dropout=0.0)     # conf/seg_config.yaml (out_channels given explicitly)
SEG_METRIC = "VQ-SEG 256^2 images/sec (enc+VQ+dec fwd+bwd, weighted BCE)"


def build_model(workload="vqimg"):
    from models import VQBASE
    torch.manual_seed(0)
    if workload == "vqseg":
        m = VQBASE(SEG_CFG, 1024, 256, 2000, 12500)
    else:
        m = VQBASE(IMG_CFG, N_EMBED, EMBED_DIM, 3000, 12500)
    with torch.no_grad():
        m.quantize.embedding.weight.normal_()
    m.quantize.q_counter = 10 ** 6
    m.train()
    return m


def cpu_threads():
    """All host cores, also under torchrun (which exports OMP_NUM_THREADS=1 to every rank)."""
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        pass
    if n > 64:          # SMT siblings: PyTorch's CPU kernels run slower with two threads per core (measured 64.6 s/step at 128)
        n //= 2
    torch.set_num_threads(n)
    return n


def cpu_reference_steps(steps, warmup, batch=2, budget=None):
    """The reference's own CPU implementation of the path, all host threads, on a sample of the workload (`batch` images
    per step instead of 32); with `budget` (seconds) the timed steps stop once they exceed it. kind "reference": the
    UNMODIFIED reference modules staged under oracle/_ref (oracle/vendor_ref.py; BASELINE.md section 3); kind "port": the
    oracle restatement, when oracle/_ref is absent."""
    from oracle import vendor_ref
    cores = cpu_threads()
    x = torch.rand(batch, 3, RES, RES, generator=torch.Generator().manual_seed(1234))
    if vendor_ref.available():
        kind = "reference"
        ref_models = vendor_ref.load_models()
        torch.manual_seed(0)
        m = ref_models.VQBASE(IMG_CFG, N_EMBED, EMBED_DIM, 3000, 12500)
        with torch.no_grad():
            m.quantize.embedding.weight.normal_()
        m.quantize.q_counter = 10 ** 6
        m.train()

        def one():
            m.zero_grad(set_to_none=True)
            dec, diff = m(x)
            ((x - dec).abs().mean() + diff).backward()
    else:
        kind = "port"
        from oracle import vqgan_oracle as O
        torch.manual_seed(0)
        sd = {k: v.detach().clone() for k, v in build_model().state_dict().items()}   # CPU parameter holders, no kernels
        params = {k: v.requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running" not in k}
        sd.update(params)

        def one():
            for p in params.values():
                p.grad = None
            dec, diff, _ = O.vqbase_forward(sd, IMG_CFG, x)
            O.proxy_loss(x, dec, diff).backward()
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        one()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
            if budget is not None and sum(times) > budget:
                break
    return dict(value=batch * len(times) / sum(times), sec=sum(times) / len(times), done=len(times), kind=kind, cores=cores,
                batch=batch)


def run_reference(args, rank):
    if rank != 0:
        return
    r = cpu_reference_steps(args.steps, args.warmup, batch=2)
    v = r["value"]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": r["done"],
            "warmup": args.warmup, "ms_per_step": r["sec"] * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "VQ-IMG 256x256 codebook=8192 dim=256 (BASELINE configs[1])",
                       "sample": "%d images per step (the batch-32 workload sampled at batch %d)" % (r["batch"], r["batch"])},
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": r["cores"], "kind": r["kind"],
                             "sample": "%d timed fwd+bwd steps of %d images (%.1f s/step; %s)" % (
                                 r["done"], r["batch"], r["sec"],
                                 "unmodified reference modules from oracle/_ref, stock PyTorch CPU kernels" if r["kind"] == "reference"
                                 else "oracle port: oracle/_ref not staged")},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def time_kernel(fn, iters=5, warm=2):
    for _ in range(warm):
        fn()
    st = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(st)
    for _ in range(iters):
        fn()
    e1.record(st)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3


def dominant_kernel_roofline(dev, pk):
    """The kernel with the largest share of the step: the 3x3 convolution on its dominant layer, conv3x3 128->128 @256x256,
    batch 32 (M=2,097,152 N=128 K=1152; 47.7% of the step's FLOPs run on this layer shape), launched as the model launches it:
    the TMA-fed fp16-operand kernel shift_gemm_t16 reading the fp16 activation shadow (forward / data gradient; bias epilogue),
    weights packed once. `others`: the shadow-fed weight-gradient kernel on the same layer and, when the TMA path is off or the
    operand format is not f16, the register-staged kernel. Achieved = algorithmic FLOPs / CUDA-event time."""
    from mas_b200 import _lib as L, ops
    x = torch.randn(BATCH, 128, RES, RES, device=dev).contiguous(memory_format=torch.channels_last)
    w = torch.randn(128, 128, 3, 3, device=dev) * 0.03
    b = torch.zeros(128, device=dev)
    flops = 2.0 * BATCH * RES * RES * 128 * 128 * 9
    tc = ops.get_impl() != L.IMPL_SIMT and ops.conv_tc_eligible(x, 128, L.CONV_S1)
    fmt = ops.get_operand_format() if tc else "fp32"
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    tj = json.load(open(tp)) if os.path.exists(tp) else {}
    others = []

    def entry(name, sec, alg_bytes, tkey):
        ach = flops / sec / 1e12
        return {"kernel": name, "bound": "tensor", "achieved": ach, "peak": pk["bf16"], "unit": "TFLOP/s", "frac": ach / pk["bf16"],
                "traffic": tj.get(tkey), "ms_per_launch": sec * 1e3, "algorithmic_bytes_per_launch": alg_bytes}

    wbytes = 2 * 128 * 128 * 9
    if fmt == "f16" and ops.conv_tma_on():
        x16 = ops.to_half(x)
        y = torch.empty_like(x)
        wt = ops._packed_conv_weight(w, w, 128, 128, False, dev, False, True)
        fn = lambda: L.call("mas_conv3x3_fprop_tc16h", x16, L.t4(x16), wt, b, None, y, L.t4(y), None, None)
        main = entry("shift_gemm_t16 (TMA-fed tcgen05 kind::f16, fp32 accumulate) conv3x3 128->128 @256^2 x32",
                     time_kernel(fn, iters=6, warm=3), 2.0 * BATCH * RES * RES * 128 + 4.0 * BATCH * RES * RES * 128 + wbytes,
                     "conv3x3_tma_128_128_256_bytes_per_launch")
        dy = torch.randn(BATCH, 128, RES, RES, device=dev).contiguous(memory_format=torch.channels_last) * 1e-6
        am = ops.amax(dy)
        dy16 = ops.to_half(dy, am)
        del dy
        gfn = lambda: ops.conv3x3_wgrad_raw(x16, dy16, 128, 128, L.CONV_S1, dy_amax=am)
        others.append(entry("wgrad_t16 + reduction (weight gradient from the fp16 shadows) conv3x3 128->128 @256^2 x32",
                            time_kernel(gfn, iters=6, warm=3), 2 * 2.0 * BATCH * RES * RES * 128 + 4.0 * 128 * 128 * 9,
                            "wgrad_t16_128_128_256_bytes_per_launch"))
        del x16, y, dy16
    xa = ops.amax(x) if fmt == "f16" else None
    fn = lambda: ops.conv3x3_raw(x, w, b, None, L.CONV_S1, x_amax=xa)
    kname = {"f16": "shift_gemm_tc<9,f16> (register-staged fp16 operands; strided / upsampling / unshadowed layers)",
             "tf32": "shift_gemm_tc<9> (tcgen05 TF32)", "fp32": "conv_fprop_simt (fp32 FFMA)"}[fmt] + " conv3x3 128->128 @256^2 x32"
    staged = entry(kname, time_kernel(fn, iters=6, warm=3), 4.0 * BATCH * RES * RES * 256 + 4 * 128 * 128 * 9,
                   "conv3x3_128_128_256_bytes_per_launch")
    if fmt == "f16" and ops.conv_tma_on():
        others.append(staged)
    else:
        main = staged
    main.update({"peak_source": pk["src"] + " bf16 burst (fp16 runs at the bf16 rate)", "operands": fmt, "others": others})
    return main


def attn_metric(dev, pk):
    """AttnBlock (modules.py:139-191) at the model's shape: batch 32, C = 512, 16x16 tokens; forward and backward of the
    whole block (GroupNorm, q/k/v and proj_out 1x1 GEMMs on TF32 tcgen05, the fused QK^T -> softmax -> PV core, the four
    gradients of the two contractions on the 3xTF32 tcgen05 GEMM, residual, next-norm statistics). Algorithmic FLOPs per image forward: 0.671 GFLOP
    (SURVEY.md 8d), backward = 2x; the 3xTF32 passes are not counted."""
    from models import modules as M
    torch.manual_seed(0)
    blk = M.AttnBlock(512).to(dev)
    x = torch.randn(BATCH, 512, 16, 16, device=dev).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    g = torch.randn(BATCH, 512, 16, 16, device=dev).contiguous(memory_format=torch.channels_last)
    fwd = time_kernel(lambda: blk(x), iters=10, warm=3)

    def both():
        y = blk(x)
        y.backward(g)
    tot = time_kernel(both, iters=10, warm=3)
    gf = 0.671 * BATCH
    return {"shape": "batch 32, 256 tokens, C=512", "fwd_ms": round(fwd * 1e3, 4), "fwd_bwd_ms": round(tot * 1e3, 4),
            "fwd_tflop_per_s": round(gf / fwd / 1e3, 1), "fwd_bwd_tflop_per_s": round(3 * gf / tot / 1e3, 1),
            "frac_of_tf32_peak_fwd": round(gf / fwd / 1e3 / (pk["bf16"] / 2), 3), "bound": "tensor (nominal); launch / latency bound at this size",
            "kernels": "gn_apply, shift_gemm_tc<1> (QKV, proj; TF32), attn_core_fwd (fused QK^T -> softmax -> PV, 2 x fp16 split); "
                       "backward: gemm3_tc (3xTF32) x4, softmax_bwd, wgrad_tc<1>, shift_gemm_tc<1>"}


def ffma_peak(dev):
    """fp32 FMA-pipe peak measured live (mas_ffma_probe, CUDA events): the roofline of the exact-fp32 VQ distance kernel."""
    import ctypes
    from mas_b200 import _lib as L
    scratch = torch.empty(148 * 4 * 512, device=dev)
    fl = ctypes.c_double(0.0)
    fn = lambda: L.call("mas_ffma_probe", scratch, 2048, ctypes.cast(ctypes.pointer(fl), ctypes.c_void_p))
    sec = time_kernel(fn, iters=5, warm=2)
    return fl.value / sec / 1e12


def vq_metric(dev, pk, sweep=True):
    """VQ argmin standalone (BASELINE configs[2]): 16x16x256 latents against the 8192-entry codebook, batch sweep
    1..4096 (R = 256*B rows), through the product call (mas_vq_forward: tensor-core filter + exact re-evaluation, indices
    bit-identical to the all-pairs kernel). Per point: algorithmic bytes (2056*R + 8,388,608) / time and the algorithmic
    4,194,304*R FLOP / time, as a fraction of (a) the live-measured fp32 FFMA peak - the roofline of an exact-fp32
    all-pairs evaluation, which the filter beats by doing the bulk of the work on the tensor cores - and (b) the tensor
    peak counting the three fp16 MMAs per K step the filter issues. The all-pairs FFMA kernel is timed beside it."""
    from mas_b200 import ops
    E = torch.randn(N_EMBED, 256, generator=torch.Generator().manual_seed(4321)).to(dev)
    peak = ffma_peak(dev)
    g = torch.Generator(device=dev).manual_seed(1234)

    def run(batches, tc):
        ops.vq_select_path(tc)
        pts = []
        try:
            for B in batches:
                z = torch.randn(B, 256, 16, 16, generator=g, device=dev).contiguous(memory_format=torch.channels_last)
                it = 10 if B <= 256 else (4 if B <= 1024 else 2)
                sec = time_kernel(lambda: ops.VQFn.apply(z, E, 0.25), iters=it, warm=2)
                R = B * 256
                byts = 2056.0 * R + 8388608.0
                tf = 4194304.0 * R / sec / 1e12
                pts.append({"batch": B, "rows": R, "ms": round(sec * 1e3, 4), "gb_per_s": round(byts / sec / 1e9, 2),
                            "tflop_per_s": round(tf, 2), "ffma_frac": round(tf / peak, 3),
                            "tensor_frac_3pass": round(3 * tf / pk["bf16"], 3) if tc else None,
                            "hbm_frac": round(byts / sec / 1e9 / pk["hbm"], 4)})
                del z
        finally:
            ops.vq_select_path(True)
        return pts
    batches = [1, 2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096] if sweep else [BATCH]
    pts = run(batches, True)
    exact = run([BATCH] + ([1024] if sweep else []), False)
    at32 = next(p for p in pts if p["batch"] == BATCH)
    return {"rows": at32["rows"], "ms": at32["ms"], "gb_per_s": at32["gb_per_s"], "tflop_per_s": at32["tflop_per_s"],
            "hbm_frac": at32["hbm_frac"], "ffma_frac": at32["ffma_frac"], "tensor_frac_3pass": at32["tensor_frac_3pass"],
            "ffma_peak_tflops_measured": round(peak, 2),
            "kernel": "vq_filter_tc (tcgen05 kind::f16, 2 x fp16 operand split) + vq_resolve (exact fp32 re-evaluation)",
            "bound": "tensor pipe for the filter (3 MMAs per K step); an exact all-pairs evaluation is bound by the fp32 FFMA pipe",
            "all_pairs_ffma_kernel": exact, "sweep": pts}


def transformer_kernel_rooflines(dev, pk, batch=8):
    """The three tensor-core kernels of the transformer step, timed live at the model's shapes (CUDA events) against the measured
    bf16 peak (fp16 MMAs run at the bf16 rate): algorithmic FLOPs only (the hi/lo operand split of the attention core and its
    second score pass are not counted)."""
    from mas_b200 import ops
    M, K, N, S, heads = batch * 640, 1024, 4096, 640, 16
    g = torch.Generator().manual_seed(7)
    x = torch.randn(M, K, generator=g).to(dev)
    dy = (torch.randn(M, N, generator=g) * 1e-4).to(dev)
    w = torch.nn.Parameter((torch.randn(N, K, generator=g) * 0.02).to(dev))
    b = torch.zeros(N, device=dev)
    x16, ax = ops.rows_to_half(x)
    dy16, ad = ops.rows_to_half(dy)
    qkv = torch.randn(batch, S, 3 * heads * 64, generator=g).to(dev)
    out = []

    def entry(name, fn, flop, note):
        sec = time_kernel(fn, iters=10, warm=3)
        out.append({"kernel": name, "ms": round(sec * 1e3, 4), "tflop_per_s": round(flop / sec / 1e12, 1),
                    "frac_of_bf16_peak": round(flop / sec / 1e12 / pk["bf16"], 3), "shape": note})
    entry("rows_gemm_t16 (Linear forward, TMA-fed fp16)", lambda: ops.gemm_rows_f16(x16, ax, w, False, b), 2.0 * M * N * K,
          "x [%d,%d] . W[%d,%d]^T + b" % (M, K, N, K))
    entry("rows_gemm_t16 (Linear data gradient)", lambda: ops.gemm_rows_f16(dy16, ad, w, True), 2.0 * M * N * K, "dy [%d,%d] . W" % (M, N))
    entry("rows_wgrad_t16 + reduction (Linear weight gradient)", lambda: ops.wgrad_rows_f16(x16, ax, dy16, ad), 2.0 * M * N * K,
          "dy^T [%d,%d] . x [%d,%d]" % (N, M, M, K))
    blocks = sum(qt + 1 for qt in range(S // 128))
    entry("attn_causal_fwd + amax (fused causal attention core)", lambda: ops.CausalAttentionFn.apply(qkv, heads),
          batch * heads * blocks * 2 * 2.0 * 128 * 128 * 64, "batch %d, %d tokens, %d heads of 64, causal key blocks only" % (batch, S, heads))
    return out


def transformer_metric(dev, pk, batch=8, steps=3, warmup=2):
    """Tier-2 row (SURVEY.md 8f-2): training-step throughput of the token transformer at BASELINE configs[4]'s model (24 layers,
    1024 wide, 16 heads of 64, 128 text + 256 segmentation + 256 image tokens; random weights, synthetic tokens): forward +
    cross-entropy over the image tokens + backward (train.py:136-153, no optimizer), CUDA-event timed. Same code as
    tools/bench_transformer.py. Reported beside the headline, not part of it."""
    from mas_b200 import _lib
    from models.transformer import MakeAScene
    cfg = dict(num_layers=24, hidden_dim=1024, num_attn_heads=16, image_vocab_size=8192, seg_vocab_size=1024, text_vocab_size=49408,
               image_tokens_per_dim=16, seg_tokens_per_dim=16, text_length=128)
    torch.manual_seed(0)
    m = MakeAScene(**cfg).to(dev).train()
    m.device = dev
    g = torch.Generator().manual_seed(1234)
    text = torch.randint(1, 40000, (batch, 128), generator=g).to(dev)
    seg = torch.randint(0, 1024, (batch, 256), generator=g).to(dev)
    img = torch.randint(0, 8192, (batch, 256), generator=g).to(dev)

    def step():
        m.zero_grad(set_to_none=True)
        loss = m.loss(text, seg, img)
        loss.backward()
        return loss
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0, t0 = _lib.launch_count(), _lib.tc_launch_count()
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) * 1e-3 / steps
    S, H, Ly, V = 640, 1024, 24, 8192
    flops = 3 * (2 * S * (12 * H * H) * Ly + 2 * 256 * H * V + 2 * 2 * S * S * H * Ly) * batch
    try:
        roofs = transformer_kernel_rooflines(dev, pk, batch)
    except Exception as e:  # noqa: BLE001
        roofs = {"error": str(e)[:200]}
    return {"metric": "token transformer training step (fwd + cross-entropy + bwd), sequence tokens/s", "value": round(batch * S / sec, 1),
            "unit": "tokens/s", "batch": batch, "seq_len": S, "ms_per_step": round(sec * 1e3, 3), "loss": round(float(loss.detach()), 5),
            "model_tflops": round(flops / sec / 1e12, 1), "gpu_launches_per_step": (_lib.launch_count() - l0) // steps,
            "tcgen05_launches_per_step": (_lib.tc_launch_count() - t0) // steps,
            "kernels": "rows_gemm_t16 / rows_wgrad_t16 (TMA-fed fp16 Linear layers), attn_causal_fwd (fused causal attention core), "
                       "gemm3_tc (3xTF32 attention gradients, causal block skipping), mas_ce_* (fused cross-entropy)",
            "kernel_rooflines": roofs}


DUMP_MAX_ELEMS = 8 << 20       # per output array: a larger one is written as a fixed, seeded sample of this many elements
GRAD_SAMPLE = 4096             # elements sampled from each parameter gradient larger than this


def _seeded_sample(t, k, seed):
    """`k` elements of `t` (flattened) at indices drawn from a fixed seed, in ascending order; all of `t` if it is smaller."""
    t = t.detach().reshape(-1)
    if t.numel() <= k:
        return t
    idx = torch.randint(0, t.numel(), (k,), generator=torch.Generator().manual_seed(seed)).sort().values
    return t[idx.to(t.device)]


def dump_outputs(out_dir, model, last):
    """Writes what the last timed step returned to its caller, as float32 / float64 .npy files under `out_dir`: the
    reconstruction `dec` (whole, or `dec_sample` when larger than DUMP_MAX_ELEMS), the codebook term `diff`, the `loss`,
    `grad_norms` (float64 L2 norm of every parameter gradient, model.named_parameters() order) and `grad_sample` (per
    parameter in that order, up to GRAD_SAMPLE gradient elements at seeded indices, concatenated). On a B200, two runs of
    one build give bit-identical dec / diff / loss; the weight gradients differ in the last bits (reduction order), so
    compare them with a tolerance."""
    import numpy as np
    dec = last["dec"].detach()
    dec_name, dec = ("dec", dec) if dec.numel() <= DUMP_MAX_ELEMS else ("dec_sample", _seeded_sample(dec, DUMP_MAX_ELEMS, 0))
    arrays = {dec_name: dec.float(), "diff": last["diff"].detach().float(), "loss": last["loss"].detach().float()}
    named = [(k, p.grad) for k, p in model.named_parameters()]
    missing = [k for k, g in named if g is None]
    assert not missing, "parameters without a gradient after the timed step: %s" % missing[:5]
    arrays["grad_norms"] = torch.stack([g.detach().double().norm() for _, g in named])
    arrays["grad_sample"] = torch.cat([_seeded_sample(g, GRAD_SAMPLE, i).float() for i, (_, g) in enumerate(named)])
    arrays = {k: t.contiguous().cpu().numpy() for k, t in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, "dumped outputs exceed 64 MB (%d bytes)" % total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return sorted(arrays)


def _fmt():
    from mas_b200 import ops
    return "fp16 (3x3 convolutions) / tf32 (1x1)" if ops.get_operand_format() == "f16" else "tf32"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="vqimg", choices=["vqimg", "vqseg"],
                    help="vqimg: BASELINE configs[1] (the headline metric); vqseg: configs[3], 159-channel maps + weighted BCE")
    ap.add_argument("--profile", action="store_true", help="print per-entry-point CUDA-event times of one extra step")
    ap.add_argument("--step-only", action="store_true",
                    help="skip the per-kernel blocks (roofline / VQ sweep / AttnBlock / CPU baseline): launch-list captures under ncu")
    ap.add_argument("--graph", action="store_true",
                    help="single GPU: replay the step from one CUDA graph (mas_b200.graph.GraphedStep) instead of launching from Python")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last timed step's outputs and gradients as .npy files to DIR (rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch.distributed as dist
    from mas_b200 import _lib
    assert torch.cuda.is_available(), "bench.py (impl ours) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    pk = peaks()
    seg = args.workload == "vqseg"
    model = build_model(args.workload).to(dev)
    net = model
    if world > 1:
        net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], gradient_as_bucket_view=True)
    B = args.batch
    gen = torch.Generator().manual_seed(1234 + rank)
    if seg:   # one-hot-like label maps (SURVEY.md 8d plumbing config, here at BASELINE configs[3]'s size)
        img_host = (torch.rand(B, 159, RES, RES, generator=gen) > 0.9).float().pin_memory()
        pos_w = torch.ones(159, device=dev)
        pos_w[153:158] = 20
    else:
        img_host = torch.rand(B, 3, RES, RES, generator=gen).pin_memory()
    img_dev = img_host.to(dev)
    last = {}       # the outputs of the latest step, kept only for --dump-outputs

    def step(img):
        net.zero_grad(set_to_none=True)
        dec, diff = net(img)
        if seg:
            from mas_b200 import ops
            loss = ops.BCELogitsFn.apply(dec, img, pos_w) + diff     # losses/loss_seg.py:15-22
        else:
            loss = (img - dec).abs().mean() + diff
        loss.backward()
        if args.dump_outputs:
            last.update(dec=dec, diff=diff, loss=loss)
        return loss

    def timed(fn, warmup, steps):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        st = torch.cuda.current_stream()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        e0.record(st)
        for _ in range(steps):
            fn()
        e1.record(st)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) * 1e-3, _lib.launch_count() - l0

    # --graph (single GPU): the step is captured once into a CUDA graph (mas_b200.graph.GraphedStep) and replayed.  Measured
    # on B200 at batch 32 it is within run-to-run noise of eager launching (the GPU is never starved: ~110 ms of kernels per
    # step against ~45 ms of host launch work), so the default stays eager, which is also what the DDP runs (N > 1) use.
    gs, graph_note = None, "eager (every kernel launched from Python through the C-ABI)"
    if world == 1 and args.graph:
        from mas_b200.graph import GraphedStep

        def loss_fn(m, x):
            dec, diff = m(x)
            if args.dump_outputs:     # during capture: these become the graph's static output buffers
                last.update(dec=dec, diff=diff)
            if seg:
                from mas_b200 import ops
                return ops.BCELogitsFn.apply(dec, x, pos_w) + diff
            return (x - dec).abs().mean() + diff
        try:
            gs = GraphedStep(net, loss_fn, img_dev, warmup=2)
            graph_note = "whole step (fwd+loss+bwd) replayed from one CUDA graph, %d kernels of this library per step" % gs.launches_per_step
        except Exception as e:  # noqa: BLE001 - report and measure the eager path instead
            gs, graph_note = None, "eager (capture failed: %s)" % str(e)[:120]
            net.zero_grad(set_to_none=True)
    run_dev = (lambda: gs(img_dev)) if gs is not None else (lambda: step(img_dev))
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    sec, launches = timed(run_dev, args.warmup, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if gs is not None:
        launches = gs.launches_per_step * args.steps
        last["loss"] = gs.loss
    if args.dump_outputs and rank == 0:
        print("outputs of the last timed step written to %s: %s" % (args.dump_outputs, ", ".join(dump_outputs(args.dump_outputs, model, last))),
              file=sys.stderr)

    def e2e_step():
        if gs is not None:
            return float(gs(img_host).item())     # pinned host batch -> static device input (H2D), replay, loss back (D2H)
        img = img_host.to(dev, non_blocking=True)
        return float(step(img).item())
    sec_e2e, _ = timed(e2e_step, max(1, args.warmup // 2), args.steps)
    if gs is not None:
        gs.close()
    value = world * B * args.steps / sec
    e2e = world * B * args.steps / sec_e2e
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.profile:
        _lib.profile_start()
        step(img_dev)
        rep = _lib.profile_report()
        tot = sum(t for _, t in rep.values())
        print("per-entry profile of one step (CUDA events, ms):", file=sys.stderr)
        for k, (c, t) in sorted(rep.items(), key=lambda kv: -kv[1][1]):
            print("  %-44s n=%4d  %9.2f ms  %5.1f%%  %7.3f ms/call" % (k, c, t, 100 * t / tot, t / c), file=sys.stderr)
        print("  total %.2f ms" % tot, file=sys.stderr)
    if args.step_only:
        print(json.dumps({"metric": METRIC, "value": value, "ms_per_step": sec / args.steps * 1e3, "gpu_launches": int(launches),
                          "step_only": True}), flush=True)
        return
    roof = dominant_kernel_roofline(dev, pk)
    if seg:
        line = {"metric": SEG_METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": sec / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "%s tcgen05 operands, fp32 accumulate / storage" % _fmt(), "data": "synthetic",
                "config": {"workload": "VQ-SEG 256x256, 159-channel maps, codebook=1024 dim=256, batch %d/GPU (BASELINE configs[3])" % B,
                           "global_batch": B * world, "parallelism": "dp%d" % world, "launch": graph_note,
                           "loss": "weighted BCE-with-logits (pos_weight 20 on channels 153-157) + codebook loss, kernels mas_bce_cl_*",
                           "edge_layers": "159-channel conv_in / conv_out zero-padded to 160 / 2x128 channels on the fp16 tcgen05 kernels"},
                "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": B * 159 * RES * RES * 4, "d2h_bytes_per_step": 4,
                        "ms_per_step": sec_e2e / args.steps * 1e3},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roof}
        print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    vq = vq_metric(dev, pk)
    attn = attn_metric(dev, pk)
    line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": sec / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "%s tcgen05 operands (11-bit significand), fp32 accumulate / storage; 3xTF32 for the attention contractions; fp32 FFMA for VQ argmin and edge layers" % _fmt(),
            "data": "synthetic",
            "config": {"workload": "VQ-IMG 256x256 codebook=8192 dim=256 batch %d/GPU (BASELINE configs[1])" % B,
                       "global_batch": B * world, "parallelism": "dp%d" % world, "launch": graph_note,
                       "l2": "per-step working set >> 126 MB L2 (one 128x256x256 activation at batch 32 is 1.07 GB); no explicit flush",
                       "optimizer": "excluded (metric is enc+VQ+dec fwd+bwd, BASELINE.md section 3)"},
            "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": B * 3 * RES * RES * 4, "d2h_bytes_per_step": 4,
                    "ms_per_step": sec_e2e / args.steps * 1e3},
            "gpu_launches": int(launches), "clocks": clocks,
            "model_tflops": FLOP_PER_IMG_FWD_BWD * value / 1e12, "roofline": roof, "vq": vq, "attn": attn}
    if world == 1:   # tier-2 row, beside the headline (never fails the bench line)
        try:
            torch.cuda.empty_cache()
            line["transformer"] = transformer_metric(dev, pk)
        except Exception as e:  # noqa: BLE001
            line["transformer"] = {"error": str(e)[:200]}
    if not args.no_cpu_baseline and world == 1:   # reported baseline: rank 0 at N=1 only
        r = cpu_reference_steps(3, 1, batch=2, budget=float(os.environ.get("MAS_CPU_ARM_SECONDS", "60")))
        line["cpu_baseline"] = {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": r["kind"],
                                "sample": "%d timed fwd+bwd steps of %d images after 1 warm-up (%.1f s/step)" % (r["done"], r["batch"], r["sec"])}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
