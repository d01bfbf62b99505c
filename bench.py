#!/usr/bin/env python
"""Benchmark of the ODISE inference hot path on B200 (contract: see the task brief / DESIGN.md §5).

    python bench.py --gpus N --steps K --warmup W                 # our arm (one rank per GPU under torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path (oracle), rank 0 only
    python bench.py --config c3|c4|c5 ...                          # the other BASELINE.json configs (c2 = default)
    python bench.py ... --dump-outputs DIR                         # + what the last timed step returned, as DIR/*.npy

A step = one pass of the per-image pipeline over a batch of synthetic images: CLIP ViT-L/14-336 image tower on every
512^2 crop + KL-VAE encoder / truncated decoder taps [unless --hot-path-only] -> implicit captioner -> UNet feature
pass on all crops -> 8 projections -> pixel decoder -> masked-attention decoder -> CLIP-text scoring -> MaskCLIP
ensemble -> semantic + panoptic + instance inference at the input resolution (odise.py:326-370; the metric says
"panoptic inference").  `value` times the CUDA-graph replay with inputs resident in HBM; `e2e` times the public call
ODISEEngine.infer(outputs="panoptic") with pinned-host uint8 images in and the panoptic map + segment table + instance
table + class logits out.

BASELINE.json configs:  c2 (default) 1xB200, batch 4 x 1024^2, ADE-150 | c3 image-sharded 8xB200, COCO-133 |
c4 MSDeformAttn + masked-attention decoder microbench (256 queries x 4 scales, HBM GB/s) | c5 ADE-847 (1342 prompts) at
1280^2 (9 overlapping crops per image), reporting the mask-embed x text GEMM TFLOP/s.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec @1024x1024 panoptic inference (ODISE hot path)"
UNET_TFLOP_PER_CROP = 0.740          # minimal feature pass, SURVEY.md §8d / BASELINE.md §2
VOCABS = {"ade150": (150, 403), "coco133": (133, 254), "ade847": (847, 1342)}
CONFIGS = {          # BASELINE.json `configs` (configs[0] is the CPU numerics case: tests, not a bench line)
    "c2": dict(size=1024, vocab="ade150", batch=4),
    "c3": dict(size=1024, vocab="coco133", batch=4),
    "c5": dict(size=1280, vocab="ade847", batch=4),
    "c4": dict(size=1024, vocab="ade150", batch=4),
}


NMMA = {"f16q8": 2, "bf16x3": 3, "bf16": 1}      # odise_gemm_desc.nmma of the operand mode


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=None, help="images per GPU per step (default: the config's)")
    ap.add_argument("--size", type=int, default=None)
    ap.add_argument("--precision", default="f16q8", choices=["f16q8", "bf16x3", "bf16"],
                    help="bf16x3: (hi, lo) bf16 pairs, 3 MMAs per k-step (2e-5 at the UNet taps).  f16q8: fp16 hi x hi + both "
                         "cross terms on e5m2 MMAs at twice the rate = 2 MMA units per k-step (1e-4 at the taps, bar 1e-3); "
                         "VAE / CLIP / UNet / projections run it, the head and the post-processing stay bf16x3.  bf16: plain "
                         "(not a parity mode)")
    ap.add_argument("--vocab", default=None, choices=sorted(VOCABS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32 / "
                         "float64, at most 64 MB in all): what ODISEEngine.infer() returned (c2 / c3 / c5), the MSDeformAttn "
                         "and decoder outputs (c4), the CPU path's logits and inference maps (--impl reference); so that "
                         "two builds can be compared output for output")
    ap.add_argument("--hot-path-only", action="store_true",
                    help="skip the KL-VAE (SURVEY.md 8f-1) and CLIP image tower (8f-2) stages: their taps / latent / "
                         "image embedding enter as synthetic tensors")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    c = CONFIGS[a.config]
    a.batch = a.batch or c["batch"]
    a.size = a.size or c["size"]
    a.vocab = a.vocab or c["vocab"]
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_burst=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    hbm=d["hbm_gbs"], source="measured")
    return dict(bf16_burst=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback")


NPY_HEADER = 256                     # bytes an .npy header takes at most for the shapes written here


def dump_outputs(arrays, out_dir, budget=64_000_000):
    """Writes each array as out_dir/<name>.npy: float64 stays float64, other floating types and integers that float32
    holds exactly become float32, larger integers float64.  The files, headers included, take at most `budget` bytes:
    it is shared out smallest array first, and an array over its share is replaced by a fixed, seeded sample of its
    flattened elements (the same indices on every run)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    conv = {}
    for name, v in arrays.items():
        v = v.detach().cpu()
        if v.dtype == torch.bool:
            v = v.to(torch.int32)
        wide = v.dtype == torch.float64 or (not v.is_floating_point() and v.numel() > 0 and int(v.abs().max()) >= 2 ** 24)
        conv[name] = v.to(torch.float64 if wide else torch.float32)
    left = budget - NPY_HEADER * len(conv)
    for i, (name, v) in enumerate(sorted(conv.items(), key=lambda kv: kv[1].numel() * kv[1].element_size())):
        share = left // (len(conv) - i)
        if v.numel() * v.element_size() > share:
            g = torch.Generator().manual_seed(0)
            v = v.flatten()[torch.randperm(v.numel(), generator=g)[:share // v.element_size()].sort().values]
        left -= v.numel() * v.element_size()
        np.save(os.path.join(out_dir, name + ".npy"), v.numpy())


def n_crops(size):
    from odise_b200.backbone import BackboneEngine
    return len(BackboneEngine.crop_grid(size, size)[0])       # feature_extractor.py:197-218 (1280 -> 3 x 3 overlapping)


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i] == "Active" for r in self.rows)]
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(sm))


# ----------------------------------------------------------------------------------------------- CPU baseline
class CpuHotPath:
    """The reference's CPU path through the oracle (oracle/ldm.py restatement driven like LdmExtractor.unet_forward;
    oracle/m2f.py == the reference's own Mask2Former/ODISE code, pinned in tests/test_oracle_cpu.py), fp32.
    Bounded sample: ONE 512^2 crop through the per-crop stages + ONE image through the head at size^2 (pixel
    decoder + decoder + scoring + MaskCLIP + post-processing); images/s = 1 / (crops * t_crop + t_head)."""

    def __init__(self, size, vocab, threads=None, full=True):
        from odise_b200 import spec
        from odise_b200.pipeline import synthetic_vocabulary
        from oracle import ldm, m2f
        self.ldm, self.m2f = ldm, m2f
        # torch CPU ops stop scaling (and regress) far below the 100+ threads of the GPU hosts: cap at 32
        self.n = threads or min(os.cpu_count(), 32)
        torch.set_num_threads(self.n)
        sd_u = spec.synth_state_dict(spec.unet_params(), 0)
        with torch.device("meta"):
            unet = ldm.UNetModel()
        unet.load_state_dict({k[len(spec.UNET_PREFIX):]: v for k, v in sd_u.items()}, assign=True)
        self.unet = unet.eval()
        self.sd_h = spec.synth_state_dict(spec.head_params(), 1)
        g = torch.Generator().manual_seed(3)
        self.x, self.ctx = torch.randn(1, 4, 64, 64, generator=g), torch.randn(1, 77, 768, generator=g)
        self.cond = torch.randn(1, 1280, generator=g)
        self.feats = {f"s{i}": torch.randn(1, 512, size // 2 ** i, size // 2 ** i, generator=g) for i in (2, 3, 4, 5)}
        self.bank, self.null, self.sizes = synthetic_vocabulary(*VOCABS[vocab])
        self.ncls = VOCABS[vocab][0]
        self.size = size
        self.crops = n_crops(size)
        self.full = full
        if full:
            sd_v = spec.synth_state_dict(spec.vae_params(), 3)
            with torch.device("meta"):
                vae = ldm.AutoencoderKL()
            vae.load_state_dict({k[len(spec.VAE_PREFIX):]: v for k, v in sd_v.items()}, assign=True)
            self.vae = vae.eval()
            self.img = torch.rand(1, 3, 512, 512, generator=g) * 2 - 1
            from oracle import clip as oclip
            self.oclip = oclip
            sd_c = spec.synth_state_dict(spec.clip_visual_params(), 5)
            with torch.device("meta"):
                vis = oclip.VisionTransformer()
            vis.load_state_dict({k[len(spec.CLIP_PREFIX):]: v for k, v in sd_c.items()}, assign=True)
            self.vis = vis.eval()
            self.img_full = torch.rand(1, 3, size, size, generator=g)
            self.ov = torch.tensor([(k % 2) == 0 for k in range(VOCABS[vocab][0])]).long()

    @torch.no_grad()
    def sample(self):
        ldm, m2f = self.ldm, self.m2f
        from oracle import postprocess as opp
        t0 = time.perf_counter()
        # as the reference executes it: output block 11 + unet.out run too, and the VAE decoder runs to the full image
        ldm.unet_features(self.unet, self.x, self.ctx, self.cond, stop_early=False)
        if self.full:
            lat, _ = ldm.encoder_features(self.vae, self.img)
            ldm.decoder_features(self.vae, lat, truncate=False)
            self.oclip.embed_image(self.vis, self.img * 0.5 + 0.5)
        t_unet = time.perf_counter() - t0
        t0 = time.perf_counter()
        mf, _, ms = m2f.pixel_decoder(self.sd_h, self.feats, "sem_seg_head.pixel_decoder.")
        out, _ = m2f.transformer_decoder(self.sd_h, ms, mf, "sem_seg_head.predictor.")
        te, ne = m2f.category_embed(self.sd_h, self.bank, self.null)
        lg = m2f.cal_pred_logits(out["mask_embed"], te, ne, out["logit_scale"], self.sizes)
        if self.full:                 # clip_head branch (odise.py:292-323): MaskCLIP over the whole image + ensemble
            oc = self.oclip
            me = oc.get_mask_embed(self.vis, self.img_full, out["pred_masks"])
            cl = oc.maskclip_pred_logits(me, self.bank, self.sizes, 100.0)
            lg = oc.merge_with_void(lg, oc.pooling_clip_ensemble(lg[..., :-1], cl, self.ov, 0.3, 0.7))
        # odise.py:326-370: upsample to the input size, semantic + panoptic inference (instance inference is a top-k
        # over the same tensors; not timed on the CPU side)
        up = opp.upsample_masks(out["pred_masks"], (self.size, self.size))[0]
        sem = opp.semantic_inference(lg[0], up)
        pan, segs = opp.panoptic_inference(lg[0], up, self.ncls, list(range(0, self.ncls, 2)))
        t_head = time.perf_counter() - t0
        self.last = dict(pred_logits=lg[0], sem_seg=sem, panoptic_seg=pan, segments_info=torch.tensor(
            [[s["id"], int(s["isthing"]), s["category_id"]] for s in segs], dtype=torch.int64).view(-1, 3))
        ips = 1.0 / (self.crops * t_unet + t_head)
        return dict(value=ips, unit="images/s", cores=self.n, kind="port",
                    sample=f"1 crop (512^2) through {'CLIP ViT-L/14 image tower + VAE enc + UNet + full VAE dec' if self.full else 'the UNet'} as the "
                           f"reference executes it ({t_unet:.2f} s) + 1 image head{' + MaskCLIP' if self.full else ''} + semantic/panoptic "
                           f"inference at {self.size}^2 ({t_head:.2f} s); images/s = 1/({self.crops}*t_crop + t_head); fp32 torch CPU, "
                           f"{self.n} threads of {os.cpu_count()}")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.config == "c4":
        print(json.dumps({"impl": "reference", "unavailable": "c4 is a GPU kernel microbench: its baseline (the reference's "
                          "own CUDA kernel, oracle/_ref) is reported inside the c4 line of the `ours` arm"}), flush=True)
        return
    cpu = CpuHotPath(args.size, args.vocab, full=args.full)
    for _ in range(args.warmup):
        cpu.sample()
    vals, info = [], None
    for _ in range(args.steps):
        info = cpu.sample()
        vals.append(info["value"])
    if args.dump_outputs:
        dump_outputs(cpu.last, args.dump_outputs)
    v = statistics.mean(vals)
    info["value"] = v
    ncls, npr = VOCABS[args.vocab]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / v, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"ODISE hot path, {args.size}x{args.size}, {args.vocab} ({npr} prompts), CPU oracle",
                   "baseline_config": args.config,
                   "note": "reference arm = CPU restatement (reference not installable: detectron2/ldm/open_clip absent)"},
        "cpu_baseline": info,
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


# ----------------------------------------------------------------------------------------------- c4 microbench
def _time_ms(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(True), torch.cuda.Event(True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def run_c4(args, dev):
    """BASELINE.json configs[3]: MSDeformAttn sampling + masked-attention decoder, 256 queries x 4 scales, HBM GB/s.
    (a) the deformable-attention op on the 4-level pyramid of a 1024^2 input (strides 8..64), N = batch images, once with
    every pixel a query (pixel-decoder encoder, Lq = S) and once with 256 queries; ours (reference ABI and fused-front
    variants) next to the REFERENCE's own CUDA kernel compiled for sm_100a (oracle/_ref);
    (b) the 9-layer masked-attention decoder + 10 prediction heads with 256 queries cycling over 4 scales."""
    from odise_b200 import lib, ops, spec
    from odise_b200.head import HeadEngine
    pk = peaks()
    N, M, D, P = args.batch, 8, 32, 4
    shapes = [(args.size // s, args.size // s) for s in (64, 32, 16, 8)]           # coarse -> fine, like the pixel decoder
    L = len(shapes)
    S = sum(h * w for h, w in shapes)
    g = torch.Generator().manual_seed(4)
    ss = torch.as_tensor(shapes, dtype=torch.int64)
    lsi = torch.cat((ss.new_zeros(1), ss.prod(1).cumsum(0)[:-1]))
    value = torch.randn(N, S, M, D, generator=g).to(dev)
    res, dumps = {}, {}
    reps, warm = args.steps, args.warmup
    for name, Lq in (("encoder_Lq=S", S), ("queries_Lq=256", 256)):
        ref_pts = torch.rand(N, Lq, L, 2, generator=g)
        offs = torch.randn(N, Lq, M, L, P, 2, generator=g) * 2.0
        logits = torch.randn(N, Lq, M, L * P, generator=g)
        norm = torch.stack([ss[:, 1], ss[:, 0]], -1).float()
        loc = (ref_pts[:, :, None, :, None, :] + offs / norm[None, None, None, :, None, :]).contiguous().to(dev)
        aw = logits.softmax(-1).view(N, Lq, M, L, P).contiguous().to(dev)
        dss, dls = ss.to(dev), lsi.to(dev)
        dref, doffs, dlog = ref_pts.to(dev), offs.to(dev), logits.to(dev)
        out = torch.empty(N, Lq, M * D, device=dev)
        L_ = lib.load()

        def ours_abi():
            lib._check(L_.odise_msda_forward_f32(value.data_ptr(), dss.data_ptr(), dls.data_ptr(), loc.data_ptr(),
                                                 aw.data_ptr(), out.data_ptr(), N, S, M, D, L, Lq, P, lib._stream()), "msda")

        def ours_fused():
            ops.msda_fused(value, dss, dls, dref, doffs, dlog, N, S, M, D, L, Lq, P, want_f32=False)

        t_abi = _time_ms(ours_abi, reps, warm)
        dumps["msda_" + name.split("_")[0]] = out.clone()          # what the last timed odise_msda_forward_f32 wrote
        t_fused = _time_ms(ours_fused, reps, warm)
        # what the gathers move through L1: 4 corners x 128 B per (query, head, sample)
        l1_bytes = 128.0 * 4 * N * Lq * M * L * P
        # compulsory bytes (SURVEY.md §8d): value once (at most what the samples can touch) + loc / attn (3 floats per
        # sample) + output, fp32
        nbytes = min(4.0 * N * S * M * D, l1_bytes) + 4.0 * N * (Lq * M * L * P * 3 + Lq * M * D)
        r = dict(Lq=Lq, compulsory_mb=nbytes / 1e6, ours_abi_us=1e3 * t_abi, ours_fused_us=1e3 * t_fused,
                 ours_abi_gbs=nbytes / t_abi / 1e6, ours_fused_gbs=nbytes / t_fused / 1e6,
                 frac_of_hbm_peak=nbytes / t_abi / 1e6 / pk["hbm"], gather_l1_tbs=l1_bytes / t_abi / 1e9)
        try:
            from oracle import refmsda
            if refmsda.available():
                ro = torch.empty_like(out)
                t_ref = _time_ms(lambda: refmsda.forward(value, dss, dls, loc, aw, 128, out=ro), reps, warm)
                ours_abi()
                torch.cuda.synchronize()
                r.update(reference_kernel_us=1e3 * t_ref, reference_kernel_gbs=nbytes / t_ref / 1e6,
                         speedup_vs_reference_kernel=t_ref / t_abi, max_abs_diff_vs_reference=float((out - ro).abs().max()))
            else:
                r["reference_kernel_us"] = None
        except Exception as ex:  # noqa
            r["reference_kernel_error"] = str(ex)
        res[name] = r
    # (b) masked-attention decoder, Q = 256, 4 scales
    Q = 256
    sd = spec.synth_state_dict(spec.pixel_decoder_params() + spec.decoder_params(Q=Q, n_levels=L) + spec.category_head_params(), 1)
    he = HeadEngine(sd, dev, nmma=NMMA[args.precision], num_queries=Q)
    ms = [torch.randn(N, 256, h, w, generator=g).to(dev) for h, w in shapes]
    mfeat = torch.randn(N, 256, args.size // 4, args.size // 4, generator=g).to(dev)
    pd = he.pd_from_tensors(ms, mfeat)
    c0 = lib.launch_count()
    he.transformer_decoder(pd, N)
    launches = lib.launch_count() - c0
    last = {}

    def dec_step():
        last["heads"] = he.transformer_decoder(pd, N)

    t_dec = _time_ms(dec_step, reps, warm)
    dumps.update({"decoder_" + k: v for k, v in last["heads"][-1].items()})      # the last prediction head
    HW = (args.size // 4) ** 2
    plane = 4.0                                     # bytes per element of a (hi, lo) bf16 operand pair
    # K and V^T planes (head-padded 8 x 64 columns) of every layer, read once by its cross-attention
    kv = sum(N * h * w * 512 * plane * 2 * len([i for i in range(9) if i % L == lv]) for lv, (h, w) in enumerate(shapes))
    heads = 10 * N * (Q * HW * 4.0            # mask logits written
                      + Q * HW * 4.0            # ... read back for the 0/1 mask + counts
                      + 2 * HW * 256 * plane)   # mask features: B operand of the mask einsum + of the pooling
    bits = 9 * N * Q * HW * 4.0                 # mask logits read again for the attention bits of the next layer
    dec_bytes = kv + heads + bits
    res["masked_attention_decoder"] = dict(queries=Q, scales=L, layers=9, ms=t_dec, launches=launches,
                                           algorithmic_mb=dec_bytes / 1e6, hbm_gbs=dec_bytes / t_dec / 1e6,
                                           frac_of_hbm_peak=dec_bytes / t_dec / 1e6 / pk["hbm"])
    enc = res["encoder_Lq=S"]
    line = {
        "metric": "MSDeformAttn + masked-attention decoder microbench, 256 queries x 4 scales, HBM GB/s",
        "value": enc["ours_abi_gbs"], "unit": "GB/s", "n_gpus": 1, "steps": reps, "warmup": warm,
        "ms_per_step": enc["ours_abi_us"] / 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"c4: MSDeformAttn forward, N={N}, 4 levels {shapes}, S={S}, M=8, D=32, P=4 (value = compulsory "
                               "bytes / time of odise_msda_forward_f32 with Lq = S); masked-attention decoder Q=256 x 4 scales",
                   "l2": "value (N x 22 MB) + loc/attn/out streams > 126 MB L2 at N = 4"},
        "roofline": {"bound": "hbm", "kernel": "msda_d32_kernel", "achieved": enc["ours_abi_gbs"], "peak": pk["hbm"],
                     "unit": "GB/s", "frac": enc["ours_abi_gbs"] / pk["hbm"], "traffic": None,
                     "note": "the gathers move 4 corners x 128 B per (query, head, sample) through L1: "
                             f"{enc['gather_l1_tbs']:.1f} TB/s of L1 wavefronts; that data path, not HBM, bounds the kernel"},
        "c4": res,
        "gpu_launches": int(launches),
    }
    if args.dump_outputs:
        dump_outputs(dumps, args.dump_outputs)
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- our arm
def main():
    args = parse()
    args.full = not args.hot_path_only
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: odise_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if args.config == "c4":
        if rank == 0:
            run_c4(args, dev)
        return
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from odise_b200 import lib, spec
    from odise_b200.pipeline import ODISEEngine, full_param_list, gather_logits
    lib.load()
    nmma = NMMA[args.precision]
    sd = spec.synth_state_dict(full_param_list(with_vae=args.full, with_clip=args.full), seed=0)
    eng = ODISEEngine(sd, dev, nmma=nmma, with_vae=args.full, with_clip=args.full, synthetic_uncond=True)
    del sd
    ncls, npr = VOCABS[args.vocab]
    eng.set_synthetic_vocabulary(args.vocab, ncls, npr)
    B, S = args.batch, args.size
    g = torch.Generator().manual_seed(1234 + rank)
    images = torch.randint(0, 256, (B, 3, S, S), generator=g, dtype=torch.uint8).pin_memory()

    graph, out = eng.capture(B, S, S, post=True)
    launches_per_step = eng.launches_per_step

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        s, e = torch.cuda.Event(True), torch.cuda.Event(True)
        s.record()
        for _ in range(steps):
            fn()
        e.record()
        barrier()
        ms = s.elapsed_time(e)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def dev_step():
        graph.replay()
        gather_logits(out["pred_logits"])

    last = {}

    def e2e_step():
        r = eng.infer(images, outputs="panoptic")
        if world > 1:
            gather_logits(out["pred_logits"])
        last["r"] = r
        return r

    for _ in range(args.warmup):
        dev_step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_dev = timed(dev_step, args.steps)
    for _ in range(max(1, args.warmup // 2)):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # infer() returns its pinned host buffers, which the next call overwrites: write them before anything else runs
        dump_outputs(last["r"], args.dump_outputs)

    # roofline of the dominant kernel (gemm_tc_kernel): one eager pass with per-launch CUDA events
    lib.profile_begin()
    eng.step_full(B, S, S)
    n_gemm, gemm_ms, gemm_flops = lib.profile_end()
    torch.cuda.synchronize()
    # the north-star stage on its own: SD-v1 UNet feature pass (minimal pass, 0.740 TFLOP per 512^2 crop) on resident inputs
    from odise_b200.backbone import SyntheticTaps
    crops = n_crops(S)
    nc_all = B * crops
    tp_ = SyntheticTaps(dev)(nc_all)
    ctx_, cemb_ = eng.backbone.conditioning(tp_["clip_embed"], nc_all)
    lat_, lh_, lw_ = tp_["latent"]
    x_ = eng.backbone.q_sample(lat_, nc_all, lh_, lw_)
    for _ in range(2):
        eng.backbone.unet.forward(x_, nc_all, lh_, lw_, ctx_, cemb_)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(True), torch.cuda.Event(True)
    ev0.record()
    for _ in range(3):
        eng.backbone.unet.forward(x_, nc_all, lh_, lw_, ctx_, cemb_)
    ev1.record()
    torch.cuda.synchronize()
    unet_ms = ev0.elapsed_time(ev1) / 3
    extra = {}
    if args.config == "c5":
        # BASELINE.json configs[4]: the mask-embed x text-bank GEMMs on their own (cal_pred_logits odise.py:192-205 on the
        # projected 256-d bank; MaskCLIP's match clip.py:352-358 on the raw 768-d bank), CUDA events over 200 launches
        from odise_b200 import ops
        v = eng.head._vocab[eng.vocab_key]
        me_p = ops.l2_normalize_split(torch.randn(B * eng.Q, 256, device=dev), lo=nmma != 1)
        sims = ops.empty(B * eng.Q, v["Kp"], dev)
        t1 = _time_ms(lambda: lib.gemm(me_p, v["te_p"], nmma=nmma, alpha=eng.head.logit_scale, out=sims), 200)
        fl1 = 2.0 * B * eng.Q * v["Kp"] * 256
        cv = eng.clip_head._vocab[eng.vocab_key] if eng.clip_head is not None else None
        extra["clip_match_gemm"] = {"category_head": {"M": B * eng.Q, "N": v["Kp"], "K": 256, "us": 1e3 * t1,
                                                      "tflops": fl1 / t1 / 1e9}}
        if cv is not None:
            ce_p = ops.l2_normalize_split(torch.randn(B * eng.Q, 768, device=dev), lo=nmma != 1)
            sims2 = ops.empty(B * eng.Q, v["Kp"], dev)
            t2 = _time_ms(lambda: lib.gemm(ce_p, cv["te_p"], nmma=nmma, alpha=100.0, out=sims2), 200)
            extra["clip_match_gemm"]["maskclip_head"] = {"M": B * eng.Q, "N": v["Kp"], "K": 768, "us": 1e3 * t2,
                                                         "tflops": 2.0 * B * eng.Q * v["Kp"] * 768 / t2 / 1e9}
        extra["clip_match_gemm"]["note"] = ("400 x 1342 outputs: one wave of 128 x 128 tiles, launch / pipeline-fill bound "
                                            "(~10 us); the same GEMM at 6400 rows runs at > 130 TFLOP/s (profiles/ncu_r1)")
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    ips = world * B * args.steps / (ms_dev / 1000.0)
    ips_e2e = world * B * args.steps / (ms_e2e / 1000.0)
    achieved = gemm_flops / (gemm_ms / 1000.0) / 1e12
    traffic = None
    tp = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    traffic_src = None
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
        except Exception:
            traffic = None
    metric = METRIC if S == 1024 else METRIC.replace("1024x1024", f"{S}x{S}")
    line = {
        "metric": metric, "value": ips, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
        "config": {"workload": f"{args.config}: ODISE(label) per-image inference, batch {B}/GPU x {S}x{S}, {crops} crops/image, "
                               f"{args.vocab} ({ncls} classes / {npr} prompts), Q=100",
                   "stages": ("CLIP ViT-L/14-336 image tower on every crop, KL-VAE encoder + truncated decoder (taps), "
                              if args.full else "") + ("MaskCLIP (100 mask tokens/image through the ViT) + alpha/beta "
                              "ensemble + void merge, " if args.full else "") +
                             "implicit-captioner front, q_sample, SD-v1 UNet feature pass (4 taps), 8 projections, "
                             "MSDeformAttn pixel decoder, 9-layer masked-attention decoder, CLIP-text scoring, semantic + "
                             f"panoptic + instance inference at {S}x{S} (odise.py:326-370), NCCL all-gather of logits",
                   "not_in_path": ("nothing of the per-image pass: CLIP image tower, KL-VAE taps, MaskCLIP and the inference heads "
                                   "ARE executed; the CLIP TEXT bank of the vocabulary is precomputed per vocabulary (as in the "
                                   "reference)") if args.full else
                                  ("KL-VAE encoder/decoder taps and CLIP image embedding enter as seeded synthetic "
                                   "tensors (SURVEY.md §8f rows f-1/f-2)"),
                   "weights": "random-init (seed 0), SD-v1 / ODISE shapes", "global_batch": world * B,
                   "parallelism": f"dp{world} (image sharded)", "precision_mode": args.precision,
                   "l2": "working set >> 126 MB L2: ~3.6 GB of weight planes + multi-GB activations stream every step",
                   "cuda_graph": True},
        "e2e": {"value": ips_e2e, "unit": "images/s", "h2d_bytes_per_step": int(images.numel()),
                "d2h_bytes_per_step": eng.d2h_bytes(), "ms_per_step": ms_e2e / args.steps,
                "returns": "panoptic map int32 [B,H,W] + segment table + instance table (scores/classes/query) + class logits"},
        "gpu_launches": int(launches_per_step * args.steps * 2),
        "gpu_launches_per_step": int(launches_per_step),
        "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 GEMM / implicit conv, all launches of a step)",
                     "achieved": achieved, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                     "frac": achieved / pk["bf16_sustained"], "peak_source": pk["source"] + " sustained cuBLAS bf16",
                     "launches": int(n_gemm), "gemm_ms_per_step": gemm_ms, "algorithmic_tflop_per_step": gemm_flops / 1e12,
                     "mma_kind": "tcgen05.mma kind::f16 (bf16 in, fp32 TMEM accumulate)" +
                                 (", 3 MMAs per k-step (bf16x3 split)" if nmma == 3 else "") +
                                 (" for the head; VAE / CLIP / UNet / projections: kind::f16 (fp16 hi x hi) + kind::f8f6f4 "
                                  "(e5m2 cross terms, K = 32) = 2 MMA units per k-step" if nmma == 2 else ""),
                     "tensor_pipe_equiv_frac": achieved * nmma / pk["bf16_sustained"],
                     "unet_frac_of_step": (UNET_TFLOP_PER_CROP * crops * B) / (gemm_flops / 1e12), "traffic": traffic,
                     "traffic_source": traffic_src,
                     "unet_feature_pass": {
                         "ms": unet_ms, "crops": nc_all, "algorithmic_tflop": UNET_TFLOP_PER_CROP * nc_all,
                         "achieved_tflops": UNET_TFLOP_PER_CROP * nc_all / (unet_ms / 1000.0),
                         "frac_of_bf16_peak": UNET_TFLOP_PER_CROP * nc_all / (unet_ms / 1000.0) / pk["bf16_sustained"],
                         "tensor_pipe_equiv_frac": nmma * UNET_TFLOP_PER_CROP * nc_all / (unet_ms / 1000.0) / pk["bf16_sustained"],
                         "note": "whole UNet pass incl. GroupNorm / attention softmax / elementwise kernels, eager launches, "
                                 "CUDA events; minimal pass FLOPs (output block 11 + out skipped)"}},
    }
    line.update(extra)
    if not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = CpuHotPath(S, args.vocab, full=args.full).sample()
        except Exception as ex:  # noqa
            line["cpu_baseline"] = {"error": str(ex)}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
