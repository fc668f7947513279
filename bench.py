#!/usr/bin/env python
"""bench.py -- images/s of the ViT-VQGAN fwd+bwd hot path (BASELINE.json metric) on N B200s.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 5 --warmup 3
    python bench.py --impl reference --steps 3 --warmup 1      # the CPU arm (reference modules / oracle port)
    python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs /tmp/out   # + the last timed step's loss and gradients

One "step" = x -> ViTEncoder -> pre_quant -> VectorQuantizer -> post_quant -> ViTDecoder ->
loss = mean((rec-x)^2) + qloss -> backward, fp32 parameters, no optimizer step (SURVEY.md
section 8d).  Workload: imagenet_vitvq_base.yaml shapes, synthetic 256x256 images, batch 128
per GPU (BASELINE.json configs[1]); weak scaling, gradients all-reduced over NCCL.

Prints ONE JSON line on rank 0 (see DESIGN.md 'Measurement' for every key).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it

DUMP_BUDGET_BYTES = 64 * 2 ** 20
DUMP_SAMPLE = 32768                     # elements kept of a larger gradient

METRIC = "images/sec (256x256) ViT-VQGAN fwd+bwd"
UNIT = "images/s"
FP32_FMA_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12     # 148 SMs x 128 FMA lanes x 2 FLOP x 1.965 GHz = 74.5


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"], bf16_tflops_sustained=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = max((int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()), default=None)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        pw = max((float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "", 1).isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm), "power_w_max": pw}


# ------------------------------------------------------------------------------------------------
# the reference's own PyTorch path (CPU arm and eager-GPU arm)
# ------------------------------------------------------------------------------------------------
def reference_modules():
    """the reference's layers.py / quantizers.py, vendored unmodified into oracle/_ref by oracle/build_ref.py
    (git-ignored; they travel to the GPU box with the snapshot).  None if absent."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref", "enhancing_ref")
    if not (os.path.exists(os.path.join(ref_dir, "layers.py")) and os.path.exists(os.path.join(ref_dir, "quantizers.py"))):
        return None
    import importlib.util
    import numpy as np
    if not hasattr(np, "float"):
        np.float = float                      # layers.py:57 uses the alias numpy removed in 1.24 (harness-side shim)
    mods = {}
    for name in ("layers", "quantizers"):
        spec = importlib.util.spec_from_file_location(f"enhancing_ref.{name}", os.path.join(ref_dir, f"{name}.py"))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        mods[name] = m
    return mods


class RefHotPath:
    """encoder -> pre_quant -> quantizer -> post_quant -> decoder -> loss with the REFERENCE's own nn.Modules
    (kind "reference"), or with the oracle port when oracle/_ref is absent (kind "port")"""

    def __init__(self, cfg_name, device, seed=0):
        import torch
        from oracle import vitvq_oracle as O
        self.torch, self.O, self.device = torch, O, device
        self.cfg = cfg = O.CONFIGS[cfg_name]
        ref = reference_modules()
        sd = O.init_vitvq_sd(cfg, seed=seed)
        if ref is not None:
            self.kind = "reference"
            e, d, q = cfg["encoder"], cfg["decoder"], cfg["quantizer"]
            self.mods = dict(encoder=ref["layers"].ViTEncoder(cfg["image_size"], cfg["patch_size"], **e),
                             decoder=ref["layers"].ViTDecoder(cfg["image_size"], cfg["patch_size"], **d),
                             quantizer=ref["quantizers"].VectorQuantizer(**q),
                             pre_quant=torch.nn.Linear(e["dim"], q["embed_dim"]), post_quant=torch.nn.Linear(q["embed_dim"], d["dim"]))
            for name, m in self.mods.items():
                m.load_state_dict({k[len(name) + 1:]: v for k, v in sd.items() if k.startswith(name + ".")}, strict=True)
                m.to(device)
            self.params = [p for m in self.mods.values() for p in m.parameters()]
        else:
            self.kind = "port"
            self.sd = {k: v.to(device).requires_grad_(v.is_floating_point() and "pos_embedding" not in k) for k, v in sd.items()}
            self.params = list(self.sd.values())

    def step(self, img):
        for p in self.params:
            p.grad = None
        if self.kind == "reference":
            m = self.mods
            quant, qloss, _ = m["quantizer"](m["pre_quant"](m["encoder"](img)))
            rec = m["decoder"](m["post_quant"](quant))
            loss = ((rec - img) ** 2).mean() + qloss
        else:
            loss, _, _ = self.O.vitvq_loss(self.sd, img, self.cfg)
        loss.backward()
        return loss


def cpu_threads():
    """torch's intra-op pool collapses when oversubscribed on the 2-socket / 128-thread GPU hosts (measured round 1:
    base B=4 takes 94 s with 128 threads, 4 s with 32): a fixed 32 threads (or every core of a smaller host)."""
    return min(32, os.cpu_count() or 1)


def cpu_model():
    try:
        with open("/proc/cpuinfo") as fh:
            for ln in fh:
                if ln.lower().startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_reference_run(cfg_name, batch, warmup, steps):
    import torch
    threads = cpu_threads()
    torch.set_num_threads(threads)
    hp = RefHotPath(cfg_name, torch.device("cpu"))
    img = torch.rand(batch, 3, hp.cfg["image_size"], hp.cfg["image_size"], generator=torch.Generator().manual_seed(0))
    for _ in range(warmup):
        hp.step(img)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        hp.step(img)
        times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return dict(value=batch / sec, unit=UNIT, cores=threads, kind=hp.kind, host_cpus=os.cpu_count(), cpu_model=cpu_model(), ms_per_step=sec * 1e3,
                sample=f"{warmup} warm-up + {steps} timed fwd+bwd steps of {batch} images, {cfg_name} config, "
                       f"{'reference nn.Modules (oracle/_ref)' if hp.kind == 'reference' else 'oracle port'} on torch CPU fp32, "
                       f"{threads} threads")


def run_reference(args):
    """--impl reference: the reference's own CPU path on the box's host cores, bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_reference_run(args.config, args.ref_batch, max(1, args.warmup), max(1, args.steps))
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"imagenet_vitvq_{args.config}.yaml shapes, synthetic 256x256, fwd+bwd, CPU sample of {args.ref_batch} images/step",
                   "global_batch": args.ref_batch, "parallelism": "host threads"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def gpu_eager_baseline(cfg_name, dev, batches=(64, 48, 32, 16, 8)):
    """the reference modules .cuda() eagerly on this B200 (cuBLAS / cuDNN / ATen): the honest 'reference on this
    box' bar (SURVEY.md section 8d), at the largest batch that fits, with TF32 matmuls off and on"""
    import torch
    out = {}
    for tf32 in (False, True):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.allow_tf32 = tf32
        for B in batches:
            hp = None
            try:
                hp = RefHotPath(cfg_name, dev)
                img = torch.rand(B, 3, 256, 256, device=dev)
                for _ in range(2):
                    hp.step(img)
                torch.cuda.synchronize(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(3):
                    hp.step(img)
                e1.record()
                torch.cuda.synchronize(dev)
                ms = e0.elapsed_time(e1) / 3
                out["tf32_matmul" if tf32 else "fp32_matmul"] = dict(value=B / ms * 1e3, unit=UNIT, batch=B, ms_per_step=ms,
                                                                     peak_mem_gib=torch.cuda.max_memory_allocated(dev) / 2 ** 30)
                break
            except torch.OutOfMemoryError:
                pass
            finally:
                del hp
                torch.cuda.empty_cache()
                torch.cuda.reset_peak_memory_stats(dev)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    out["kind"] = "reference" if reference_modules() is not None else "port"
    out["note"] = "3 timed fwd+bwd steps after 2 warm-ups, eager PyTorch (cuBLAS/ATen), largest batch of (64,48,32,16,8) that fits"
    return out


def vq_block(dev, peaks):
    """BASELINE metric part 2: the fused VQ lookup alone, M = 131072 tokens, 8192 codes, D = 32 (SURVEY.md section 8d:
    264 B/token + 1 MiB codebook algorithmic bytes; 524288 FLOP/token/depth -- compute-bound by construction)"""
    import torch
    import enhancing_transformers_b200 as etb
    ops = etb.ops
    M, K, D = 131072, 8192, 32
    g = torch.Generator(device="cpu").manual_seed(0)
    E = torch.randn(K, D, generator=g).to(dev)
    z_rand = torch.randn(M, D, generator=g).to(dev)
    z_clu = (E[torch.randint(0, 45, (M,), generator=g).to(dev)] + 0.01 * torch.randn(M, D, generator=g).to(dev)).contiguous()
    flush = torch.empty(160 * 2 ** 20 // 4, device=dev)           # > 126 MB L2: written between timed launches

    def timed(fn, iters=5):
        for _ in range(2):
            fn()
        tot = 0.0
        for _ in range(iters):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); fn(); e.record()
            torch.cuda.synchronize(dev)
            tot += s.elapsed_time(e)
        return tot / iters
    res = {"tokens": M, "n_embed": K, "embed_dim": D, "l2_hygiene": "160 MB buffer written between timed launches"}
    for name, z, depth in (("depth1", z_rand, 1), ("depth4", z_rand, 4), ("depth1_clustered", z_clu, 1)):
        ms = timed(lambda: ops.vq_fwd(z, E, depth, 0.25))
        bytes_alg = M * (128 + 128 + 8 * depth) + K * D * 4
        flops = 2.0 * D * K * M * depth
        res[name] = dict(ms=ms, gb_s=bytes_alg / ms / 1e6, gb_s_frac_of_hbm=bytes_alg / ms / 1e6 / peaks["hbm_gbs"],
                         tflops=flops / ms / 1e9, frac_of_fp32_fma_peak=flops / ms / 1e9 / FP32_FMA_PEAK_TFLOPS)
        _, _, idx = ops.vq_fwd(z, E, depth, 0.25)
        g_out, g_loss = torch.randn(M, D, device=dev), torch.ones((), device=dev)
        msb = timed(lambda: ops.vq_bwd(z, E, idx, g_out, g_loss, depth > 1, 0.25))
        res[name]["bwd_ms"] = msb
        res[name]["bwd_gb_s"] = (M * (392 + 8 * (depth - 1)) + K * D * 4) / msb / 1e6
        res[name]["live_codes"] = int(idx[:, 0].unique().numel())
    res["note"] = ("forward time includes vq_prep (codebook normalise + transpose) and the loss reduction; the lookup is FP32-FMA "
                   "bound (1986 FLOP/B), so GB/s is a few % of HBM by construction and the kernel is graded on frac_of_fp32_fma_peak "
                   f"(peak {FP32_FMA_PEAK_TFLOPS:.1f} TFLOP/s = 148 SM x 128 lanes x 2 x 1.965 GHz)")
    return res


def dump_outputs(out_dir, loss, named_params):
    """what the caller of one timed step receives -- the loss and every parameter's gradient -- as float32 .npy files:
    loss.npy and grad.<parameter name>.npy.  A gradient of more than DUMP_SAMPLE elements is stored as the elements at
    DUMP_SAMPLE fixed positions (a permutation seeded by the parameter name, sorted), so that two builds of the project can
    be compared output for output."""
    import zlib

    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.detach().float().cpu().numpy()}
    for name, p in named_params:
        if p.grad is None:
            continue
        flat = p.grad.detach().float().reshape(-1)
        if flat.numel() > DUMP_SAMPLE:
            g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
            idx = torch.randperm(flat.numel(), generator=g)[:DUMP_SAMPLE].sort().values
            flat = flat[idx.to(flat.device)]
        arrays["grad." + name] = flat.cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_BUDGET_BYTES, f"--dump-outputs: {total} bytes exceed the {DUMP_BUDGET_BYTES}-byte budget"
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="base", choices=["tiny", "small", "base", "base_rq4", "large"])
    ap.add_argument("--batch", type=int, default=128, help="images per GPU per step")
    ap.add_argument("--precision", default=None, choices=["fp16", "tf32", "parity"], help="data path (default: fp16)")
    ap.add_argument("--cta-group", type=int, default=int(os.environ.get("B200VQ_CTA_GROUP", "2")))
    ap.add_argument("--ref-batch", type=int, default=4, help="images per CPU step for --impl reference / cpu_baseline")
    ap.add_argument("--ddp", action="store_true", help="torch DistributedDataParallel (overlapped buckets) instead of one flat all-reduce")
    ap.add_argument("--no-fuse-pos", action="store_true", help="keep post_quant and the decoder's positional add separate")
    ap.add_argument("--extras", default="vq,secondary,eager,cpu",
                    help="comma list of the 1-GPU extra blocks to measure after the timed regions: vq, secondary, eager, cpu ('' = none)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's loss and parameter gradients (sampled, float32) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import torch.nn as nn

    import enhancing_transformers_b200 as etb
    from enhancing_transformers_b200.configs import CONFIGS, flops_per_image, gemm_flops_per_image

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    etb.functional.GEMM_CTA_GROUP = args.cta_group
    if args.precision:
        etb.set_precision(args.precision)
    precision = etb.get_precision()

    class HotPath(nn.Module):
        """the five modules of ViTVQ.forward (vitvqgan.py:35-39,44-72) + the bench loss"""

        def __init__(self, cfg):
            super().__init__()
            e, d, q = cfg["encoder"], cfg["decoder"], cfg["quantizer"]
            self.encoder = etb.ViTEncoder(cfg["image_size"], cfg["patch_size"], **e)
            self.decoder = etb.ViTDecoder(cfg["image_size"], cfg["patch_size"], **d)
            self.quantizer = etb.VectorQuantizer(**q)
            self.pre_quant = etb.QuantLinear(e["dim"], q["embed_dim"])
            self.post_quant = etb.QuantLinear(q["embed_dim"], d["dim"])
            if not args.no_fuse_pos:
                etb.fuse_post_quant_pos(self)      # SURVEY.md 8f-1: + de_pos_embedding in post_quant's GEMM epilogue (bit-identical)

        def forward(self, x):
            quant, qloss, _ = self.quantizer(self.pre_quant(self.encoder(x)))
            rec = self.decoder(self.post_quant(quant))
            return ((rec - x) ** 2).mean() + qloss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_step(model, net, comm_events=None):
        params = list(model.parameters())
        flat = etb.FlatGradients(params) if (world > 1 and not args.ddp) else None

        def step(x, second_forward=False):
            if flat is not None:
                flat.zero_()                   # .grad = views into one flat buffer: the all-reduce needs no bucket copies
            else:
                for p in params:
                    p.grad = None
            if second_forward:                 # the reference training_step runs forward twice per batch (vitvqgan.py:101-127)
                with torch.no_grad():
                    net(x)
            loss = net(x)
            loss.backward()
            if flat is not None:
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                flat.allreduce()
                e.record()
                if comm_events is not None:
                    comm_events.append((s, e))
            return loss
        return step

    cfg = CONFIGS[args.config]
    torch.manual_seed(0)
    model = HotPath(cfg).to(dev)
    net = nn.parallel.DistributedDataParallel(model, device_ids=[local], gradient_as_bucket_view=True) if (world > 1 and args.ddp) else model
    B = args.batch
    gen = torch.Generator().manual_seed(1234 + rank)
    host_imgs = [torch.rand(B, 3, cfg["image_size"], cfg["image_size"], generator=gen).pin_memory() for _ in range(2)]
    dev_imgs = host_imgs[0].to(dev, non_blocking=True)
    torch.cuda.synchronize()
    comm_events = []
    step = make_step(model, net, comm_events)

    # ---- warm-up -----------------------------------------------------------------------------
    warm = max(args.warmup, 3)
    for _ in range(warm):
        step(dev_imgs)
    barrier()
    comm_events.clear()

    # ---- device-resident timed region (value) + per-GEMM events (roofline) -------------------
    gemm_events = []
    orig_gemm = etb.ops.gemm

    def timed_gemm(a, b, M, N, K, **kw):
        s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = orig_gemm(a, b, M, N, K, **kw)
        t.record()
        passes = 3 if kw.get("a_lo") is not None else 1
        gemm_events.append((s, t, 2.0 * M * N * K * kw.get("splits", 1), a.dtype == torch.float16, passes))
        return out

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    etb.ops.gemm = timed_gemm
    launches0 = etb.ops.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        step(dev_imgs)
    ev1.record()
    barrier()
    launches = etb.ops.launch_count() - launches0
    etb.ops.gemm = orig_gemm
    ms_total = ev0.elapsed_time(ev1)
    gemm_ms = sum(s.elapsed_time(t) for s, t, *_ in gemm_events)
    gemm_flops = sum(f for _, _, f, *_ in gemm_events)
    f16_ms = sum(s.elapsed_time(t) for s, t, _, h, _ in gemm_events if h)
    f16_flops = sum(f for _, _, f, h, _ in gemm_events if h)
    n_gemm = len(gemm_events)
    comm_ms = sum(s.elapsed_time(e) for s, e in comm_events) / max(1, args.steps)
    comm_events.clear()

    # ---- end-to-end timed region: pinned host images in (prefetched on a copy stream), loss out, every step ----
    copy_stream = torch.cuda.Stream(device=dev)
    barrier()
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev2.record()
    last = 0.0
    with torch.cuda.stream(copy_stream):
        nxt = host_imgs[0].to(dev, non_blocking=True)
    for i in range(args.steps):
        torch.cuda.current_stream().wait_stream(copy_stream)
        x = nxt
        x.record_stream(torch.cuda.current_stream())
        if i + 1 < args.steps:
            with torch.cuda.stream(copy_stream):       # step i+1's images travel while step i computes
                nxt = host_imgs[(i + 1) % 2].to(dev, non_blocking=True)
        loss = step(x)
        last = float(loss.item())                      # device -> host read of the step's result
    ev3.record()
    barrier()
    ms_e2e = ev2.elapsed_time(ev3)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, sorted(model.named_parameters()))

    t = torch.tensor([ms_total, ms_e2e, comm_ms], device=dev, dtype=torch.float64)
    per_rank = comm_rank = None
    if world > 1:
        gathered = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(gathered, t)
        per_rank = [float(g[0]) / args.steps for g in gathered]
        comm_rank = [float(g[2]) for g in gathered]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e, comm_ms = float(t[0]), float(t[1]), float(t[2])

    line = None
    if rank == 0:
        peaks = load_peaks()
        imgs = world * B * args.steps
        value = imgs / (ms_total / 1e3)
        e2e = imgs / (ms_e2e / 1e3)
        flops_step = 3.0 * flops_per_image(cfg) * B
        achieved = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
        peak = peaks["bf16_tflops_sustained"]
        kern = {"fp16": "gemm_tc_kernel<KIND=f16> (tcgen05 kind::f16, fp32 accumulate)", "tf32": "gemm_tc_kernel<KIND=tf32> (tcgen05 kind::tf32)",
                "parity": "gemm_tc_kernel<KIND=tf32>, 3 passes (3xTF32)"}[precision]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp16": "fp16 tensor-core operands / fp32 accumulate (block GEMMs and attention core), 3xtf32 (patch embed, to_pixel, pre/post_quant), fp32 (everything else)",
                      "tf32": "tf32", "parity": "3xtf32 (fp32-grade)"}[precision], "data": "synthetic",
            "config": {"workload": f"imagenet_vitvq_{args.config}.yaml shapes (ViT-VQGAN-{args.config}), synthetic 256x256x3, "
                                   f"fwd+bwd, batch {B}/GPU", "global_batch": world * B, "per_gpu_batch": B,
                       "parallelism": f"dp{world}", "l2_hygiene": "inputs_exceed_l2 (activations >> 126 MB per step)",
                       "gemm_cta_group": args.cta_group, "precision": precision, "post_quant_pos_fused": not args.no_fuse_pos,
                       "grad_reduce": ("torch DDP buckets (overlapped)" if args.ddp else "one flat NCCL all-reduce after backward") if world > 1 else "none"},
            "model_tflops_per_gpu": flops_step / (ms_total / args.steps / 1e3) / 1e12,
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": host_imgs[0].numel() * 4, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps, "last_loss": last,
                    "note": "images prefetched from pinned host memory on a copy stream (step i+1 travels while step i computes); loss.item() every step"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": kern, "achieved": achieved, "peak": peak,
                         "unit": "TFLOP/s", "frac": achieved / peak,
                         "traffic": 7.544e8 if (args.config == "base" and B == 128 and precision == "fp16") else None,
                         "traffic_note": "dram read+write bytes of one to_qkv launch (M=131072 N=2304 K=768, fp16 in/out) from profiles/r02_ncu_gemm_f16.txt "
                                         "(ncu --set full); algorithmic bytes of that launch: 8.09e8 (A 201 MB + B 3.5 MB + C 604 MB); tensor pipe 86 % "
                                         "active there, 90 % on the K=3072 net.2 launch",
                         "peak_source": peaks["source"] + ": cuBLAS bf16 sustained (kind::f16 issues at the bf16 rate; kind::tf32 at half of it)",
                         "launches_timed": n_gemm, "share_of_step": gemm_ms / ms_total,
                         "algorithmic_gemm_tflop_per_step": 3.0 * gemm_flops_per_image(cfg) * B / 1e12,
                         "f16_gemms": {"achieved": f16_flops / (f16_ms / 1e3) / 1e12 if f16_ms > 0 else None,
                                       "frac": f16_flops / (f16_ms / 1e3) / 1e12 / peak if f16_ms > 0 else None,
                                       "share_of_step": f16_ms / ms_total},
                         "hbm_peak_gbs": peaks["hbm_gbs"]},
        }
        if world > 1:
            line["comm"] = {"allreduce_ms": min(comm_rank) if not args.ddp else None,
                            "wait_for_slowest_rank_ms": (max(comm_rank) - min(comm_rank)) if not args.ddp else None,
                            "allreduce_ms_per_rank": comm_rank if not args.ddp else None,
                            "per_rank_ms_per_step": per_rank,
                            "note": "flat all-reduce issued after backward on the compute stream, bracketed by events on every rank: the "
                                    "rank that arrives last sees the all-reduce alone (allreduce_ms = min over ranks; tools/nccl_probe.py "
                                    "measures the same 0.65 GB buffer at 1.26 ms on an idle pair); what the other ranks see on top of that "
                                    "is time spent waiting for the slowest GPU, not communication" if not args.ddp else
                                    "DDP: bucketed all-reduce overlapped with backward on NCCL's stream"}
    del model, net, step
    torch.cuda.empty_cache()

    # ---- extras (rank 0, one GPU): VQ block, secondary configs, eager-GPU reference, CPU reference --------------
    extras = set(x for x in args.extras.split(",") if x) if (rank == 0 and world == 1) else set()
    def guarded(key, fn):
        """an extra block must never cost the headline line: record its error instead"""
        try:
            line[key] = fn()
        except Exception as exc:
            line[key] = {"error": f"{type(exc).__name__}: {exc}"}
            torch.cuda.empty_cache()

    def secondary_block():
        sec = {}
        for name, cname, b, second in (("base_rq4_B128", "base_rq4", 128, False), ("large_B32", "large", 32, False),
                                       ("base_B128_2fwd_1bwd", "base", 128, True), ("base_B32_parity_mode", "base", 32, False)):
            etb.set_precision("parity" if name.endswith("parity_mode") else precision)
            torch.manual_seed(0)
            m2 = HotPath(CONFIGS[cname]).to(dev)
            st = make_step(m2, m2)
            x = torch.rand(b, 3, 256, 256, device=dev)
            for _ in range(3):
                st(x, second)
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(3):
                st(x, second)
            e.record()
            torch.cuda.synchronize()
            ms = s.elapsed_time(e) / 3
            sec[name] = dict(value=b / ms * 1e3, unit=UNIT, ms_per_step=ms, batch=b,
                             model_tflops=(4.0 if second else 3.0) * flops_per_image(CONFIGS[cname]) * b / ms / 1e9)
            del m2, st, x
            torch.cuda.empty_cache()
        try:
            sec.update(stage2_entry())
        except Exception as exc:
            sec["stage2_gpt_w1024_L8_B32"] = {"error": f"{type(exc).__name__}: {exc}"}
            torch.cuda.empty_cache()
        etb.set_precision(precision)
        sec["note"] = ("3 timed steps after 3 warm-ups each; base_rq4 = BASELINE config 3 (use_residual, num_quantizers=4); large_B32 = the per-GPU "
                       "share of BASELINE config 4 (batch 256 over 8 GPUs); 2fwd_1bwd = the reference training_step shape (vitvqgan.py:101-127); parity_mode = the 3xTF32 data path "
                       "(etb.set_precision('parity'): reconstructions within 3e-5 of the fp64 oracle, tests/test_gpu_model.py)")
        return sec

    def stage2_entry():
        """BASELINE config 5 (stage-2 transformer on 1 class token + 32 x 32 codes) at a width the kernels cover"""
        import torch.nn.functional as F
        gcfg = dict(vocab_cond_size=1000, vocab_img_size=8192, embed_dim=1024, cond_num_tokens=1, img_num_tokens=1024, n_heads=16, n_layers=8)
        torch.manual_seed(0)
        gpt = etb.GPT(**gcfg).to(dev)
        gb = 32
        codes = torch.randint(0, 8192, (gb, 1024), device=dev)
        conds = torch.randint(0, 1000, (gb, 1), device=dev)

        def gstep():
            gpt.zero_grad(set_to_none=True)
            lg = gpt(codes, conds)
            F.cross_entropy(lg.view(-1, 8192), codes.view(-1)).backward()
        etb.set_precision("fp16")
        for _ in range(3):
            gstep()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(3):
            gstep()
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e) / 3
        C, L, T, V = 1024, 8, 1025, 8192
        out = {"stage2_gpt_w1024_L8_B32": dict(value=gb * T / ms * 1e3, unit="tokens/s", ms_per_step=ms, batch=gb,
                                               model_tflops=3.0 * (L * (24 * C * C + 2 * T * C) + 2 * C * V) * gb * T / ms / 1e9,
                                               note="stage-2 GPT fwd+bwd (cross-entropy), fp16-operand Linear layers + tf32 masked attention core, "
                                                    "reduced width (the YAML's 6144 / 384-per-head model is not covered by the kernels)")}
        del gpt, codes, conds
        torch.cuda.empty_cache()
        return out

    if "vq" in extras:
        guarded("vq", lambda: vq_block(dev, peaks))
    if "secondary" in extras:
        guarded("secondary", secondary_block)
    if "eager" in extras:
        guarded("gpu_eager_baseline", lambda: gpu_eager_baseline(args.config, dev))
    if "cpu" in extras:
        guarded("cpu_baseline", lambda: cpu_reference_run(args.config, args.ref_batch, 1, 3))
        if args.config == "base":      # BASELINE config 1 (imagenet_vitvq_small.yaml, batch 4: the reference's CPU-runnable case)
            guarded("cpu_baseline_config1", lambda: cpu_reference_run("small", 4, 1, 3))
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
