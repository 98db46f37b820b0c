#!/usr/bin/env python
"""bench.py — images/sec of the PASSL self-supervised hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W [--config c2|c3|c4|c5]     (N>1: launched by torch.distributed.run, one rank per GPU)
  python bench.py ... --dump-outputs DIR                                   also writes what the last timed step computed (seeded inputs)
  python bench.py --impl reference ...                                     the reference math on the host CPU cores (oracle port)

Workloads (BASELINE.json `configs`; default c2 = the one the metric is quoted on):
  c2  SimCLR ResNet-50, bf16 tensor-core math, 224^2, 512 samples x 2 views per GPU (global 4096 at 8 GPUs), all-gathered negatives,
      NT-Xent + CO2 head, LARS                                       (configs/simclr/simclr_r50_IM.yaml)
  c3  MoCo v2 ResNet-50, K=65536 queue, 256 samples x 2 views per GPU, InfoNCE over the queue, Momentum   (configs/moco/moco_v2_r50.yaml)
  c4  MAE ViT-B/16, mask 0.75, norm_pix, 512 images per GPU, AdamW   (configs/mae/mae_vit_b_pretrain.yaml)
  c5  CLIP ViT-B/16 + text 12x512, 1024 image-text pairs per GPU (global 8192), AdamW                      (configs/clip)
A "step" = forward + loss + backward + gradient all-reduce + optimizer (+ EMA / queue for MoCo) on synthetic inputs of that shape.

Prints ONE JSON line (rank 0).  `value`: inputs resident in HBM; `e2e`: same step fed from pinned host memory every step with a
device->host read of the loss; `roofline`: the tcgen05 GEMM / implicit-GEMM launches of one instrumented step classed by their
binding roofline; `roofline_infonce`: the fused InfoNCE kernel (MoCo C3 shape) against the measured HBM peak — the second half of
BASELINE's metric; `cpu_baseline`: the oracle port of BASELINE configs[0] (MoCo v2 bs 16) timed on this box's host cores.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IMG = 224
METRIC = "images/sec (224^2) at 1/2/4/8 B200; fused InfoNCE HBM GB/s vs roofline"
PER_GPU_BATCH = {"c2": 512, "c3": 256, "c4": 512, "c5": 1024}
if os.environ.get("PASSL_B200_BENCH_BATCH"):
    PER_GPU_BATCH = {k: int(os.environ["PASSL_B200_BENCH_BATCH"]) for k in PER_GPU_BATCH}


def workload_config(cfg, world):
    """The `config` object of the JSON line — identical for our arm and the reference arm."""
    B = PER_GPU_BATCH[cfg]
    common = {"global_batch": B * world, "per_gpu_batch": B, "parallelism": "dp%d" % world,
              "l2_policy": "inputs and activations of one step (>= 300 MB of images, tens of GB of activations) exceed the 126 MB L2"}
    if cfg == "c2":
        return dict(common, workload="simclr_r50_224_2views_bs%d_per_gpu (BASELINE configs[1]: global bs %d at 8 GPUs)" % (B, 8 * B),
                    backbone="ResNet-50 v1.5 (stem max-pool; reference ResNetsimclr variant available as stem_maxpool=False)",
                    views=2, head="NT-Xent+CO2, all-gathered negatives", optimizer="LARS",
                    images_counted="samples per step (each sample = two 224^2 views = 2 backbone passes)")
    if cfg == "c3":
        return dict(common, workload="moco_v2_r50_224_K65536_bs%d_per_gpu (BASELINE configs[2])" % B, backbone="ResNet-50 v1.5 x2 (query + EMA key)",
                    views=2, head="fused InfoNCE over the 65536-key queue (T=0.2)", optimizer="Momentum",
                    images_counted="samples per step (query view fwd+bwd, key view fwd)")
    if cfg == "c4":
        return dict(common, workload="mae_vit_b16_mask075_bs%d_per_gpu (BASELINE configs[3])" % B, backbone="ViT-B/16 encoder (49+1 tokens) + 8x512 decoder",
                    views=1, head="masked-patch MSE (norm_pix)", optimizer="AdamW", images_counted="images per step")
    return dict(common, workload="clip_vit_b16_text12x512_bs%d_pairs_per_gpu (BASELINE configs[4]: global 8192 at 8 GPUs)" % B,
                backbone="ViT-B/16 image tower + 12x512 causal text tower", views=1, head="symmetric InfoNCE (all-gathered features)",
                optimizer="AdamW", images_counted="image-text pairs per step")


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_burst=d["bf16_tflops"], bf16_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons DURING the timed region (every 0.2 s).  In-process NVML (nvidia_ml_py), initialised before the
    timed region starts: spawning `nvidia-smi` inside it cost 70-120 ms of stalled launches per run (the first invocation loads
    NVML and takes the driver lock) — visible as `value` < `e2e` in the first round-2 lines.  nvidia-smi is only the fallback."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.nvml, self.handle, self.max_mhz = None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            for _ in range(2):                   # every query once outside the timed region (the first calls take ~20 ms each)
                self._sample()
        except Exception:
            self.nvml = None

    def _sample(self):
        if self.nvml is not None:
            mhz = int(self.nvml.nvmlDeviceGetClockInfo(self.handle, self.nvml.NVML_CLOCK_SM))
            try:
                mask = int(self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                mask = int(self.nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            return mhz, self.max_mhz, [n for n, bit in self.REASONS if mask & bit]
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=5).stdout.strip()
        f = [x.strip() for x in o.split(",")]
        return int(f[0]), int(f[1]), [n for (n, _), v in zip(self.REASONS, f[2:6]) if v.lower().startswith("active")]

    def run(self):
        while not self.stop_flag:
            try:
                self.samples.append(self._sample())
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["unavailable"])
        sm = sorted(s[0] for s in self.samples)
        reasons = set()
        for s in self.samples:
            reasons.update(s[2])
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=self.samples[0][1], reasons=sorted(reasons), samples=len(self.samples),
                    source="nvml" if self.nvml is not None else "nvidia-smi")


# ----------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: oracle ports of the reference's training iterations on the host cores
# (the only places bench.py may execute oracle/)
# ----------------------------------------------------------------------------------------------------------------
def cpu_threads():
    """(logical host cores, threads given to torch).  torch-CPU convolutions stop scaling (and thrash) far below the core count of
    a GPU host, so the intra-op pool is capped (PASSL_B200_CPU_THREADS, default 32); both numbers are reported."""
    logical = os.cpu_count() or 1
    return logical, min(logical, int(os.environ.get("PASSL_B200_CPU_THREADS", "32")))


def _time_steps(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    ts.sort()
    return ts[len(ts) // 2], sum(ts) / len(ts)


def cpu_moco_c1(steps=10, warmup=3, bs=16):
    """BASELINE.md §3: configs[0] = MoCo v2 ResNet-50 (NonLinearNeckV1, T=0.2, K=65536, m=0.999), 2x224^2 views, bs 16, single
    process, full train_iter + Momentum step (lr 0.015, wd 1e-4), fp32 torch-CPU oracle port; median of `steps` after `warmup`."""
    import torch
    from oracle import moco_step as M
    logical, threads = cpu_threads()
    torch.set_num_threads(threads)
    st = M.init_params(0, K=65536)
    g = torch.Generator().manual_seed(1234)
    a = torch.randn(bs, 3, IMG, IMG, generator=g)
    b = torch.randn(bs, 3, IMG, IMG, generator=g)
    med, mean = _time_steps(lambda: M.train_step(st, a, b, lr=0.015, T=0.2, m=0.999, momentum=0.9, wd=1e-4), steps, warmup)
    # the unfused InfoNCE head alone (matmul -> concat -> /T -> CE), N = 16 and 256
    head = {}
    for n in (16, 256):
        q = torch.nn.functional.normalize(torch.randn(n, 128, generator=g), dim=1)
        k = torch.nn.functional.normalize(torch.randn(n, 128, generator=g), dim=1)
        hm, _ = _time_steps(lambda: M.infonce_head_unfused(q, k, st["queue"], 0.2), 10, 3)
        by = (2 * n * 128 + 128 * 65536) * 4 + 4 * n
        head["N%d" % n] = {"ms": hm * 1e3, "algorithmic_gbs": by / hm / 1e9}
    return {"value": bs / med, "unit": "images/s", "cores": threads, "host_logical_cores": logical, "thread_cap": threads,
            "kind": "port", "ms_per_step_median": med * 1e3, "ms_per_step_mean": mean * 1e3, "timed_steps": steps, "warmup_steps": warmup,
            "sample": "BASELINE configs[0]: MoCo v2 R50 bs %d x 2 views of 3x224x224, K=65536, full train_iter + Momentum step, torch-CPU fp32 "
                      "oracle port (oracle/moco_step.py); median of %d steps after %d warm-up" % (bs, steps, warmup),
            "infonce_head_unfused_cpu": head}


def cpu_workload_sample(cfg, steps, warmup):
    """A bounded sample of the benchmarked workload itself on the host cores: (images/s, s/step, threads, sample text)."""
    import torch
    logical, threads = cpu_threads()
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(1234)
    if cfg == "c2":
        from oracle import simclr_step as S
        n = 8
        p, vel = S.init_params(0), {}
        a, b = torch.randn(n, 3, IMG, IMG, generator=g), torch.randn(n, 3, IMG, IMG, generator=g)
        med, _ = _time_steps(lambda: S.train_step(p, vel, a, b, lr=1e-3), steps, warmup)
        return n / med, med, threads, "%d samples x 2 views of 3x224x224 per step (ResNet-50 + fc3 neck fwd+bwd, NT-Xent+CO2, LARS), oracle/simclr_step.py" % n
    if cfg == "c3":
        from oracle import moco_step as M
        n = 16
        st = M.init_params(0, K=65536)
        a, b = torch.randn(n, 3, IMG, IMG, generator=g), torch.randn(n, 3, IMG, IMG, generator=g)
        med, _ = _time_steps(lambda: M.train_step(st, a, b, lr=0.03), steps, warmup)
        return n / med, med, threads, "%d samples x 2 views of 3x224x224 per step (query fwd+bwd, EMA, key fwd, InfoNCE over K=65536, Momentum), oracle/moco_step.py" % n
    return None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    r = cpu_workload_sample(args.config, args.steps, args.warmup)
    if r is None:
        print(json.dumps({"impl": "reference", "unavailable": "no CPU port of the full %s training step (oracle/ holds forward twins of MAE / CLIP only)" % args.config}))
        return
    ips, dt, threads, sample = r
    logical, _ = cpu_threads()
    line = {"impl": "reference", "metric": METRIC, "value": ips, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args.config, world),
            "cpu_baseline": {"value": ips, "unit": "images/s", "cores": threads, "host_logical_cores": logical, "thread_cap": threads,
                             "kind": "port", "sample": sample + "; median of %d steps after %d warm-up" % (args.steps, args.warmup)},
            "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
def build_workload(cfg, dev, world, rank):
    """-> dict(step(inputs) -> loss tensor, make_inputs(gen) -> list of device tensors, stores)"""
    import torch
    from passl_b200.core import ParamStore
    from passl_b200.distributed import grad_sync, model_sync
    from passl_b200.modeling import build_model
    B = PER_GPU_BATCH[cfg]
    torch.manual_seed(0)
    it = [0]
    if cfg == "c2":
        from passl_b200.optimizer import LarsMomentumOptimizer
        model = build_model(dict(name="SimCLR", backbone=dict(name="ResNet", depth=50, with_pool=True),
                                 neck=dict(name="NonLinearNeckfc3", in_channels=2048, hid_channels=2048, out_channels=128,
                                           with_avg_pool=False),
                                 head=dict(name="SimCLRContrastiveHead", temperature=0.1, multi_rank=True))).to(dev)
        store = ParamStore(model.encoder)
        model_sync(model, (store,))
        base_lr = 0.075 * (B * world) ** 0.5            # learning_rate_scaling: sqrt  (configs/simclr/simclr_r50_IM.yaml)
        warm_steps = 10 * 1281167 // (B * world)
        opt = LarsMomentumOptimizer(store, lr=0.0)

        def step(inp):
            opt.set_lr(base_lr * min(1.0, (it[0] + 1) / warm_steps))
            opt.clear_grad()
            out = model(inp[0], inp[1])
            out["loss"].backward()
            grad_sync(store)
            opt.step()
            it[0] += 1
            return out["loss"]
        shapes = [((B, 3, IMG, IMG), torch.float32)] * 2
    elif cfg == "c3":
        from passl_b200.optimizer import Momentum
        from passl_b200.utils.config import get_config
        y = get_config(os.path.join(ROOT, "configs/moco/moco_v2_r50.yaml"))
        model = build_model(dict(y.model)).to(dev)
        store, sk = model.build_param_stores()
        model_sync(model, (store, sk))
        opt = Momentum(store, lr=0.03, momentum=0.9, weight_decay=1e-4)

        def step(inp):
            opt.clear_grad()
            out = model(inp[0], inp[1])
            out["loss"].backward()
            grad_sync(store)
            opt.step()
            return out["loss"]
        shapes = [((B, 3, IMG, IMG), torch.float32)] * 2
    elif cfg == "c4":
        from passl_b200.models import build_model as build_v25
        from passl_b200.optimizer import AdamW
        model = build_v25(dict(name="mae_vit_base_patch16", norm_pix_loss=True)).to(dev)
        store = ParamStore(model)
        model_sync(model, (store,))
        opt = AdamW(store, lr=1.5e-4, beta2=0.95, weight_decay=0.05, one_dim_no_decay=True)

        def step(inp):
            opt.clear_grad()
            loss, _, _ = model(inp[0], 0.75)
            loss.backward()
            grad_sync(store)
            opt.step()
            return loss
        shapes = [((B, 3, IMG, IMG), torch.float32)]
    else:
        from passl_b200.optimizer import AdamW
        arch = dict(name="CLIP", embed_dim=512, image_resolution=224, vision_layers=12, vision_width=768, vision_patch_size=16,
                    pre_norm=True, proj=True, patch_bias=False, context_length=77, vocab_size=49408, transformer_width=512,
                    transformer_heads=8, transformer_layers=12, qkv_bias=True)
        model = build_model(dict(name="CLIPWrapper", architecture=arch, head=dict(name="CLIPHead"))).to(dev)
        with torch.no_grad():                       # the reference's (2*depth)x projection init overflows bf16 activations at depth 12
            for blk in model.model.text.blocks:
                blk.proj.weight.mul_(1.0 / 24)
                blk.fc2.weight.mul_(1.0 / 24)
        store = ParamStore(model)
        model_sync(model, (store,))
        opt = AdamW(store, lr=1e-4, beta2=0.98, weight_decay=0.0005)

        def step(inp):
            opt.clear_grad()
            out = model(inp[0], inp[1])
            out["loss"].backward()
            grad_sync(store)
            opt.step()
            return out["loss"]
        shapes = [((B, 3, IMG, IMG), torch.float32), ((B, 77), torch.int64)]

    def make(device, gen=None, pinned=False):
        out = []
        for shp, dt in shapes:
            if dt == torch.float32:
                t = torch.randn(shp, device=device, generator=gen)
            else:   # token ids with the EOT id (vocab - 1) at a random position >= 1 (SURVEY §8d synthetic-input spec)
                t = torch.randint(1, 49407, shp, device=device, generator=gen)
                t[torch.arange(shp[0], device=device), torch.randint(1, shp[1], (shp[0],), device=device, generator=gen)] = 49407
            out.append(t.pin_memory() if pinned else t)
        return out
    return dict(step=step, make=make, B=B, store=store, model=model)


def bench_infonce(dev, pk):
    """Fused InfoNCE (MoCo C3 shape: N=256, K=65536, D=128, bf16) forward and backward against the HBM roofline: CUDA-graph replay
    of 8 calls over 8 different queues (134 MB > L2), L2 flushed between replays, events on the replay stream."""
    import torch
    from passl_b200 import kernels as K
    N, D, Kq, T = 256, 128, 65536, 0.2
    NQ = 8
    q = torch.nn.functional.normalize(torch.randn(N, D, device=dev), dim=1)
    kpos = torch.nn.functional.normalize(torch.randn(N, D, device=dev), dim=1)
    queues = [torch.nn.functional.normalize(torch.randn(Kq, D, device=dev), dim=1).bfloat16() for _ in range(NQ)]
    qb = q.bfloat16()
    out, lse, tgt, _ = K.infonce_tc_fwd(qb, queues[0], pos=kpos, scale=1 / T)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def graph_us(fn):
        gph = torch.cuda.CUDAGraph()
        st = torch.cuda.Stream()
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            fn(queues[0])
            with torch.cuda.graph(gph, stream=st):
                for qq in queues:
                    fn(qq)
        torch.cuda.synchronize()
        ts = []
        for _ in range(20):
            flush.zero_()                              # L2 flush between replays
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            gph.replay()
            e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e) / NQ)
        ts.sort()
        return ts[len(ts) // 2] * 1e3
    us_f = graph_us(lambda qq: K.infonce_tc_fwd(qb, qq, pos=kpos, scale=1 / T))
    us_b = graph_us(lambda qq: K.infonce_tc_bwd(qb, qq, lse, tgt, pos=kpos, scale=1 / T))
    alg = (2 * N * D + D * Kq) * 2 + 4 * N
    alg_b = D * Kq * 2 + 3 * N * D * 4
    traffic, tsrc = None, None
    tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(tp):
        rec = json.load(open(tp)).get("infonce_fwd_N256_K65536_D128")
        if rec:
            traffic, tsrc = rec["dram_bytes"], rec["source"]
    gbs = alg / us_f / 1e3
    return {"kernel": "infonce_tc_fwd_kernel<2> — ONE launch (MoCo C3: N=256, K=65536, D=128, bf16)", "bound": "hbm", "achieved": gbs,
            "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"], "traffic": traffic, "traffic_source": tsrc,
            "algorithmic_bytes": alg, "us_per_launch": us_f, "peak_source": pk["src"] + " (burst)",
            "backward": {"kernel": "infonce_tc_bwd_kernel<2> (+ zero fill of dq)", "us_per_launch": us_b, "algorithmic_bytes": alg_b,
                         "achieved": alg_b / us_b / 1e3, "frac": alg_b / us_b / 1e3 / pk["hbm_gbs"], "ratio_to_forward": us_b / us_f},
            "method": "CUDA graph of %d calls over %d different queues (working set %d MB > L2, flushed between replays), device time / %d"
                      % (NQ, NQ, NQ * D * Kq * 2 >> 20, NQ)}


DUMP_SAMPLE = 4 << 20          # elements kept of each dumped buffer: params + grads stay at 32 MB for every config


def dump_outputs(path, loss, store):
    """What the last timed step hands back, as float32 .npy files: `loss`, and the parameters it updated (`params`, the fp32
    master buffer of the ParamStore) with the gradients it updated them from (`grads`).  Buffers longer than DUMP_SAMPLE are
    sampled at positions drawn from a fixed seed.  The step itself sums split-K partials in a fixed order, so two runs with the
    same arguments write the same bits (c2, measured on a B200 at 1000 W)."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    idx = None
    if store.numel > DUMP_SAMPLE:
        pick = np.sort(np.random.default_rng(0).choice(store.numel, size=DUMP_SAMPLE, replace=False))
        idx = torch.from_numpy(pick).to(store.master.device)
    for name, t in (("loss", loss.detach().reshape(())), ("params", store.master), ("grads", store.grad)):
        if t.dim() and idx is not None:
            t = t[idx]
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints its version banner to STDOUT at NCCL_DEBUG=VERSION (the default of some launchers); the contract is ONE JSON line
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    from passl_b200 import _lib, kernels as K
    lib = _lib.load()
    pk = peaks()
    cfg = args.config
    wl = build_workload(cfg, dev, world, rank)
    B, step = wl["B"], wl["step"]
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    dev_in = wl["make"](dev, gen)
    host_in = wl["make"]("cpu", None, pinned=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    per_step = {}

    def timed(fn, steps, tag=None):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        s.record()
        for i in range(steps):
            loss = fn()
            marks[i].record()                      # per-step device times (diagnostic only; the metric is the whole region)
        e.record()
        barrier()
        if tag:
            prev, out = s, []
            for m in marks:
                out.append(round(prev.elapsed_time(m), 3))
                prev = m
            per_step[tag] = out
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), loss

    for _ in range(args.warmup):
        step(dev_in)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lib.passl_b200_launch_count()
    ms, loss = timed(lambda: step(dev_in), args.steps, tag="value")
    launches = lib.passl_b200_launch_count() - launches0
    sampler.stop_flag = True
    loss_val = float(loss.item())
    value = B * world * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, wl["store"])

    # ---- e2e: inputs from pinned host memory every step + D2H read of the loss -------------------------------------
    # The user-facing loop (engine/trainer.py IterLoader with prefetch) double-buffers the input: the H2D copy of step t+1 runs
    # on a copy stream under the compute of step t.  Every timed step still performs one full H2D copy of its inputs (K copies
    # inside the timed region for K steps) and one D2H read of its loss.
    copy_stream = torch.cuda.Stream()
    bufs = [[torch.empty_like(t) for t in dev_in] for _ in range(2)]
    ev_ready = [torch.cuda.Event(), torch.cuda.Event()]
    ev_free = [torch.cuda.Event(), torch.cuda.Event()]
    kk = [0]

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_free[i])
            for d, h in zip(bufs[i], host_in):
                d.copy_(h, non_blocking=True)
            ev_ready[i].record(copy_stream)

    def e2e_step():
        i = kk[0] & 1
        prefetch(i ^ 1)                                 # next step's inputs: overlaps this step's compute
        torch.cuda.current_stream().wait_event(ev_ready[i])
        l = step(bufs[i])
        ev_free[i].record()
        kk[0] += 1
        return l.item()                                 # D2H read of the step result (sync), like loop.py:86
    for e_ in ev_free:
        e_.record()
    prefetch(0)
    for _ in range(2):
        e2e_step()
    ms_e2e, _ = timed(e2e_step, args.steps, tag="e2e")
    e2e_value = B * world * args.steps / (ms_e2e / 1e3)
    h2d = sum(t.numel() * t.element_size() for t in host_in)

    line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": workload_config(cfg, world), "final_loss": loss_val,
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "ms_each_step": per_step}

    # ---- roofline of the tcgen05 launches: instrumented (untimed) step with CUDA events around every launch.
    #      Every rank runs the step (it contains collectives); only rank 0 reports.
    if rank == 0:
        line["clocks"] = sampler.summary()
    rec, desc = [], []
    orig = {n: getattr(K, n) for n in ("gemm", "conv2d_fwd", "conv2d_dgrad", "conv2d_wgrad")}

    def cost_of(name, a, kw, res):
        """(algorithmic FLOPs, algorithmic HBM bytes) of one launch: operands read once, output written once."""
        def nb(t):
            return 0 if t is None else t.numel() * t.element_size()
        extra = nb(kw.get("residual")) + nb(kw.get("aux")) + nb(kw.get("preact_out"))
        if name == "gemm":
            A, Bm = a[0], a[1]
            Kd = A.shape[0] if kw.get("a_t") else A.shape[1]
            acc = nb(res) if kw.get("accumulate") else 0
            return 2.0 * res.shape[0] * res.shape[1] * Kd, nb(A) + nb(Bm) + nb(res) + acc + extra
        if name == "conv2d_fwd":
            x, w = a[0], a[1]
            return 2.0 * res.numel() * w.shape[1] * w.shape[2] * w.shape[3], nb(x) + nb(w) + nb(res) + extra
        if name == "conv2d_dgrad":
            dy, w = a[0], a[1]
            acc = nb(res) if kw.get("accumulate") else 0
            return 2.0 * dy.numel() * w.shape[1] * w.shape[2] * w.shape[3], nb(dy) + nb(w) + nb(res) + acc
        x, dy, ws = a[0], a[1], a[2]
        return 2.0 * dy.numel() * ws[1] * ws[2] * ws[3], nb(x) + nb(dy) + 2 * nb(res)

    def wrap(name):
        def f(*a, **kw):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = orig[name](*a, **kw)
            e.record()
            rec.append((s, e) + cost_of(name, a, kw, r))
            desc.append("%s %s -> %s%s" % (name, " x ".join(str(tuple(t.shape)) for t in a[:2] if torch.is_tensor(t)), tuple(r.shape),
                                          "".join(" +" + k for k in ("bias", "residual", "aux", "preact_out", "col_stats", "act", "a_t",
                                                                      "b_t", "accumulate") if kw.get(k) is not None and kw.get(k) is not False)))
            return r
        return f
    from passl_b200.core import streams
    side_was = streams.ENABLED
    streams.ENABLED = False                         # serial launches: per-launch durations are not inflated by overlap
    for n in orig:
        setattr(K, n, wrap(n))
    step(dev_in)
    torch.cuda.synchronize()
    for n, f in orig.items():
        setattr(K, n, f)
    streams.ENABLED = side_was
    if rank == 0:
        # Every tcgen05 launch is classed by ITS binding roofline: t_tensor = FLOPs / bf16 peak, t_hbm = bytes / HBM peak.
        # ResNet-50's 1x1 convolutions at 56^2 / 28^2 have < 218 FLOP/B and are HBM-bound even on tensor cores.
        pk_tf, pk_bw = pk["bf16_sustained"] * 1e12, pk["hbm_gbs"] * 1e9
        cls = {"tensor": [0.0, 0.0, 0.0, 0], "hbm": [0.0, 0.0, 0.0, 0]}      # ms, flops, bytes, launches
        t_bind = 0.0
        for s_, e_, fl, by in rec:
            dt = s_.elapsed_time(e_)
            k = "tensor" if fl / pk_tf >= by / pk_bw else "hbm"
            c = cls[k]
            c[0] += dt; c[1] += fl; c[2] += by; c[3] += 1
            t_bind += max(fl / pk_tf, by / pk_bw) * 1e3
        tc_ms = cls["tensor"][0] + cls["hbm"][0]
        tc_flops = cls["tensor"][1] + cls["hbm"][1]
        table = os.environ.get("PASSL_B200_BENCH_LAUNCH_TABLE")
        if table:                                   # developer aid: one line per tcgen05 launch of the instrumented step
            with open(table, "w") as f:
                for (s_, e_, fl, by), d in zip(rec, desc):
                    dt = s_.elapsed_time(e_)
                    bind = max(fl / pk_tf, by / pk_bw) * 1e3
                    f.write("%8.1f us  %5.2f of %s roofline  %7.1f TF/s %7.0f GB/s  %s\n" % (
                        dt * 1e3, bind / dt if dt else 0.0, "tensor" if fl / pk_tf >= by / pk_bw else "hbm   ", fl / dt / 1e9,
                        by / dt / 1e6, d))
        traffic_db = {}
        tp = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tp):
            traffic_db = json.load(open(tp))

        def roof(k):
            ms_k, fl, by, nl = cls[k]
            if k == "tensor":
                ach, peak, unit = fl / (ms_k / 1e3) / 1e12 if ms_k else 0.0, pk["bf16_sustained"], "TFLOP/s"
            else:
                ach, peak, unit = by / (ms_k / 1e3) / 1e9 if ms_k else 0.0, pk["hbm_gbs"], "GB/s"
            # traffic: dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of this class at the benchmarked shape, taken
            # from an `ncu --set full` capture and recorded (with its source file) in profiles/r02_traffic.json; null when no
            # capture at this shape exists
            t = traffic_db.get("%s_%s" % (cfg, k))
            return {"kernel": "gemm_tcgen05_kernel (implicit-GEMM conv fwd/dgrad/wgrad + linears), %s-bound launches" % k,
                    "bound": k, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak if peak else 0.0,
                    "traffic": t["dram_bytes"] if t else None, "traffic_source": t["source"] if t else None,
                    "traffic_launch": t.get("launch") if t else None,
                    "peak_source": pk["src"] + " (sustained)" if k == "tensor" else pk["src"], "launches": nl,
                    "share_of_step": ms_k / (ms / args.steps)}
        dom = "hbm" if cls["hbm"][0] >= cls["tensor"][0] else "tensor"
        other = "tensor" if dom == "hbm" else "hbm"
        line["roofline"] = roof(dom)
        line["roofline"].update({
            "all_launches": len(rec), "all_share_of_step": tc_ms / (ms / args.steps), "flops_per_step": tc_flops,
            "all_tflops": tc_flops / (tc_ms / 1e3) / 1e12 if tc_ms else 0.0,
            "frac_of_binding_roofline_all_launches": t_bind / tc_ms if tc_ms else 0.0,
            "note": "one instrumented step (side stream off), CUDA events around each of the %d tcgen05 GEMM / conv launches; each is "
                    "classed by its binding roofline (algorithmic FLOPs / bf16 peak vs algorithmic bytes / HBM peak); this object "
                    "is the class with the larger time share, roofline_other the rest" % len(rec)})
        line["roofline_other"] = roof(other)
        line["roofline_infonce"] = bench_infonce(dev, pk)
        # ---- cpu_baseline (N=1 only): BASELINE.md §3 on this box's host cores ------------------------------------------
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_moco_c1()
            r = cpu_workload_sample(cfg, 3, 1)
            if r is not None:
                line["cpu_baseline"]["same_workload_sample"] = {"value": r[0], "unit": "images/s", "ms_per_step": r[1] * 1e3, "cores": r[2],
                                                                "sample": r[3] + "; median of 3 steps after 1 warm-up"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss, parameters and gradients of the last timed step "
                                                          "to DIR/<name>.npy (float32, sampled to <= 32 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints "NCCL version ..." from its C side at
    # communicator creation): everything goes to stderr while the run is in progress, the real stdout comes back for the result line.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    buf = io.StringIO()
    try:
        with contextlib.redirect_stdout(buf):
            if args.impl == "reference":
                run_reference(args)
            else:
                run_ours(args)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    out = [l for l in buf.getvalue().splitlines() if l.strip()]
    for l in out[:-1]:
        print(l, file=sys.stderr)
    if out:
        print(out[-1], flush=True)


if __name__ == "__main__":
    main()
