#!/usr/bin/env python
"""Benchmark of the Dino U-Net forward path (BASELINE.json metric: 2D 512x512 patches/sec, dinounet_l forward).

    python bench.py --gpus N --steps K --warmup W            # our arm (hand-written sm_100a kernels, C-ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU forward (oracle port) on host cores

One "step" = one forward over one batch of synthetic 3x512x512 patches (per-GPU batch fixed -> weak scaling).  For N>1
the driver launches one rank per GPU with torch.distributed.run; each rank runs its own batch shard (no data-path
collective inside the forward) and the step ends with ONE NCCL all-gather of the logits (SURVEY.md section 8e).
Rank 0 prints exactly one JSON line.
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


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-cuda"])
    ap.add_argument("--mode", default="infer", choices=["infer", "train"],
                    help="train = BASELINE.json config 3: forward + backward (Dice+CE) + SGD step of the trainable parameters")
    ap.add_argument("--model", default="dinounet_l", choices=["dinounet_s", "dinounet_b", "dinounet_l", "dinounet_7b"])
    ap.add_argument("--batch", type=int, default=32, help="patches per GPU per step")
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--vit-dtype", default="bf16")
    ap.add_argument("--rest-dtype", default="fp16")
    ap.add_argument("--query-dtype", default="fp32", choices=["16", "fp32"],
                    help="adapter query stream storage: fp32 = the reference's dtype (default), 16 = opt-in reduced storage")
    ap.add_argument("--train-gemm", default="tf32", choices=["tf32", "fp32"],
                    help="--mode train: matrix products of the trainable part on tcgen05 kind::tf32 (default) or the fp32 SIMT tier")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--gemm-pair", default="on", choices=["on", "off"], help="CTA-pair (cta_group::2) GEMM tiles (A/B switch)")
    ap.add_argument("--pdl", default="off", choices=["on", "off"], help="programmatic dependent launch across the plan (A/B switch; measured slower, default off)")
    ap.add_argument("--cpu-sample", type=int, default=8, help="patches in the bounded CPU-baseline sample (0 = skip)")
    ap.add_argument("--eager-steps", type=int, default=10, help="timed steps of the torch-eager CUDA arm at N=1 (0 = skip)")
    ap.add_argument("--ops-out", default="", help="write the per-kernel timing breakdown (JSON) here")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (rank 0): infer = "
                         "logits.npy (fp32 [n, classes, S, S]) and labels.npy (argmax as fp32 [n, S, S]) of n <= batch "
                         "patches picked by a fixed seed, as many as fit in 63 MiB; train = loss.npy (fp64 [1])")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm only")
    return a


DUMP_BYTES = 63 << 20


def dump_outputs(out_dir, arrays):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def sample_patches(logits, labels):
    """logits [B, C, S, S] fp32 and labels [B, S, S] uint8 (device) -> the same fp32 rows of both for a seeded subset of
    the batch that fits in DUMP_BYTES, as host arrays."""
    import numpy as np
    B, C, S, _ = logits.shape
    n = min(B, DUMP_BYTES // ((C + 1) * S * S * 4))
    idx = np.sort(np.random.default_rng(0).choice(B, n, replace=False)).tolist()
    return {"logits": logits[idx].float().cpu().numpy(), "labels": labels[idx].float().cpu().numpy()}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampling (B200_PROFILING.md clocks line).  Started before the warm-up (the tool
    needs ~1 s to emit its first line); `summary(t0, t1)` keeps only the samples that arrived inside the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self, t0, t1):
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.06 and r and r[0].isdigit()]
        if not rows:   # region shorter than the sampling period: fall back to the samples nearest to it
            rows = [r for t, r in self.rows if t0 - 0.5 <= t <= t1 + 0.5 and r and r[0].isdigit()]
        sm = sorted(int(r[0]) for r in rows)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == "Active" for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(rows[0][1]), "reasons": reasons, "samples": len(sm),
                "power_w_max": max(float(r[2]) for r in rows)}


def cpu_forward_patches_per_s(model, size, n_patches, threads=None):
    """The reference's algorithm on host cores: the oracle restatement (bit-identical to the reference forward,
    tests/test_oracle_vs_reference.py), fp32, eval, all host threads; bounded sample of the same workload."""
    import torch
    from oracle import dinounet_oracle as O
    threads = threads or min(16, os.cpu_count())   # measured on the GPU box: 16 threads is the fastest (32: 1.2x, 64: 2.8x, 128: 76x slower)
    torch.set_num_threads(threads)
    sd = O.make_state_dict(model, 2, seed=0)
    x = O.make_input(1, size, 0)
    O.forward(sd, model, x)  # warm-up (allocator, thread pools)
    t0 = time.perf_counter()
    for i in range(n_patches):
        O.forward(sd, model, O.make_input(1, size, i + 1))
    dt = time.perf_counter() - t0
    return n_patches / dt, threads, dt


class SyntheticParams(dict):
    """Reference-keyed random parameters generated ON THE DEVICE, tensor by tensor, when the engine packs them (same shapes
    and per-kind magnitudes as oracle.make_state_dict; values differ).  Only for the 7B benchmark line: materialising its
    6.95 B fp32 parameters in host memory once per rank (8 x 28 GB) is what this avoids; throughput does not depend on the
    weight values."""

    def __init__(self, model, num_classes, device):
        super().__init__()
        import torch
        from oracle import dinounet_oracle as O
        self._spec = {k: (shape, kind) for k, shape, kind in O.param_spec(model, num_classes)}
        self._dev, self._torch, self._O = device, torch, O

    def __contains__(self, k):
        return k in self._spec

    def get(self, k, default=None):
        return self[k] if k in self._spec else default

    def __getitem__(self, k):
        import math
        import zlib
        torch = self._torch
        shape, kind = self._spec[k]
        g = torch.Generator(device=self._dev).manual_seed(zlib.crc32(k.encode()) & 0x7FFFFFFF)
        rn = lambda: torch.randn(*shape, generator=g, device=self._dev, dtype=torch.float32)
        ru = lambda lo, hi: torch.rand(*shape, generator=g, device=self._dev, dtype=torch.float32) * (hi - lo) + lo
        if kind in ("w", "w_off"):
            return rn() / math.sqrt(max(1, math.prod(shape[1:]) if kind == "w" else shape[1]))
        if kind == "wT":
            return rn() / math.sqrt(shape[0])
        if kind in ("b", "b_off"):
            return rn() * 0.05
        if kind in ("nw",):
            return ru(0.8, 1.2)
        if kind in ("nb", "rm"):
            return rn() * 0.1
        if kind == "rv":
            return ru(0.5, 1.5)
        if kind == "ls":
            return ru(0.25, 0.75)
        if kind == "tok":
            return rn() * 0.5
        if kind == "bias_mask":
            D = shape[0] // 3
            return torch.cat([torch.ones(D), torch.zeros(D), torch.ones(D)]).to(self._dev)
        if kind == "periods":
            d4 = shape[0]
            return (100.0 ** (2 * torch.arange(d4, dtype=torch.float32) / (2 * d4))).to(self._dev)
        if kind == "nbt":
            return torch.zeros((), dtype=torch.int64, device=self._dev)
        return torch.zeros(*shape, device=self._dev)


class _EngineNet:
    """What StreamedPredictor needs from a network, around a bare ForwardEngine (7B line: no host-side nn.Module)."""

    def __init__(self, eng, dev):
        import torch
        self._eng, self._p = eng, torch.zeros(1, device=dev)

    def parameters(self):
        yield self._p

    def _get_engine(self, dev):
        return self._eng


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = max(1, a.steps)
    import torch
    from oracle import dinounet_oracle as O
    threads = min(16, os.cpu_count())   # fastest thread count for this forward on the GPU box's host (see cpu_forward_patches_per_s)
    torch.set_num_threads(threads)
    sd = O.make_state_dict(a.model, 2, seed=0)
    for _ in range(max(1, min(a.warmup, 1))):
        O.forward(sd, a.model, O.make_input(1, a.size, 0))
    t0 = time.perf_counter()
    for i in range(n):
        O.forward(sd, a.model, O.make_input(1, a.size, i + 1))   # one step = a bounded sample: 1 patch of the workload
    dt = time.perf_counter() - t0
    v = n / dt
    print(json.dumps({
        "impl": "reference", "metric": "2D patches/sec (512x512) forward", "value": v, "unit": "patches/s",
        "n_gpus": a.gpus, "steps": n, "warmup": a.warmup, "ms_per_step": 1e3 * dt / n, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{a.model} forward, {a.size}x{a.size}x3, per-GPU batch {a.batch} (reference arm: 1 patch/step sample)"},
        "cpu_baseline": {"value": v, "unit": "patches/s", "cores": threads, "kind": "port",
                         "sample": f"{n} x 1 patch {a.model}@{a.size} fp32 eval forward, oracle port of the reference"},
        "e2e": {"value": v, "unit": "patches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def eager_cuda_patches_per_s(model, B, S, steps, warmup, dev):
    import torch
    from oracle import dinounet_oracle as O
    sd = {k: v.to(dev) for k, v in O.make_state_dict(model, 2, seed=0).items()}
    xs = [O.make_input(B, S, 300 + i).to(dev) for i in range(2)]
    with torch.no_grad():
        for i in range(warmup):
            O.forward(sd, model, xs[i % 2], autocast_like_reference=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            O.forward(sd, model, xs[i % 2], autocast_like_reference=True)
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"value": B / ms * 1e3, "unit": "patches/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
            "what": "reference algorithm (oracle port) as torch eager on the same GPU: cuBLAS/cuDNN/SDPA kernels, outer fp16 / "
                    "inner bf16 autocast, inputs resident in HBM, batch %d" % B}


def run_train(a):
    """BASELINE.json configs[2]: `dinounet_b random-init, batch 64x512x512x3 synthetic, 1xB200 fwd+bwd (Dice+CE loss)`.
    One step = nnUNetTrainer.train_step: frozen ViT on the 16-bit tensor-core engine, trainable part forward + backward on the
    kernels of train_path.py (matrix products: tcgen05 kind::tf32 by default, --train-gemm fp32 = the SIMT parity tier), Dice+CE,
    (N > 1: one NCCL all-reduce of the gradients), clip + SGD-nesterov."""
    import torch
    import torch.distributed as dist
    os.environ.setdefault("DINOUNET_B200_ALLOW_RANDOM_BACKBONE", "1")
    import dinounet_b200
    from dinounet_b200 import config, lib
    from dinounet_b200.loss import DC_and_CE_loss
    from dinounet_b200.train_path import FusedSGD, train_step
    from oracle import dinounet_oracle as O
    rank, local, world = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    B, S, K, W = a.batch, a.size, a.steps, max(3, a.warmup)
    sd = O.make_state_dict(a.model, 2, seed=0)
    net = dinounet_b200.DinoUNet.from_config({"architecture": dict(config.DEFAULT_ARCHITECTURE)}, 3, 2, None, a.model)
    net.load_state_dict(sd, strict=True)
    net.train_gemm = a.train_gemm
    net = net.to(dev).train()
    crit = DC_and_CE_loss({"batch_dice": True, "smooth": 1e-5, "do_bg": False, "ddp": False}, {}, weight_ce=1, weight_dice=1)
    opt = FusedSGD(net.parameters(), lr=1e-2, weight_decay=3e-5)
    xs = [O.make_input(B, S, 100 + rank * 7 + i).to(dev) for i in range(2)]
    ts = [torch.randint(0, 2, (B, 1, S, S), generator=torch.Generator().manual_seed(i)).float().to(dev) for i in range(2)]
    n0 = lib.launch_count()
    with ClockSampler(local) as clk:
        for i in range(W):
            loss = train_step(net, crit, opt, xs[i % 2], ts[i % 2])
        torch.cuda.synchronize()
        launches_per_step = (lib.launch_count() - n0) // W
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for i in range(K):
            loss = train_step(net, crit, opt, xs[i % 2], ts[i % 2])
        e1.record()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = ms.item()
    if rank == 0:
        v = config.VARIANTS[a.model]
        fwd = O.algorithmic_flops_per_patch(a.model, S)
        T = (S // 16) ** 2 + config.N_PREFIX
        vit = v.depth * (2 * T * v.embed_dim * 3 * v.embed_dim + 4 * T * T * v.embed_dim + 2 * T * v.embed_dim ** 2 +
                         4 * T * v.embed_dim * v.ffn_hidden) + 2 * (S // 16) ** 2 * 768 * v.embed_dim
        flops = fwd + 2 * (fwd - vit)                       # backward of the trainable (non-ViT) part = 2x its forward
        value = world * B * K / (ms / 1e3)
        pk = peaks()
        tf32 = a.train_gemm == "tf32"
        print(json.dumps({
            "metric": "2D patches/sec (512x512) fwd+bwd (Dice+CE) + SGD step", "value": value, "unit": "patches/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": ("bf16/fp16 frozen ViT (tcgen05) + trainable part: tf32 tensor-core matrix products (tcgen05 kind::tf32, fp32 "
                      "accumulate), fp32 everything else" if tf32 else
                      "bf16/fp16 frozen ViT (tcgen05) + fp32 trainable part (SIMT forward/backward kernels)"), "data": "synthetic",
            "impl": "b200", "mode": "train",
            "config": {"workload": f"{a.model} train step, {S}x{S}x3, per-GPU batch {B}, Dice+CE, SGD-nesterov + clip 12",
                       "global_batch": B * world, "l2": "two resident batches alternated; the per-step working set is >> 126 MB L2",
                       "train_gemm": a.train_gemm,
                       "parallelism": f"dp{world} + 1 NCCL all-reduce of the gradients" if world > 1 else "single GPU"},
            "gpu_launches": K * launches_per_step, "kernels_per_step": launches_per_step, "loss": float(loss),
            "clocks": clk.summary(t0, t1),
            "roofline": ({"bound": "tensor", "achieved": value / world * flops / 1e12, "peak": pk["tflops"] / 2, "unit": "TFLOP/s",
                          "frac": value / world * flops / 1e12 / (pk["tflops"] / 2), "algorithmic_gflop_per_patch": flops / 1e9,
                          "peak_source": "half of the measured sustained bf16 peak (TF32 dense = 0.5 x bf16 on B200; no measured TF32 entry)",
                          "note": "whole step (frozen ViT + trainable forward/backward + loss + SGD) over the algorithmic FLOPs; the "
                                  "tf32 GEMM's operands go through registers (gathers no tensor map expresses), so it is bound by "
                                  "L2->SM operand traffic and LSU issue, not by the tensor pipe"} if tf32 else
                         {"bound": "fp32-simt", "achieved": value / world * flops / 1e12, "unit": "TFLOP/s",
                          "algorithmic_gflop_per_patch": flops / 1e9,
                          "note": "fp32 FMA peak of a B200 is ~72 TF/s (148 SMs x 128 lanes x 2 x 1.9 GHz); --train-gemm fp32 runs the "
                                  "trainable part on plain fp32 SIMT kernels (the gradient-parity tier)"}),
            "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}))
        if a.dump_outputs:
            import numpy as np
            dump_outputs(a.dump_outputs, {"loss": np.array([float(loss)], dtype=np.float64)})
    if world > 1:
        dist.destroy_process_group()


def run_reference_cuda_train(a):
    """The reference's training step as torch eager + autograd on the B200 (library kernels, the reference's autocast regime,
    its differentiable pure-PyTorch deformable-attention core instead of the CUDA extension): forward, Dice+CE, backward, clip,
    SGD-nesterov.  Informational arm beside `--mode train`."""
    import torch
    from oracle import dinounet_oracle as O
    from oracle import grad_oracle as G
    from oracle import loss_oracle as LO
    dev = torch.device("cuda", 0)
    sd = {k: v.to(dev) for k, v in O.make_state_dict(a.model, 2, seed=0).items()}
    keys = G.trainable_keys(a.model, 2)
    P = dict(sd)
    leaves = {k: P[k].clone().requires_grad_(True) for k in keys}
    for k, v in O.expand_aliases(leaves).items():
        P[k] = v
    opt = torch.optim.SGD(list(leaves.values()), lr=1e-2, weight_decay=3e-5, momentum=0.99, nesterov=True)
    v = O.VARIANTS[a.model]
    B, S = a.batch, a.size
    xs = [O.make_input(B, S, 100 + i).to(dev) for i in range(2)]
    ts = [torch.randint(0, 2, (B, 1, S, S), generator=torch.Generator().manual_seed(i)).float().to(dev) for i in range(2)]

    def step(i):
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.float16):
            logits = O.decoder_forward(P, O.encoder_forward(P, v, xs[i % 2], True, None), None)
            loss, _, _ = LO.dc_and_ce_loss(logits.float(), ts[i % 2], batch_dice=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(list(leaves.values()), 12)
        opt.step()
        return loss

    for i in range(max(2, a.warmup)):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(a.steps):
        loss = step(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    print(json.dumps({"impl": "reference-cuda", "mode": "train", "metric": "2D patches/sec (512x512) fwd+bwd (Dice+CE) + SGD step",
                      "value": B / ms * 1e3, "unit": "patches/s", "n_gpus": 1, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms,
                      "higher_is_better": True, "dtype": "fp16/bf16 autocast (torch eager + autograd, library kernels)", "data": "synthetic",
                      "config": {"workload": f"{a.model} train step, {S}x{S}x3, batch {B}"}, "loss": float(loss),
                      "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}))


def run_reference_cuda(a):
    """SURVEY.md section 8(d): the same oracle port run by PyTorch eager on the B200 in the reference's GPU precision
    regime (outer fp16 autocast, inner bf16 ViT, fp32 MSDA) — what a user gets from the reference code on this GPU
    (cuBLAS/cuDNN/SDPA library kernels).  Informational third arm; not part of the driver contract."""
    import torch
    from oracle import dinounet_oracle as O
    dev = torch.device("cuda", 0)
    sd = {k: v.to(dev) for k, v in O.make_state_dict(a.model, 2, seed=0).items()}
    x = O.make_input(a.batch, a.size, 0).to(dev)
    with torch.no_grad():
        for _ in range(max(1, a.warmup)):
            O.forward(sd, a.model, x, autocast_like_reference=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.steps):
            O.forward(sd, a.model, x, autocast_like_reference=True)
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    print(json.dumps({
        "impl": "reference-cuda", "metric": "2D patches/sec (512x512) forward", "value": a.batch / ms * 1e3,
        "unit": "patches/s", "n_gpus": 1, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms,
        "higher_is_better": True, "dtype": "fp16/bf16 autocast", "data": "synthetic",
        "config": {"workload": f"{a.model} forward, {a.size}x{a.size}x3, batch {a.batch}, torch eager (library kernels), "
                               "inputs resident in HBM"},
        "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}))


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)
    if a.impl == "reference-cuda":
        return run_reference_cuda_train(a) if a.mode == "train" else run_reference_cuda(a)
    if a.mode == "train":
        return run_train(a)
    import torch
    import torch.distributed as dist
    os.environ.setdefault("DINOUNET_B200_ALLOW_RANDOM_BACKBONE", "1")
    import dinounet_b200
    from dinounet_b200 import config, lib
    from dinounet_b200.parallel import AsyncGatherer
    from oracle import dinounet_oracle as O   # synthetic weights/inputs + FLOP model + cpu_baseline only

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib.load().b2u_set_option(3, 1 if a.gemm_pair == "off" else 0)
    lib.load().b2u_set_option(5, 1 if a.pdl == "on" else 0)

    B, S, K, W = a.batch, a.size, a.steps, max(3, a.warmup)
    if a.model == "dinounet_7b":
        from dinounet_b200.engine import ForwardEngine
        eng = ForwardEngine(a.model, SyntheticParams(a.model, 2, dev), 2, dev, a.vit_dtype, a.rest_dtype, query_dtype=a.query_dtype)
        net = _EngineNet(eng, dev)
    else:
        sd = O.make_state_dict(a.model, 2, seed=0)
        net = dinounet_b200.DinoUNet.from_config({"architecture": dict(config.DEFAULT_ARCHITECTURE)}, 3, 2, None, a.model)
        net.load_state_dict(sd, strict=True)
        net.vit_dtype, net.rest_dtype, net.query_dtype = a.vit_dtype, a.rest_dtype, a.query_dtype
        net = net.to(dev).eval()
        del sd
        eng = net._get_engine(dev)
    plan, bufs = eng.get_plan(B, S)
    n_kernels = len(plan.calls)
    # three resident input batches (3 x 100 MB at B=32 > 126 MB L2) rotated between steps; the per-step activation
    # working set (GBs) is itself >> L2, so no step starts with a warm cache.
    xs = [O.make_input(B, S, 100 + rank * 7 + i).to(dev) for i in range(3)]
    use_graph = not a.no_graph

    # the ONE collective of the step: NCCL all-gather of the fp16 logits (SURVEY.md section 8e: 33.5 MB/rank), enqueued on a
    # side stream right after the forward and double-buffered, so it overlaps the next step's kernels; every gather is
    # joined into the timed stream before the closing event.
    gat = AsyncGatherer(B * world, dev, torch.float16) if world > 1 else None

    def step(i):
        logits, labels = eng.forward(xs[i % 3], use_graph=use_graph)
        if gat is not None:
            gat.submit(logits)
        return logits, labels

    with torch.no_grad(), ClockSampler(local) as clk:
        for i in range(W):
            step(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_region0 = time.perf_counter()
        e0.record()
        for i in range(K):
            last = step(i)
        if gat is not None:
            gat.wait_all()
        e1.record()
        torch.cuda.synchronize()
        t_region1 = time.perf_counter()
        # the engine's output buffers are overwritten by the passes below: copy the sample out now
        dumped = sample_patches(*last) if a.dump_outputs and rank == 0 else None
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
        value = world * B * K / (ms / 1e3)

        # ---- e2e: the public API with HOST buffers — every step uploads its own input batch from pinned host memory and
        # downloads its logits to pinned host memory inside the timed region.  API: dinounet_b200.inference.StreamedPredictor
        # (copies on side streams overlap the kernels of the neighbouring steps; nothing is skipped).
        from dinounet_b200.inference import StreamedPredictor
        hx = [O.make_input(B, S, 200 + i).pin_memory() for i in range(3)]
        # N > 1: the gather happens on the device, straight from the forward's output and before / independent of this
        # rank's own D2H copy (no host round trip of the logits)
        pred = StreamedPredictor(net, use_graph=use_graph, gatherer=gat)
        acc = 0.0
        for y in pred.run(hx[i % 3] for i in range(3)):       # warm-up of the streamed path
            acc += float(y[0, 0, 0, 0])
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for y in pred.run(hx[i % 3] for i in range(K)):
            acc += float(y[0, 0, 0, 0])                           # touch the downloaded result on the host
        if gat is not None:
            gat.wait_all()
        torch.cuda.synchronize()
        te = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = world * B * K / te.item()

        # ---- per-kernel timing (one extra eager step with CUDA events around every launch, same stream)
        breakdown, roof, roof_hbm = {}, None, None
        if rank == 0:
            stream = torch.cuda.current_stream(dev)
            evs = []
            for name, fn, args in plan.calls:
                s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s_.record(stream)
                rc = fn(*args, __import__("ctypes").c_void_p(stream.cuda_stream))
                e_.record(stream)
                assert rc == 0, (name, lib.last_error())
                evs.append((name, s_, e_))
            torch.cuda.synchronize()
            fam = {}
            for name, s_, e_ in evs:
                base = name.split(".")[-1] if name[0] in "be" and name[1].isdigit() else name
                key = ("vit." + base) if name.startswith("b") and name[1].isdigit() else (
                    "extractor." + base if name.startswith("e") and name[1].isdigit() else name.split(".")[0])
                fam[key] = fam.get(key, 0.0) + s_.elapsed_time(e_)
            breakdown = dict(sorted(fam.items(), key=lambda kv: -kv[1]))
            # dominant kernel: the tcgen05 GEMM family of the ViT (qkv, proj, fc1, fc2) -> tensor-core roofline
            v = config.VARIANTS[a.model]
            T = B * ((S // 16) ** 2 + config.N_PREFIX)
            flops = v.depth * 2 * T * v.embed_dim * (3 * v.embed_dim + v.embed_dim + 2 * v.ffn_hidden)
            t_gemm = sum(fam.get(k, 0) for k in ("vit.qkv", "vit.proj", "vit.fc1", "vit.fc2"))
            pk = peaks()
            traffic, traffic_src = None, None
            tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
            tj = None
            if os.path.exists(tpath) and (a.model, B, S, a.vit_dtype) == ("dinounet_l", 32, 512, "bf16"):
                # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu pass over one step of exactly
                # this workload (tools/one_step.py + tools/ncu_table.py), averaged over the four ViT GEMM shapes
                tj = json.load(open(tpath))
                traffic = tj["vit_gemm_family_avg_per_launch"]
                traffic_src = "profiles/r02_traffic.json (ncu per-launch dram bytes, qkv/proj/fc1/fc2 of one step)"
            ach = flops / (t_gemm * 1e-3) / 1e12
            roof = {"bound": "tensor", "kernel": "gemm_tc2_kernel<256,EPI,ACT,%s> = persistent tcgen05 GEMM (ViT qkv/proj/fc1/fc2, %d launches/step)" % (a.vit_dtype, 4 * v.depth),
                    "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": ach / pk["tflops"], "traffic": traffic, "traffic_source": traffic_src,
                    "algorithmic_bytes_per_launch": (T * v.embed_dim * 2 * 2 + T * v.ffn_hidden * 2 * 2 + T * 3 * v.embed_dim * 2 + 2 * T * v.embed_dim * 8
                                                     + 2 * (4 * v.embed_dim * v.embed_dim + 2 * v.embed_dim * v.ffn_hidden)) / 4,
                    "peak_source": pk["src"] + " (bf16 sustained)", "share_of_step": t_gemm / sum(fam.values())}
            # top HBM-bound kernel: the 512^2 decoder conv (2f -> f channels, implicit GEMM, halo mode): reads the concat
            # buffer once, writes the conv output once (+ the per-(n,c) statistics); SURVEY.md section 8(d): bytes = (Cin+Cout)*2 B/px
            per_op = {n: s_.elapsed_time(e_) for n, s_, e_ in evs}
            f0 = eng.features[0]
            hb = B * S * S * (2 * f0 + f0) * 2 + 9 * 2 * f0 * f0 * 2
            t_conv = per_op.get("d2.conv0")
            if t_conv:
                ach_h = hb / (t_conv * 1e-3) / 1e9
                roof_hbm = {"bound": "hbm", "kernel": "gemm_tc2_kernel<32,...> conv3x3 halo mode (decoder stage 2 conv 0, %d->%d ch @ %dx%d)" % (2 * f0, f0, S, S),
                            "achieved": ach_h, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach_h / pk["hbm_gbs"],
                            "algorithmic_bytes_per_launch": hb, "us": t_conv * 1e3,
                            "traffic": (tj or {}).get("per_launch_dram_bytes", {}).get("d2.conv0"), "peak_source": pk["src"]}
            if a.ops_out:
                os.makedirs(os.path.dirname(a.ops_out) or ".", exist_ok=True)
                json.dump({"per_family_ms": breakdown, "per_op_ms": [(n, s_.elapsed_time(e_)) for n, s_, e_ in evs]},
                          open(a.ops_out, "w"), indent=1)

    if rank == 0:
        cpu = None
        if a.cpu_sample > 0 and a.model != "dinounet_7b":   # the 7B CPU forward needs ~30 GB and minutes: not a bounded sample
            v_cpu, cores, dt = cpu_forward_patches_per_s(a.model, S, a.cpu_sample)
            cpu = {"value": v_cpu, "unit": "patches/s", "cores": cores, "kind": "port",
                   "sample": f"{a.cpu_sample} x 1 patch {a.model}@{S} fp32 eval forward ({dt:.1f} s), oracle port of the reference"}
        eager = None
        if world == 1 and a.eager_steps > 0 and a.model != "dinounet_7b":
            # the reference algorithm as PyTorch eager on THIS GPU (library kernels, the reference's autocast regime):
            # the "reference already on Blackwell libraries" bar of SURVEY.md section 8(d), same box, same batch
            eng.clear_plans()
            torch.cuda.empty_cache()
            eager = eager_cuda_patches_per_s(a.model, B, S, a.eager_steps, 3, dev)
        total_flops = O.algorithmic_flops_per_patch(a.model, S)
        out = {
            "metric": "2D patches/sec (512x512) forward", "value": value, "unit": "patches/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": f"{a.vit_dtype} (ViT GEMMs/attention) + {a.rest_dtype} (adapter/FAPM/decoder), fp32 accumulate/residuals",
            "data": "synthetic", "impl": "b200",
            "config": {"workload": f"{a.model} forward, {S}x{S}x3, per-GPU batch {B}, random-init weights" + (" (generated on device)" if a.model == "dinounet_7b" else " (seed 0)"),
                       "global_batch": B * world, "parallelism": f"batch-sharded dp{world} + 1 NCCL all-gather of fp16 logits per step (side stream, double-buffered)" if world > 1 else "single GPU",
                       "l2": "3 resident input batches rotated (3x%.0f MB) and a per-step activation working set >> 126 MB L2" % (B * 3 * S * S * 4 / 1e6),
                       "cuda_graph": use_graph, "programmatic_dependent_launch": a.pdl == "on"},
            "e2e": {"value": e2e, "unit": "patches/s", "h2d_bytes_per_step": B * 3 * S * S * 4,
                    "d2h_bytes_per_step": B * 2 * S * S * 4},
            "gpu_launches": K * n_kernels, "kernels_per_step": n_kernels,
            "clocks": clk.summary(t_region0, t_region1),
            "roofline": roof, "roofline_hbm": roof_hbm, "cpu_baseline": cpu, "eager_cuda": eager,
            "model_tflops": value / world * total_flops / 1e12,
            "breakdown_ms": {k: round(v, 3) for k, v in list(breakdown.items())[:14]},
        }
        print(json.dumps(out))
        if dumped is not None:
            dump_outputs(a.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
