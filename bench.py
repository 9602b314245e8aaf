#!/usr/bin/env python
"""Benchmark of the TokenPacker projector hot path on B200 (contract: see the task brief / DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload projector|hd5|train] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one TokenPacker.forward over one batch of synthetic CLIP features per GPU.  Workload at every N:
BASELINE.json configs[1] per GPU — batch=64 crops of 576x1024 (+576x4096 multi-level) bf16 features, scale_factor=2,
hidden=4096 -> 9,216 compressed tokens per GPU per step (weak scaling: crops shard across ranks, no data-path
collective; weights replicated).  Prints ONE JSON line on rank 0.  Besides the contract's keys the line carries:
  sustained  the same step for >= 2 s with clocks sampled inside the region (power-capped regime), rated against the sustained peak
  hd5        (N > 1) BASELINE configs[4]: 256 HD crops, s=4, sharded across the ranks, packed per-image sequences on every rank:
             NCCL all-gather + assembly vs the fused peer-store GEMM, strong-scaling efficiency, bit-exactness vs one GPU
  train      (N = 1) forward + backward of the projector (the reference trains it: train.py:950-958) vs eager autograd
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "compressed_visual_tokens_per_sec"
UNIT = "tokens/s"
N_CROPS, SCALE, HIDDEN = 64, 2, 4096
TOKENS_PER_CROP = (24 // SCALE) ** 2


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_burst": p["bf16_tflops"], "bf16_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock / throttle-reason sampling DURING the timed region.  NVML is polled from a thread (~1 kHz, so that even a 20 ms
    region holds a dozen samples); nvidia-smi -lms (B200_PROFILING.md recipe) is the fallback.  Samples carry their own
    timestamps and are filtered to the timed window."""
    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.thread = [], None, None
        self.gpu_index = gpu_index
        self.samples = []          # (epoch, sm_mhz, max_mhz, power_w, reasons bitmask)
        self._stop = False
        self.nvml = None

    def _nvml_loop(self):
        nv, h = self.nvml
        while not self._stop:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                self.samples.append((time.time(), float(sm), self.max_mhz, pw, int(reasons)))
            except Exception:
                pass
            time.sleep(0.0008)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            # NVML enumerates physical GPUs: map through the PCI bus id of the CUDA device
            bus = torch.cuda.get_device_properties(self.gpu_index)
            h = None
            try:
                pci = f"{bus.pci_domain_id:08x}:{bus.pci_bus_id:02x}:{bus.pci_device_id:02x}.0"
                h = nv.nvmlDeviceGetHandleByPciBusId(pci.encode())
            except Exception:
                h = nv.nvmlDeviceGetHandleByIndex(self.gpu_index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.nvml = (nv, h)
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    @staticmethod
    def _epoch(ts: str):
        import datetime
        try:
            return datetime.datetime.strptime(ts.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self, t0=None, t1=None):
        """t0 / t1: time.time() bounds of the timed region."""
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        if self.nvml is not None:
            self._stop = True
            self.thread.join(timeout=2)
            nv = self.nvml[0]
            bits = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            parsed = [(t, sm, mx, pw, [("active" if r & bits[n] else "no") for n in names]) for t, sm, mx, pw, r in self.samples]
            source = "nvml"
        else:
            if self.proc is None:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock source available"]}
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            if self.thread is not None:
                self.thread.join(timeout=2)
            parsed = []
            for r in self.rows:
                f = [v.strip() for v in r.split(",")]
                if len(f) < 8:
                    continue
                try:
                    parsed.append((self._epoch(f[0]), float(f[1]), float(f[2]), float(f[3]), f[4:8]))
                except ValueError:
                    continue
            source = "nvidia-smi -lms 20"
        inside = [p for p in parsed if p[0] is not None and t0 is not None and t1 is not None and t0 <= p[0] <= t1]
        use = inside if len(inside) >= 3 else parsed
        if not use:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        reasons = set()
        for p in use:
            for name, v in zip(names, p[4]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median([p[1] for p in use])), "sm_max_mhz": float(max(p[2] for p in use)),
                "power_w_max": float(max(p[3] for p in use)), "samples": len(use), "in_timed_region": len(inside) >= 3,
                "source": source, "reasons": sorted(reasons)}


def cpu_reference_run(steps: int, warmup: int, crops: int):
    """The reference's own algorithm as PyTorch-CPU ops (oracle/torch_port.py, pinned to the reference fixtures) on all
    host threads, fp32 (the reference's CPU dtype).  One step = one forward over ``crops`` crops of the configs[1] workload
    (64 = the whole configs[1] batch); exactly ``steps`` steps are timed after ``warmup`` untimed ones."""
    from oracle import tokenpacker_oracle as tpo
    from oracle import torch_port
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    params = {k: torch.from_numpy(v) for k, v in tpo.make_params(HIDDEN, seed=0).items()}
    x0, xm = tpo.make_inputs(crops, seed=1234)
    x0, xm = torch.from_numpy(x0), torch.from_numpy(xm)
    # "all the host threads it can use": torch's intra-op pool degrades badly past the point where GEMM panels get too
    # thin (and on boxes whose cgroup quota is below the visible core count), so probe a few pool sizes up to every
    # visible core (on an 8-crop slice) and keep the FASTEST — the baseline is the best the reference's CPU path does on this host.
    cands = sorted({c for c in (avail, avail // 2, avail // 4, 32, 16, 8) if 1 <= c <= avail}, reverse=True)
    best_t, best_c = None, avail
    px0, pxm = x0[:8], xm[:8]
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            torch_port.forward(params, px0, pxm, SCALE)
            t0 = time.perf_counter()
            torch_port.forward(params, px0, pxm, SCALE)
            dt = time.perf_counter() - t0
            if best_t is None or dt < best_t:
                best_t, best_c = dt, c
    torch.set_num_threads(best_c)
    with torch.no_grad():
        for _ in range(warmup):
            torch_port.forward(params, x0, xm, SCALE)
        t0 = time.perf_counter()
        for _ in range(steps):
            torch_port.forward(params, x0, xm, SCALE)
        dt = (time.perf_counter() - t0) / steps
        # BASELINE configs[0]: ONE image (576x1024 feats, s=2 -> 144 tokens), the reference forward on the CPU, fp32
        torch_port.forward(params, x0[:1], xm[:1], SCALE)
        t0 = time.perf_counter()
        for _ in range(5):
            torch_port.forward(params, x0[:1], xm[:1], SCALE)
        single_ms = (time.perf_counter() - t0) / 5 * 1e3
    return {"value": crops * TOKENS_PER_CROP / dt, "unit": UNIT, "cores": int(torch.get_num_threads()), "kind": "port",
            "pinned": "oracle/torch_port.py is held to fixtures generated by the reference module itself (tests/golden, < 1e-6) and to the "
                      "reference's answers on seeded random cases (tests/test_reference_live.py)",
            "configs0_single_image_ms": single_ms,
            "sample": f"{crops} crops/step x {steps} steps of the configs[1] workload (fp32, torch {torch.__version__} CPU ops, "
                      f"oracle/torch_port.py restatement of builder.py:107-137; best of pool sizes {cands} on {avail} visible cores), {dt * 1e3:.1f} ms/step"}, dt


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (the pinned PyTorch-CPU port; /root/reference is
    not present on the GPU box and the reference is pure Python) on the host cores, same metric/config: the full configs[1]
    batch (64 crops) per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    crops = N_CROPS
    cb, dt = cpu_reference_run(args.steps, min(args.warmup, 3), crops)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "BASELINE configs[1] per GPU: batch=64 crops, CLIP-ViT-L/14-336 feats 576x1024 + 576x4096, "
                                   "scale_factor=2 (144 tok/crop), hidden=4096, bf16, seeded random weights",
                       "crops_per_gpu": crops, "note": "reference algorithm on the host CPU (fp32), one 64-crop batch per step; "
                                                       "a CPU run has no per-GPU sharding, so the value does not depend on n_gpus"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
# BASELINE configs[4]
# ----------------------------------------------------------------------------------------------------------------------
HD5_GRIDS = [(5, 5)] * 9 + [(3, 7)]                    # 9 x 26 + 22 = 256 crops (patch_num = 25 grids)


def hd5_measure(steps, warmup, rank, world, dev, dist, verify=True):
    """BASELINE configs[4]: TokenPacker-HD patch_num=25, scale_factor=4, 256 crops sharded across the ranks, per-image token
    sequences reassembled on every rank.  Two exchange implementations are timed: the NCCL all-gather + assembly baseline and
    the fused one (last GEMM TMA-stores straight into the packed rows of every peer).  Rank 0 additionally runs all 256 crops
    alone (the strong-scaling reference) and checks that the fused result is bit-identical to it.  tokens/s counts projected
    tokens (256 x 36), not separator rows."""
    from tokenpacker_b200 import TokenPackerB200
    from tokenpacker_b200 import synthetic as syn
    from tokenpacker_b200._lib import lib
    from tokenpacker_b200.dist import FusedGatherTokenPacker, ShardedTokenPacker, shard_bounds, shard_counts
    from tokenpacker_b200.hd import n_crops
    s, hidden = 4, HIDDEN
    total = sum(n_crops(a, b) for a, b in HD5_GRIDS)
    hb, wb = [a for a, _ in HD5_GRIDS], [b for _, b in HD5_GRIDS]
    model = TokenPackerB200(hidden_size=hidden, scale_factor=s)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in syn.synthetic_state_dict(hidden, seed=0).items()})
    model = model.to(dev, torch.bfloat16).eval()
    counts = shard_counts(total, world)

    def shard_inputs(r):
        lo, hi = shard_bounds(total, world, r)
        g = torch.Generator(device=dev).manual_seed(99 + r)
        return (torch.randn(hi - lo, 576, 1024, device=dev, generator=g).to(torch.bfloat16),
                torch.randn(hi - lo, 576, 4096, device=dev, generator=g).to(torch.bfloat16))

    x0, xm = shard_inputs(rank)
    g = torch.Generator(device=dev).manual_seed(7)
    sep = torch.randn(hidden, device=dev, generator=g).to(torch.bfloat16)
    ret = torch.randn(hidden, device=dev, generator=g).to(torch.bfloat16)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step):
        with torch.no_grad():
            for _ in range(warmup):
                step()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = lib.tp_launch_count()
            e0.record()
            for _ in range(steps):
                res = step()
            e1.record()
            l1 = lib.tp_launch_count()
            barrier()
            ms = e0.elapsed_time(e1) / steps
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, res, (l1 - l0) / steps

    rec = {"workload": "BASELINE configs[4]: TokenPacker-HD patch_num=25 grids, scale_factor=4 (36 tok/crop), 256 crops sharded across "
                       "ranks, packed per-image sequences on every rank", "crops": total, "tokens": total * 36, "steps": steps}
    if world == 1:
        ms, (packed, cu), launches = timed(lambda: model.forward_packed((x0, xm), hb, wb, sep, ret))
        rec.update({"one_gpu_ms": ms, "tokens_per_s": total * 36 / (ms * 1e-3), "packed_rows": int(cu[-1]), "tp_launches_per_step": launches})
        return rec
    nccl = ShardedTokenPacker(model)
    fused = FusedGatherTokenPacker(model)
    ms_n, (packed_n, cu), _ = timed(lambda: nccl.forward_hd((x0, xm), counts, hb, wb, sep, ret))
    packed_n = packed_n.clone()
    ms_f, (packed_f, _), launches = timed(lambda: fused.forward_hd((x0, xm), counts, hb, wb, sep, ret))
    packed_f = packed_f.clone()
    rec.update({"nccl_allgather_ms": ms_n, "fused_peer_store_ms": ms_f, "fused_vs_nccl": ms_n / ms_f,
                "tokens_per_s_fused": total * 36 / (ms_f * 1e-3), "tokens_per_s_nccl": total * 36 / (ms_n * 1e-3),
                "packed_rows": int(cu[-1]), "tp_launches_per_step_fused": launches,
                "exchange": "fused: the last GEMM's TMA stores write each crop's rows into the packed sequence of EVERY rank (peer-mapped "
                            "symmetric memory over NVLink), one symmetric-memory barrier, no assembly pass; nccl: all_gather_into_tensor + "
                            "scatter/fill assembly on every rank"})
    # where the fused step's time goes: this rank's share of the compute alone (packed rows of its own crops only), and the
    # cross-rank barrier alone
    lo_r, hi_r = shard_bounds(total, world, rank)
    n_local = hi_r - lo_r
    ms_local, _, _ = timed(lambda: model.forward_packed((x0, xm), [1] * n_local, [1] * n_local, sep, ret))
    buf, hdl = fused._buffers((int(cu[-1]), hidden), dev)
    ms_bar, _, _ = timed(lambda: hdl.barrier(channel=0))
    rec.update({"rank_local_compute_ms": ms_local, "symm_barrier_ms": ms_bar,
                "note": "rank_local_compute_ms = this rank's 1/N of the crops through forward_packed into a local buffer (max over ranks); "
                        "fused_peer_store_ms - rank_local_compute_ms = exchange + barrier + separator fill not hidden under compute"})
    # every rank checks that both exchanges gave it the same packed sequences
    same = torch.tensor([1 if torch.equal(packed_f, packed_n) else 0], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    rec["fused_equals_nccl_on_every_rank"] = bool(same.item())
    if verify:
        one_ms = None
        ok = None
        if rank == 0:
            parts = [shard_inputs(r) for r in range(world)]
            ax0, axm = torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])
            del parts
            with torch.no_grad():
                for _ in range(2):
                    ref, _ = model.forward_packed((ax0, axm), hb, wb, sep, ret)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                reps = max(3, min(steps, 10))
                e0.record()
                for _ in range(reps):
                    ref, _ = model.forward_packed((ax0, axm), hb, wb, sep, ret)
                e1.record()
                torch.cuda.synchronize()
            one_ms = e0.elapsed_time(e1) / reps
            ok = bool(torch.equal(ref, packed_f))
            del ax0, axm, ref
        dist.barrier()
        if rank == 0:
            rec.update({"one_gpu_ms": one_ms, "fused_bit_identical_to_one_gpu": ok,
                        "strong_scaling_efficiency_fused": one_ms / (world * ms_f), "strong_scaling_efficiency_nccl": one_ms / (world * ms_n)})
    return rec


def run_hd5(args, rank, world, dev, dist):
    rec = hd5_measure(args.steps, args.warmup, rank, world, dev, dist)
    if rank == 0:
        ms = rec.get("fused_peer_store_ms", rec.get("one_gpu_ms"))
        print(json.dumps({"metric": METRIC, "value": rec["tokens"] / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                          "dtype": "bf16", "data": "synthetic", "config": {"workload": rec["workload"]}, "hd5": rec}), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
# training step (SURVEY.md §8f N1)
# ----------------------------------------------------------------------------------------------------------------------
def train_measure(model, x0, xm, steps=10, warmup=3):
    """Forward + backward of the projector at the configs[1] batch (the reference trains this module through autograd,
    train.py:950-958) next to PyTorch eager autograd over the reference's op sequence (oracle/torch_port.py, bf16, same GPU)."""
    from tokenpacker_b200._lib import lib
    model.train()
    for p in model.parameters():
        p.requires_grad_(True)

    params = list(model.parameters())

    def step():
        for p in params:                 # what optimizer.zero_grad(set_to_none=True) (the default) does every training step: without
            p.grad = None                # it autograd ACCUMULATES into the old gradients (23 extra elementwise launches per step)
        out = model((x0, xm))
        out.backward(go)
        return out

    go = torch.randn(x0.shape[0], model.num_queries, model.hidden_size, device=x0.device).to(torch.bfloat16) * 0.01
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = lib.tp_launch_count()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    l1 = lib.tp_launch_count()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    peak_gib = torch.cuda.max_memory_allocated() / 2 ** 30
    for p in model.parameters():
        p.grad = None
    model.eval()
    rec = {"fwd_bwd_ms": ms, "steps": steps, "tp_launches_per_step": (l1 - l0) / steps, "peak_mem_gib": peak_gib,
           "what": "TokenPackerB200.forward + backward (tp_forward_train / tp_backward: every parameter gradient), N=64 crops, s=2, H=4096, bf16"}
    try:
        from oracle import torch_port
        pd = {k: v.detach().clone().requires_grad_(True) for k, v in model.state_dict().items()}

        def estep():
            for v in pd.values():
                v.grad = None
            o = torch_port.forward(pd, x0, xm, SCALE)
            o.backward(go)
        for _ in range(2):
            estep()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            estep()
        e1.record()
        torch.cuda.synchronize()
        rec["eager_autograd_ms"] = e0.elapsed_time(e1) / 5
        rec["eager_what"] = "PyTorch eager autograd over oracle/torch_port.py (the reference's op sequence), bf16, same GPU, same weights and inputs"
        del pd
    except Exception as e:          # the baseline is context; never let it take the line down
        rec["eager_autograd_ms"] = None
        rec["eager_error"] = repr(e)[:200]
    torch.cuda.empty_cache()
    return rec


def hd_tile_measure(dev, peaks):
    """BASELINE configs[3]'s front end: the tiling block (train.py:695-731) for a batch of 32 seeded image sizes, patch_num = 9
    (231 crops), as ONE launch of the batched kernel.  HBM-bound: algorithmic bytes = every source pixel read once + every crop
    pixel written once."""
    from tokenpacker_b200 import hd_tile_batch
    g = torch.Generator().manual_seed(0)
    hs = torch.randint(224, 1345, (32,), generator=g).tolist()
    ws = torch.randint(224, 1345, (32,), generator=g).tolist()
    gg = torch.Generator(device=dev).manual_seed(3)
    imgs = [torch.randn(3, h, w, device=dev, generator=gg) for h, w in zip(hs, ws)]
    from tokenpacker_b200._lib import lib, check
    for _ in range(3):
        crops, hb, wb = hd_tile_batch(imgs, 9)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    e0.record()
    for _ in range(reps):
        crops, hb, wb = hd_tile_batch(imgs, 9)
    e1.record()
    torch.cuda.synchronize()
    ms_call = e0.elapsed_time(e1) / reps
    # the kernel on its own: the same launch re-issued through the C ABI with the tables already on the device
    crops, hb, wb, (tables, table_off, n_crops) = hd_tile_batch(imgs, 9, _return_launch=True)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for _ in range(3):
        check(lib.tp_hd_tile_batch(tables.data_ptr(), tables.data_ptr() + table_off, n_crops, crops.data_ptr(), stream), "tp_hd_tile_batch")
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        check(lib.tp_hd_tile_batch(tables.data_ptr(), tables.data_ptr() + table_off, n_crops, crops.data_ptr(), stream), "tp_hd_tile_batch")
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    bytes_alg = sum(3 * h * w * 4 for h, w in zip(hs, ws)) + crops.numel() * 4
    return {"what": "hd_tile_batch: 32 images (seeded sizes 224..1344), patch_num=9 -> %d crops [3,336,336] fp32, one launch, thumbnails fused" % crops.shape[0],
            "ms": ms, "ms_public_call": ms_call,
            "includes": "ms: the tp_hd_tile_batch launch alone (tables resident); ms_public_call: hd_tile_batch() incl. the host plan for 32 images and "
                        "its one asynchronous table upload (host-bound at this batch size)",
            "algorithmic_bytes": bytes_alg,
            "achieved_gbs": bytes_alg / (ms * 1e-3) / 1e9, "peak_gbs": peaks["hbm_gbs"], "frac": bytes_alg / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"]}


DUMP_ROWS = 2048                 # of the N_CROPS x TOKENS_PER_CROP = 9,216 output rows: 2048 x 4096 fp32 = 32 MiB


def dump_outputs(out, path):
    """What the timed forward returned in its last step, for comparing two builds output for output: a fixed seeded sample
    of DUMP_ROWS whole token rows (ascending row order, fp32) and the fp64 sum of every row of the full output."""
    os.makedirs(path, exist_ok=True)
    rows = out.reshape(-1, out.shape[-1])
    pick = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    np.save(os.path.join(path, "out_sampled_rows.npy"), rows[pick.to(rows.device)].float().cpu().numpy())
    np.save(os.path.join(path, "out_row_sums.npy"), out.double().sum(dim=-1).cpu().numpy())


def bind_numa(local_rank):
    try:
        from tokenpacker_b200.numa import bind_to_gpu_node
        return bind_to_gpu_node(local_rank)
    except Exception as e:          # placement is an optimisation, never a failure
        return {"bound": False, "error": repr(e)[:200]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="projector", choices=["projector", "hd5", "train"],
                    help="projector: BASELINE configs[1] (default, the driver's line; carries hd5 at N > 1 and train at N = 1 as records); "
                         "hd5: configs[4] HD reassembly across ranks as its own line; train: forward + backward as its own line")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU baseline leg (profiling runs)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer end-to-end leg (profiling runs)")
    ap.add_argument("--no-extras", action="store_true", help="skip the sustained / hd5 / train / eager records (profiling runs)")
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="projector workload: after the timed steps, write rank 0's output of the last timed step to DIR/*.npy "
                         "(a seeded sample of whole rows, plus every row's sum)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "projector"):
        ap.error("--dump-outputs applies to --impl ours --workload projector")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference(args)
        return

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch multi-GPU runs with torch.distributed.run (one process per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a B200: tokenpacker_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # host placement BEFORE any pinned allocation: this rank's CPU threads (and therefore its first-touch pinned buffers) go to the
    # NUMA node its GPU hangs off — the e2e leg is PCIe/host-memory bound
    orig_affinity = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa = bind_numa(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from tokenpacker_b200 import TokenPackerB200
    from tokenpacker_b200 import synthetic as syn       # seeded synthetic weights + algorithmic FLOP/byte model
    from tokenpacker_b200._lib import lib

    if args.workload == "hd5":
        run_hd5(args, rank, world, dev, dist)
        if dist is not None:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    torch.manual_seed(0)
    model = TokenPackerB200(hidden_size=HIDDEN, scale_factor=SCALE)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in syn.synthetic_state_dict(HIDDEN, seed=0).items()})
    model = model.to(dev, torch.bfloat16).eval()
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    x0 = torch.randn(N_CROPS, 576, 1024, device=dev, generator=g).to(torch.bfloat16)
    xm = torch.randn(N_CROPS, 576, 4096, device=dev, generator=g).to(torch.bfloat16)

    if args.workload == "train":
        rec = train_measure(model, x0, xm, steps=args.steps, warmup=args.warmup)
        if rank == 0:
            print(json.dumps({"metric": "projector_train_step_ms", "value": rec["fwd_bwd_ms"], "unit": "ms", "n_gpus": world, "steps": rec["steps"],
                              "warmup": args.warmup, "ms_per_step": rec["fwd_bwd_ms"], "higher_is_better": False, "scaling": "weak", "dtype": "bf16",
                              "data": "synthetic", "config": {"workload": "configs[1] batch, forward + backward"}, "train": rec}), flush=True)
        if dist is not None:
            dist.destroy_process_group()
        return

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(n_steps, sample_clocks):
        """Exactly n_steps forwards bracketed by barrier + synchronize; device-timed, max over ranks."""
        sampler = ClockSampler(local_rank) if (sample_clocks and rank == 0) else None
        if sampler is not None:
            sampler.start()
            time.sleep(0.05)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lib.tp_launch_count()
        t_wall0 = time.time()
        e0.record()
        for _ in range(n_steps):
            o = model((x0, xm))
        e1.record()
        l1 = lib.tp_launch_count()
        barrier()
        t_wall1 = time.time()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        clocks = sampler.stop(t_wall0, t_wall1) if sampler is not None else None
        return ms / n_steps, clocks, l1 - l0, o

    flops_step = syn.flops_per_crop(SCALE, HIDDEN) * N_CROPS
    bytes_step = syn.bytes_per_crop(SCALE, HIDDEN) * N_CROPS + syn.weight_bytes(HIDDEN)
    tokens_per_step = N_CROPS * TOKENS_PER_CROP * world

    # ------------------------------------------------------------------ device-resident throughput ("value")
    with torch.no_grad():
        for _ in range(args.warmup):
            out = model((x0, xm))
        ms_per_step, clocks, launches, out = timed_steps(args.steps, True)
    value = tokens_per_step / (ms_per_step * 1e-3)
    assert torch.isfinite(out.float()).all()
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    region_s = ms_per_step * args.steps * 1e-3
    regime = "sustained" if region_s >= 1.0 else "burst"

    # ------------------------------------------------------------------ the same step, sustained (power-capped regime)
    sustained = None
    if not args.no_extras:
        n_sus = max(args.steps, int(math.ceil(args.sustained_seconds / (ms_per_step * 1e-3))))
        with torch.no_grad():
            ms_sus, clocks_sus, _, _ = timed_steps(n_sus, True)
        tf = flops_step / (ms_sus * 1e-3) / 1e12
        sustained = {"steps": n_sus, "ms_per_step": ms_sus, "value": tokens_per_step / (ms_sus * 1e-3), "unit": UNIT, "seconds": ms_sus * n_sus * 1e-3,
                     "achieved_tflops": tf, "peak": peaks["bf16_sustained"], "frac": tf / peaks["bf16_sustained"],
                     "peak_source": peaks["source"] + ": sustained figure (this region is long enough to sit under the power cap)",
                     "clocks": clocks_sus}

    # ------------------------------------------------------------------ end to end through the public API, HOST buffers
    e2e = None
    if not args.no_e2e:
        hx0 = x0.cpu().pin_memory()
        hxm = xm.cpu().pin_memory()
        hout = torch.empty((N_CROPS, TOKENS_PER_CROP, HIDDEN), dtype=torch.bfloat16).pin_memory()
        with torch.no_grad():
            for _ in range(2):
                model.forward_host((hx0, hxm), out=hout, chunk_crops=8)
            barrier()
            t0 = time.perf_counter()
            e2e_steps = min(args.steps, 100)       # PCIe-bound at ~7.4 ms/step: 100 steps are plenty
            for _ in range(e2e_steps):
                model.forward_host((hx0, hxm), out=hout, chunk_crops=8)      # synchronous: result is in hout on return
            torch.cuda.synchronize()
            dt_local = (time.perf_counter() - t0) / e2e_steps
        dt = dt_local
        per_rank = [dt_local]
        if dist is not None:
            t = torch.tensor([dt_local], device=dev)
            gathered = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(gathered, t)
            per_rank = [float(v.item()) for v in gathered]
            dt = max(per_rank)
        assert torch.equal(hout, out.cpu()), "host-buffer path and device path disagree"
        h2d = int(hx0.numel() * 2 + hxm.numel() * 2)
        e2e = {"value": tokens_per_step / dt, "unit": UNIT,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(hout.numel() * 2),
               "ms_per_step": dt * 1e3, "steps_timed": e2e_steps,
               "per_rank_ms": [round(v * 1e3, 3) for v in per_rank], "per_rank_h2d_gbs": [round(h2d / v / 1e9, 1) for v in per_rank],
               "numa": numa,
               "api": "TokenPackerB200.forward_host -> tp_forward_host (pinned host buffers, 8-crop chunks with a tapered tail, cached copy streams)"}
        del hx0, hxm, hout

    # ------------------------------------------------------------------ roofline of the dominant kernel
    # tp_gemm2_kernel on its largest launch: h_kv = GELU(xm . [W_k0;W_v0]^T + b)  (M=36864, N=2048, K=4096), 45% of the
    # step's FLOPs.  Timed live with CUDA events on the launching stream, 10 back-to-back launches after 3 warm-ups (a burst
    # measurement, rated against the burst peak).
    roofline = None
    if rank == 0:
        from tokenpacker_b200.kernels import gemm_bf16
        m_, n_, k_ = N_CROPS * 576, 2048, 4096
        wkv = torch.cat([model.k_proj_1[0].weight, model.v_proj_1[0].weight], 0).detach().contiguous()
        bkv = torch.cat([model.k_proj_1[0].bias, model.v_proj_1[0].bias], 0).detach().float()
        a2 = xm.reshape(m_, k_)
        c2 = torch.empty((m_, n_), dtype=torch.bfloat16, device=dev)
        for _ in range(3):
            gemm_bf16(a2, wkv, bias=bkv, gelu=True, out=c2)
        torch.cuda.synchronize()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        r0.record()
        for _ in range(reps):
            gemm_bf16(a2, wkv, bias=bkv, gelu=True, out=c2)
        r1.record()
        torch.cuda.synchronize()
        k_ms = r0.elapsed_time(r1) / reps
        flops = 2.0 * m_ * n_ * k_
        achieved = flops / (k_ms * 1e-3) / 1e12
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        step_tf = flops_step / (ms_per_step * 1e-3) / 1e12
        step_peak = peaks["bf16_sustained"] if regime == "sustained" else peaks["bf16_burst"]
        roofline = {"bound": "tensor", "kernel": "tp_gemm2_kernel (CTA-pair tcgen05 GEMM; largest launch: k/v_proj.0, M=36864 N=2048 K=4096, bias+GELU epilogue)",
                    "achieved": achieved, "peak": peaks["bf16_burst"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16_burst"],
                    "peak_source": peaks["source"] + ": burst figure (this kernel is timed alone, 10 launches)",
                    "traffic": traffic, "ms_per_launch": k_ms, "flops_per_launch": flops,
                    "step": {"what": f"whole step of the timed `value` region ({args.steps} steps, {region_s * 1e3:.0f} ms: a {regime} measurement, rated against the "
                                     f"{regime} peak; the >= 2 s run is in `sustained`)",
                             "achieved_tflops": step_tf, "peak": step_peak, "regime": regime, "frac": step_tf / step_peak,
                             "flops_alg_per_step": flops_step,
                             "hbm_gbs": bytes_step / (ms_per_step * 1e-3) / 1e9, "hbm_frac": bytes_step / (ms_per_step * 1e-3) / 1e9 / peaks["hbm_gbs"]}}
        del a2, c2, wkv

    # ------------------------------------------------------------------ BASELINE configs[4] across the ranks
    hd5 = None
    if world > 1 and not args.no_extras:
        hd5 = hd5_measure(max(5, min(args.steps, 50)), 5, rank, world, dev, dist)

    # ------------------------------------------------------------------ the reference's op sequence, eager on THIS GPU
    # (SURVEY.md §8d "second baseline": the reference ships no Blackwell kernel, so its own ATen/cuBLAS eager path on the same
    # box is the real bar.)  oracle/torch_port.py = the reference forward as PyTorch ops in the reference's order; bf16.
    gpu_eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.no_extras:
        from oracle import torch_port
        pd = {k: v.detach() for k, v in model.state_dict().items()}
        with torch.no_grad():
            for _ in range(3):
                ref_out = torch_port.forward(pd, x0, xm, SCALE)
            torch.cuda.synchronize()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(20):
                ref_out = torch_port.forward(pd, x0, xm, SCALE)
            g1.record()
            torch.cuda.synchronize()
        g_ms = g0.elapsed_time(g1) / 20
        diff = (ref_out.float() - out.float())
        gpu_eager = {"value": N_CROPS * TOKENS_PER_CROP / (g_ms * 1e-3), "unit": UNIT, "ms_per_step": g_ms, "kind": "port",
                     "what": "oracle/torch_port.py (reference op sequence: F.linear/gelu/layer_norm/interpolate/multi_head_attention_forward) "
                             "eager bf16 on the same B200, same weights and inputs",
                     "rel_rms_vs_ours": float(diff.pow(2).mean().sqrt() / ref_out.float().pow(2).mean().sqrt())}
        del ref_out

    # ------------------------------------------------------------------ BASELINE configs[0]: one image through the public forward
    single = None
    if rank == 0:
        with torch.no_grad():
            for _ in range(5):
                model((x0[:1], xm[:1]))
            torch.cuda.synchronize()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(50):
                model((x0[:1], xm[:1]))
            s1.record()
            torch.cuda.synchronize()
        single = {"gpu_ms": s0.elapsed_time(s1) / 50, "what": "configs[0]: 1 image, s=2 -> 144 tokens, TokenPackerB200.forward, 50 calls back to back"}

    # ------------------------------------------------------------------ training step (N = 1 only)
    train = None
    if rank == 0 and world == 1 and not args.no_extras:
        train = train_measure(model, x0, xm, steps=10)

    hd_tile = None
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            hd_tile = hd_tile_measure(dev, peaks)
        except Exception as e:
            hd_tile = {"error": repr(e)[:300]}

    # ------------------------------------------------------------------ CPU baseline (rank 0, N=1 only)
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # in a child process with the ORIGINAL cpu affinity: this process (and the thread pools it has spawned) is pinned to one
        # NUMA node for the host-buffer leg, and the reference's CPU path must get every host core
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "10", "--warmup", "1"],
                               capture_output=True, text=True, timeout=900,
                               preexec_fn=(lambda: os.sched_setaffinity(0, orig_affinity)) if orig_affinity else None)
            cpu_baseline = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as e:
            cpu_baseline = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"CPU baseline leg failed: {e!r}"[:300]}
        if single is not None:
            single["cpu_reference_ms"] = cpu_baseline.get("configs0_single_image_ms")

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic",
                "config": {"workload": "BASELINE configs[1] per GPU: batch=64 crops, CLIP-ViT-L/14-336 feats 576x1024 + 576x4096, "
                                       "scale_factor=2 (144 tok/crop), hidden=4096, bf16, seeded random weights",
                           "crops_per_gpu": N_CROPS, "tokens_per_step": tokens_per_step,
                           "l2": "inputs 377 MB/step per GPU exceed the 126 MB L2 (no explicit flush needed)",
                           "parallelism": f"dp{world} (crops sharded, weights replicated, no data-path collective)"},
                "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "sustained": sustained, "hd5": hd5,
                "train": train, "hd_tile": hd_tile, "cpu_baseline": cpu_baseline, "gpu_eager_baseline": gpu_eager, "configs0_single_image": single}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
