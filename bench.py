#!/usr/bin/env python
"""bench.py -- attention-forward TFLOP/s on B200 (the one hot path), per the driver contract.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload (config.workload): BASELINE.json configs[4], the configuration the metric's "1/2/4/8 B200"
clause is quoted on -- B=64 H=32 S=4096 D=128 bf16 causal, sharded over (B*H).  It fits one GPU
(Q,K,V,O = 8.6 GB), so N=1 runs ALL of it and N>1 splits the batch: total work fixed => "strong" scaling.
A step = one forward pass over the whole job: every rank runs the sm_100a kernel on its B/N batches and,
for N>1, the O shards are all-gathered (NCCL) so every rank ends the step holding the full O.

Printed JSON (rank 0, one line):
  value        whole-job TFLOP/s, F = 2*B*H*S^2*D (BASELINE.json's "effective FLOPs"; equals the usual
               causal count 4*B*H*S^2*D/2), inputs resident in HBM, CUDA-event time, max over ranks.
  e2e          the same metric through the C ABI host-buffer call tfa_fwd_host(): pinned HOST q/k/v in,
               HOST out/lse back, copies inside the timed region.
  roofline     tensor-core bound: achieved = F_per_launch / mean kernel time (CUDA events on the launch
               stream, measured live here), peak = MEASURED_PEAKS.json bf16_tflops (burst).
  cpu_baseline the reference's own C++ CPU attention (oracle/_ref, compiled unmodified) timed on this box's
               host cores on a bounded head-sample of the same workload (rank 0, N=1 only).
  configs      BASELINE.json configs[1..3] timed the same way (N=1 only), for the headline table.
`--impl reference` times only that CPU path (all host threads) on the same config/metric/unit.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "tiny-flash-attention_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

WORKLOAD = {"name": "cfg5: B=64 H=32 S=4096 D=128 bf16 causal, sharded over (B*H)", "B": 64, "H": 32, "S": 4096,
            "D": 128, "causal": True}
EXTRA_CONFIGS = {
    "cfg2: B=4 H=16 S=2048 D=64 bf16 non-causal": (4, 16, 2048, 64, False),
    "cfg3: B=4 H=32 S=4096 D=128 bf16 causal": (4, 32, 4096, 128, True),
    "cfg4: B=1 H=32 S=16384 D=128 bf16 causal": (1, 32, 16384, 128, True),
}
FALLBACK_PEAK_TFLOPS = 1590.0   # /opt/skills/guides/B200_PROFILING.md fallback
METRIC = "attention TFLOPs/s (bf16, seqlen\u00d7head_dim) at 1/2/4/8 B200 vs roofline"   # BASELINE.json's metric, verbatim
try:
    METRIC = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "BASELINE.json")))["metric"]
except Exception:  # noqa: BLE001  (file absent: keep the literal above)
    pass


def flops_effective(B, H, S, D):
    return 2.0 * B * H * S * S * D


def flops_std(B, H, S, D, causal):
    return 4.0 * B * H * S * S * D * (0.5 if causal else 1.0)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["bf16_tflops"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "measured"
        except Exception:  # noqa: BLE001
            pass
    return FALLBACK_PEAK_TFLOPS, 1400.0, "fallback"


class ClockSampler:
    """Samples SM clock and throttle reasons DURING the timed region (NVML), as the profiling recipe asks."""

    def __init__(self, index=0, period=0.004):
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:  # noqa: BLE001
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=1.0)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# --------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own CPU attention on the host cores
# --------------------------------------------------------------------------------------------
def cpu_reference_runner():
    """Returns (fn(q,k,v,causal,scale)->out, kind, cores). Prefers oracle/_ref (the reference's C++ compiled
    unmodified); falls back to the C oracle port of the same row-wise algorithm."""
    from oracle import oracle as orc
    import torch

    cores = os.cpu_count() or 1
    ker = orc.load_ref_kernels()
    if ker is not None:
        torch.set_num_threads(cores)
        return (lambda q, k, v, c, s: ker.flash_attn(q, k, v, c, s)), "reference", cores
    return (lambda q, k, v, c, s: torch.from_numpy(orc.rowwise_online(q.numpy(), k.numpy(), v.numpy(), c, s))), \
        "port", orc.num_threads()


def time_cpu_sample(fn, heads, S, D, causal, scale, steps, warmup, seed=20):
    import torch
    g = torch.Generator().manual_seed(seed)
    q, k, v = (torch.empty(1, heads, S, D).normal_(0, 0.5, generator=g).to(torch.bfloat16).float() for _ in range(3))
    for _ in range(warmup):
        fn(q, k, v, causal, scale)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn(q, k, v, causal, scale)
        ts.append(time.perf_counter() - t0)
    return ts


def pick_sample_heads(fn, S, D, causal, scale, target_s, max_heads):
    t = time_cpu_sample(fn, 2, S, D, causal, scale, 1, 0)[0] / 2.0        # seconds per head (also a warm-up)
    return max(1, min(max_heads, int(target_s / max(t, 1e-6)))), t


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    W = WORKLOAD
    scale = 1.0 / math.sqrt(W["D"])
    fn, kind, cores = cpu_reference_runner()
    heads, per_head = pick_sample_heads(fn, W["S"], W["D"], W["causal"], scale, target_s=3.0,
                                        max_heads=W["B"] * W["H"])
    ts = time_cpu_sample(fn, heads, W["S"], W["D"], W["causal"], scale, args.steps, args.warmup)
    total = sum(ts)
    F = flops_effective(1, heads, W["S"], W["D"])
    val = F * len(ts) / total / 1e12
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "TFLOP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / len(ts) * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic N(0,0.5^2), seed 20",
        "config": {"workload": W["name"], "B": W["B"], "H": W["H"], "S": W["S"], "D": W["D"], "causal": W["causal"],
                   "step": f"bounded sample: {heads} of {W['B'] * W['H']} (batch*head) problems per step"},
        "cpu_baseline": {"value": val, "unit": "TFLOP/s", "cores": cores, "kind": kind,
                         "sample": f"{heads} heads x S{W['S']} x D{W['D']} causal fp32 per step, "
                                   f"/root/reference/flash_attention_c flash_attn (OpenMP, all host threads)"},
        "e2e": {"value": val, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------
def bind_to_gpu_numa(index):
    """Pin this process (and with it the first-touch placement of the pinned host buffers and the copy-issuing thread)
    to the CPUs NVML reports as local to GPU `index`.  Under torchrun the 8 ranks otherwise all allocate their pinned
    buffers wherever the launcher happened to run, and 7 of 8 PCIe streams cross the socket interconnect (r01: e2e at N=8
    was 2.2x the PCIe-ideal time)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        after = sorted(os.sched_getaffinity(0))
        node = None
        try:
            bus = pynvml.nvmlDeviceGetPciInfo(h).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            node = int(open(f"/sys/bus/pci/devices/{bus[-12:].lower()}/numa_node").read())
        except Exception:  # noqa: BLE001
            pass
        return {"bound": True, "cpus_before": before, "cpus_after": len(after), "first_cpu": after[0] if after else None,
                "numa_node": node}
    except Exception as e:  # noqa: BLE001
        return {"bound": False, "why": repr(e)[:120]}


def make_inputs(B, H, S, D, seed, device, dtype):
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    return [torch.empty(B, H, S, D, dtype=dtype, device=device).normal_(0.0, 0.5, generator=g) for _ in range(3)]


def time_kernel(tfa, q, k, v, causal, scale, out, lse, reps, warm, flush=None):
    """Mean/median device time of the kernel alone (CUDA events on the launch stream)."""
    import torch
    for _ in range(warm):
        tfa.fwd(q, k, v, causal, scale, out=out, lse=lse)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tfa.fwd(q, k, v, causal, scale, out=out, lse=lse)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    ts.sort()
    return sum(ts) / len(ts), ts[len(ts) // 2], ts[0]


def run_ours(args):
    import torch
    import torch.distributed as dist
    import tfa_ctypes as tfa

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    tfa.lib()                                     # fail loudly if the CUDA library is missing
    numa = bind_to_gpu_numa(local_rank)           # before any pinned allocation: first touch places it on the GPU's node
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    W = WORKLOAD
    B, H, S, D, causal = W["B"], W["H"], W["S"], W["D"], W["causal"]
    scale = 1.0 / math.sqrt(D)
    from sharded import shard_batch
    lo, hi = shard_batch(B, rank, world)
    Bl = hi - lo
    q, k, v = make_inputs(Bl, H, S, D, 20 + rank, dev, torch.bfloat16)
    out = torch.empty_like(q)
    lse = torch.empty(Bl, H, S, dtype=torch.float32, device=dev)
    o_full = torch.empty(B, H, S, D, dtype=torch.bfloat16, device=dev) if world > 1 else None
    peak, peak_sus, peak_src = load_peaks()

    # N>1: the local batch is processed in chunks; the NCCL all-gather of chunk c (async, NCCL's own stream)
    # overlaps the kernel of chunk c+1.  Every rank ends the step holding the full O (north_star's exchange).
    n_chunks = min(args.chunks, Bl) if world > 1 else 1
    cb = [(Bl * c // n_chunks, Bl * (c + 1) // n_chunks) for c in range(n_chunks)]
    stage = [torch.empty((world * (hi_ - lo_), H, S, D), dtype=torch.bfloat16, device=dev) for lo_, hi_ in cb] \
        if world > 1 else []

    # exchange: "fused" = the kernel's epilogue stores O straight into every peer's gathered buffer over NVLink
    # (sharded.FusedGather, no collective on the data path); "nccl" = kernel then ncclAllGather.
    fused = None
    exchange = "none"
    if world > 1:
        exchange = args.exchange
        if exchange == "fused":
            try:
                from sharded import FusedGather
                fused = FusedGather(B, H, S, D, torch.bfloat16, dev)
            except Exception as e:  # noqa: BLE001
                sys.stderr.write(f"[bench] fused exchange unavailable ({e!r}); using the NCCL all-gather\n")
                exchange = "nccl"
        flag = torch.tensor([1 if exchange == "fused" else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)          # every rank must agree
        if int(flag.item()) == 0:
            fused, exchange = None, "nccl"

    kernel_events = []          # (start, end) CUDA events around every kernel launch of the timed region

    def launch_kernel(lo_, hi_, record):
        if record:
            e_a, e_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e_a.record()
        tfa.fwd(q[lo_:hi_], k[lo_:hi_], v[lo_:hi_], causal, scale, out=out[lo_:hi_], lse=lse[lo_:hi_])
        if record:
            e_b.record()
            kernel_events.append((e_a, e_b))

    def step(record=False):
        if world == 1:
            launch_kernel(0, Bl, record)
            return
        if fused is not None:
            if record:
                e_a, e_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e_a.record()
            fused.launch(q, k, v, causal, scale, lse=lse)
            if record:
                e_b.record()
                kernel_events.append((e_a, e_b))
            fused.barrier()
            return
        if n_chunks == 1:
            launch_kernel(0, Bl, record)
            dist.all_gather_into_tensor(o_full, out)       # straight into the batch-major result
            return
        works = []
        for c, (lo_, hi_) in enumerate(cb):
            launch_kernel(lo_, hi_, record)
            works.append(dist.all_gather_into_tensor(stage[c], out[lo_:hi_], async_op=True))
        for w_ in works:
            w_.wait()
        # staged chunks -> batch-major O (rank r owns batches [r*Bl, (r+1)*Bl))
        of = o_full.view(world, Bl, H, S, D)
        for c, (lo_, hi_) in enumerate(cb):
            of[:, lo_:hi_].copy_(stage[c].view(world, hi_ - lo_, H, S, D))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    exchange_check = None
    if fused is not None:
        step()
        dist.all_gather_into_tensor(o_full, fused.buf[lo:hi].contiguous())
        torch.cuda.synchronize()
        ok = torch.tensor([1 if torch.equal(fused.buf, o_full) else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        exchange_check = "fused result == ncclAllGather result on every rank" if int(ok.item()) else "MISMATCH"

    # ---- value: K timed steps, device time, max over ranks ----
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    n0 = tfa.launch_count()
    with ClockSampler(local_rank) as clk:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(args.steps):
            step(record=True)
        e1.record()
        barrier()
    launches = tfa.launch_count() - n0
    result = fused.buf if fused is not None else (o_full if world > 1 else out)      # (B,H,S,D) at N>1, local at N=1
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"out": result.view(-1, D), "lse": lse.view(-1)})
    t_total = e0.elapsed_time(e1) * 1e-3
    if world > 1:
        tt = torch.tensor([t_total], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_total = float(tt.item())
    t_step = t_total / args.steps
    F_job = flops_effective(B, H, S, D)
    value = F_job / t_step / 1e12

    kernel_main = kernel_name(tfa).replace("_kernel ", "_kernel<128,causal,bf16> ", 1)
    # ---- roofline: the dominant (only) kernel, from the events recorded INSIDE the timed region ----
    k_times = [a_.elapsed_time(b_) * 1e-3 for a_, b_ in kernel_events]
    k_mean, k_min = sum(k_times) / len(k_times), min(k_times)
    launches_per_step = len(k_times) // args.steps
    F_launch = flops_effective(Bl, H, S, D) / launches_per_step
    achieved = F_launch / k_mean / 1e12
    compute_only_value = flops_effective(B, H, S, D) / (k_mean * launches_per_step) / 1e12   # all ranks, kernels only

    # fused compute+collective kernel: target = slower of (FLOPs / tensor peak) and (bytes that must leave this GPU
    # over NVLink / measured 770 GB/s per direction), per /opt/skills/guides/B200_PROFILING.md
    fused_roofline = None
    if fused is not None:
        nv_bytes = (world - 1) * Bl * H * S * D * 2
        t_flops = F_launch / (peak * 1e12)
        t_link = nv_bytes / 770e9
        target = max(t_flops, t_link)
        fused_roofline = {"kernel": kernel_main + " + peer stores (tfa_fwd_multi)", "nvlink_bytes_out_per_launch": nv_bytes,
                          "nvlink_peak_GBps": 770.0, "t_tensor_ms": t_flops * 1e3, "t_nvlink_ms": t_link * 1e3,
                          "target_ms": target * 1e3, "achieved_ms": k_mean * 1e3, "frac": target / k_mean,
                          "bound": "nvlink" if t_link > t_flops else "tensor"}

    # ---- e2e: host buffers through the C ABI ----
    e2e = None
    if not args.no_e2e:
        hq, hk, hv = (torch.empty(Bl, H, S, D, dtype=torch.bfloat16).pin_memory() for _ in range(3))
        for h_, d_ in ((hq, q), (hk, k), (hv, v)):
            h_.copy_(d_)
        hout = torch.empty(Bl, H, S, D, dtype=torch.bfloat16).pin_memory()
        hlse = torch.empty(Bl, H, S, dtype=torch.float32).pin_memory()
        chunks = 8
        tfa.fwd_host(hq, hk, hv, hout, hlse, causal, scale, n_chunks=chunks)          # warm (allocates workspace)
        barrier()
        e2e_steps = max(2, min(args.steps, 5))
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            tfa.fwd_host(hq, hk, hv, hout, hlse, causal, scale, n_chunks=chunks)
        barrier()
        te = (time.perf_counter() - t0) / e2e_steps
        if world > 1:
            tt = torch.tensor([te], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            te = float(tt.item())
        dev_head = (fused.buf[lo, 0] if fused is not None else out[0, 0])      # fused mode never writes `out`
        same = bool(torch.equal(hout[0, 0], dev_head.cpu()))
        e2e = {"value": F_job / te / 1e12, "unit": "TFLOP/s",
               "h2d_bytes_per_step": int(3 * q.numel() * 2 * world), "d2h_bytes_per_step": int((out.numel() * 2 + lse.numel() * 4) * world),
               "ms_per_step": te * 1e3, "api": "tfa_fwd_host (C ABI, pinned host buffers, 8 chunks on 4 streams)",
               "matches_device_path": same, "timer": "host wall clock around synchronous calls", "numa": numa}
        tfa.lib().tfa_host_release()
        del hq, hk, hv, hout, hlse

    # ---- parity: the result every rank holds after a step, against fp32 torch, on heads picked to cover the launch
    #      order's first and last chunk and (N>1) a head computed by ANOTHER rank and delivered by the exchange ----
    peer_head = None
    if world > 1:
        src = 1                                                  # rank 1's first (batch, head): inputs live there
        pq = torch.empty(3, S, D, dtype=torch.bfloat16, device=dev)
        if rank == src:
            pq.copy_(torch.stack([q[0, 0], k[0, 0], v[0, 0]]))
        dist.broadcast(pq, src)
        peer_head = (pq[0], pq[1], pq[2], shard_batch(B, src, world)[0], 0)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    def check_head(qh, kh, vh, got, label):
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        s_ = (qh.float() @ kh.float().t()) * scale
        if causal:
            s_.masked_fill_(torch.ones(S, S, device=dev, dtype=torch.bool).triu_(1), float("-inf"))
        want = torch.softmax(s_, dim=-1) @ vh.float()
        torch.backends.cuda.matmul.allow_tf32 = old
        diff = (got.float() - want).abs()
        ok = diff <= 1e-3 + 1e-3 * want.abs()
        return {"head": label, "max_abs_err": float(diff.max()), "pass_frac_rtol1e-3_atol1e-3": float(ok.float().mean())}

    parity = None
    parity_ok = True
    try:
        gb = lo if world > 1 else 0                              # global batch index of this rank's first batch in `result`
        heads = [check_head(q[0, 0], k[0, 0], v[0, 0], result[gb, 0], f"first local (b={gb},h=0)"),
                 check_head(q[Bl - 1, H - 1], k[Bl - 1, H - 1], v[Bl - 1, H - 1], result[gb + Bl - 1, H - 1],
                            f"last local (b={gb + Bl - 1},h={H - 1})")]
        if peer_head is not None:
            pq_, pk_, pv_, pb, ph = peer_head
            heads.append(check_head(pq_, pk_, pv_, result[pb, ph], f"computed by rank 1, delivered by the exchange (b={pb},h={ph})"))
        worst = min(h_["pass_frac_rtol1e-3_atol1e-3"] for h_ in heads)
        parity = {"vs": "fp32 torch softmax(scale QK^T)V on the buffer every rank holds after a step"
                        + (" (fused.buf: written by the kernel epilogues of all ranks)" if fused is not None else ""),
                  "max_abs_err": max(h_["max_abs_err"] for h_ in heads), "pass_frac_rtol1e-3_atol1e-3": worst,
                  "heads": heads,
                  "note": "misses are bf16 output rounding on early causal rows (half an ulp at |O|>=0.5 exceeds 1e-3); "
                          "the fp32-output build passes strictly (tests/test_fwd_parity.py)"}
        parity_ok = worst >= 0.999
    except Exception as e:  # noqa: BLE001
        parity = {"error": repr(e)}
        parity_ok = False

    configs = {}
    if world == 1 and not args.no_extras:
        del q, k, v, out, lse
        torch.cuda.empty_cache()
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        for name, (b_, h_, s_, d_, c_) in EXTRA_CONFIGS.items():
            qq, kk, vv = make_inputs(b_, h_, s_, d_, 20, dev, torch.bfloat16)
            oo = torch.empty_like(qq)
            ll = torch.empty(b_, h_, s_, dtype=torch.float32, device=dev)
            mean, med, mn = time_kernel(tfa, qq, kk, vv, c_, 1.0 / math.sqrt(d_), oo, ll, reps=20, warm=5, flush=flush)
            Fe, Fs = flops_effective(b_, h_, s_, d_), flops_std(b_, h_, s_, d_, c_)
            configs[name] = {"kernel": kernel_name(tfa).split(" ")[0], "ms": med * 1e3, "tflops": Fe / med / 1e12, "tflops_std": Fs / med / 1e12,
                             "roofline_frac": Fe / med / 1e12 / peak, "roofline_frac_std": Fs / med / 1e12 / peak,
                             "l2": "256 MB flush between reps"}
            del qq, kk, vv, oo, ll

    # ---- SURVEY 8f rows 2-3 (grouped K/V heads, Sq != Sk, split-KV): timed the same way, reported beside ----
    next_rows = {}
    if world == 1 and not args.no_extras:
        try:
            try:
                hbm_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
            except Exception:  # noqa: BLE001
                hbm_peak = 6500.0          # profiling recipe fallback

            def time_general(qq, kk, vv, causal_, ns):
                sc = 1.0 / math.sqrt(qq.shape[-1])
                for _ in range(3):
                    tfa.attn_fwd(qq, kk, vv, causal_, sc, num_splits=ns)
                torch.cuda.synchronize()
                ts = []
                used = 1
                for _ in range(10):
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    _, _, used = tfa.attn_fwd(qq, kk, vv, causal_, sc, num_splits=ns, return_splits=True)
                    e1.record()
                    torch.cuda.synchronize()
                    ts.append(e0.elapsed_time(e1) * 1e-3)
                ts.sort()
                return ts[len(ts) // 2], used

            g = torch.Generator(device=dev).manual_seed(20)
            mk = lambda *shape: torch.empty(*shape, dtype=torch.bfloat16, device=dev).normal_(0.0, 0.5, generator=g)
            # (a) cfg3 with 4 query heads per K/V head
            qq, kk, vv = mk(4, 32, 4096, 128), mk(4, 8, 4096, 128), mk(4, 8, 4096, 128)
            med, _ = time_general(qq, kk, vv, True, 1)
            next_rows["gqa: cfg3 with Hkv=8 (B4 Hq32 S4096 D128 causal)"] = {
                "ms": med * 1e3, "tflops": flops_effective(4, 32, 4096, 128) / med / 1e12,
                "roofline_frac": flops_effective(4, 32, 4096, 128) / med / 1e12 / peak}
            del qq, kk, vv
            # (b) few query rows, long keys: HBM-bound (K and V are read once), only split-KV fills the GPU
            Bq, Hh, Sq_, Sk_, Dd = 1, 8, 128, 65536, 128
            qq, kk, vv = mk(Bq, Hh, Sq_, Dd), mk(Bq, Hh, Sk_, Dd), mk(Bq, Hh, Sk_, Dd)
            one, _ = time_general(qq, kk, vv, False, 1)
            spl, used = time_general(qq, kk, vv, False, 0)
            byts = 2 * Bq * Hh * Sk_ * Dd * 2 + 2 * Bq * Hh * Sq_ * Dd * 2
            next_rows["splitkv: B1 H8 Sq128 Sk65536 D128 non-causal"] = {
                "single_pass_ms": one * 1e3, "split_ms": spl * 1e3, "num_splits": used,
                "speedup": one / spl, "algorithmic_GBps": byts / spl / 1e9,
                "roofline": {"bound": "hbm", "achieved": byts / spl / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": (byts / spl / 1e9 / hbm_peak) if hbm_peak else None,
                             "note": "forward + combine kernels together; bytes = K,V once + Q + O"}}
            del qq, kk, vv
        except Exception as e:  # noqa: BLE001
            next_rows["error"] = repr(e)

    cpu_baseline = None
    if world == 1 and not args.no_cpu:
        try:
            fn, kind, cores = cpu_reference_runner()
            heads, _ = pick_sample_heads(fn, S, D, causal, scale, target_s=10.0, max_heads=B * H)
            ts = time_cpu_sample(fn, heads, S, D, causal, scale, 1, 0)
            cpu_baseline = {"value": flops_effective(1, heads, S, D) / ts[0] / 1e12, "unit": "TFLOP/s", "cores": cores,
                            "kind": kind, "sample": f"{heads} of {B * H} (batch*head) problems of the workload, fp32 "
                                                    f"copies of the same-distribution inputs, 1 pass ({ts[0]:.1f} s)"}
            # the same C++ CPU path on BASELINE configs 2-4 (bounded head samples, ~2 s each) ...
            others = {}
            for name, (b_, h_, s_, d_, c_) in EXTRA_CONFIGS.items():
                hs, _ = pick_sample_heads(fn, s_, d_, c_, 1.0 / math.sqrt(d_), target_s=2.0, max_heads=b_ * h_)
                t1 = time_cpu_sample(fn, hs, s_, d_, c_, 1.0 / math.sqrt(d_), 1, 0)[0]
                others[name] = {"tflops": flops_effective(1, hs, s_, d_) / t1 / 1e12, "heads_sampled": hs, "of": b_ * h_,
                                "seconds": t1, "kind": kind, "cores": cores}
            cpu_baseline["configs"] = others
            # ... and the reference's naive-Python path at BASELINE config 1 (B1 H2 S128 D64 fp32, no scale, no mask)
            cpu_baseline["naive_python_cfg1"] = time_naive_python_cfg1()
        except Exception as e:  # noqa: BLE001
            cpu_baseline = {"error": repr(e)}

    comparators = None
    if world == 1 and not args.no_extras and not args.no_comparators:
        comparators = run_comparators()

    # denominator: the measured BURST cuBLAS figure.  The sustained figure only applies to a seconds-long region whose
    # sampled SM clock actually sat well below max (VERDICT r01 / ADVICE r01: a 0.1-0.2 s region at ~1.9 GHz is burst).
    clocks = clk.summary()
    region_s = args.steps * launches_per_step * k_mean
    sustained_applies = (region_s >= 1.0 and clocks.get("sm_mhz") and clocks.get("sm_max_mhz")
                         and clocks["sm_mhz"] < 0.8 * clocks["sm_max_mhz"])
    roof_peak = peak_sus if sustained_applies else peak
    roof_peak_name = ("bf16_tflops_sustained (%.1f s region, median SM clock %.0f MHz < 0.8 max)" % (region_s, clocks["sm_mhz"])
                      if sustained_applies else "bf16_tflops (burst)")
    traffic, traffic_src = profiled_traffic(Bl * H / launches_per_step)
    line = {
        "metric": METRIC, "value": value, "unit": "TFLOP/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": t_step * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic N(0,0.5^2), seed 20+rank, random Q/K/V",
        "config": {"workload": W["name"], "B": B, "H": H, "S": S, "D": D, "causal": causal,
                   "softmax_scale": "1/sqrt(D)", "parallelism": f"batch-sharded x{world}" + ("" if world == 1 else (
                       " + O gathered by fused NVLink peer stores in the kernel epilogue (no collective)" if fused is not None
                       else f" + NCCL all-gather of O ({n_chunks} chunk(s))")),
                   "exchange": exchange, "exchange_check": exchange_check,
                   "flops": "2*B*H*S^2*D", "l2": "inputs (3 x %.0f MB per rank) larger than the 126 MB L2" % (q_bytes(Bl, H, S, D) / 1e6)},
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": roof_peak, "unit": "TFLOP/s",
                     "frac": achieved / roof_peak,
                     "frac_of_burst_peak": achieved / peak, "frac_of_sustained_peak": achieved / peak_sus,
                     "peak_source": f"MEASURED_PEAKS.json ({peak_src}): " + roof_peak_name,
                     "kernel": kernel_main, "kernel_ms_mean": k_mean * 1e3, "kernel_ms_min": k_min * 1e3,
                     "timing": "CUDA events around each launch inside the timed region",
                     "flops_per_launch": F_launch, "launches_per_step_per_rank": launches_per_step,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "algorithmic_bytes_per_launch": (4 * S * D * 2 + 4 * S) * (Bl * H) / launches_per_step},
        "fused_roofline": fused_roofline,
        "compute_only": {"value": compute_only_value, "unit": "TFLOP/s", "note": "kernel only, no all-gather"},
        "cpu_baseline": cpu_baseline,
        "parity": parity,
        "configs": configs,
        "comparators": comparators,
        "next_rows": next_rows,
    }
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not parity_ok:
        sys.stderr.write("[bench] PARITY FAILED: " + json.dumps(parity) + "\n")
        sys.exit(3)


DUMP_ROWS = 1 << 16      # sampled rows of O: 32 MiB of float32 at D=128, so out.npy + lse.npy stay under 64 MB


def dump_outputs(path, arrays, seed=0):
    """--dump-outputs: write each array (rows along dim 0) as float32 <path>/<name>.npy.  An array with more than
    DUMP_ROWS rows is written as the rows at a fixed, seeded sample of DUMP_ROWS indices (ascending), so two builds run
    with the same arguments can be compared element for element; at N=1, out.npy[i] and lse.npy[i] are the same query
    row (b, h, s)."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        if t.shape[0] > DUMP_ROWS:
            idx = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(seed))[:DUMP_ROWS].sort().values
            t = t[idx.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def q_bytes(B, H, S, D):
    return B * H * S * D * 2


def kernel_name(tfa):
    """Name of the kernel the library's AUTO choice (csrc/tfa_api.cu choose_kernel) used for the last launch."""
    try:
        v = int(tfa.lib().tfa_internal_last_variant())
    except Exception:  # noqa: BLE001
        v = 0
    return {0: "fa_fwd_sm100_kernel (one CTA per work item)",
            4: "fa_fwd_sm100_persist_kernel (persistent, TMA-store epilogue)"}.get(v, str(v))



def profiled_traffic(heads_per_launch):
    """roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full`
    capture of the SAME kernel source (profiles/traffic.json records the capture's commit and the digest of the kernel
    sources it was taken from); null when the kernel sources changed since -- a stale constant is worse than none."""
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        import hashlib
        h = hashlib.sha256()
        for f in rec["sources"]:
            h.update(open(os.path.join(ROOT, f), "rb").read())
        if h.hexdigest() != rec["sources_sha256"]:
            return None, f"profiles/traffic.json is from commit {rec.get('commit')} and the kernel sources changed since: no traffic claim"
        return rec["dram_bytes_per_head"] * heads_per_launch, (
            f"{rec['capture']} (commit {rec.get('commit')}): {rec['dram_bytes_per_head'] / 1e6:.3f} MB per (batch*head) "
            f"for {rec['algorithmic_bytes_per_head'] / 1e6:.3f} MB algorithmic, scaled by heads per launch")
    except Exception as e:  # noqa: BLE001
        return None, f"no profiles/traffic.json ({e!r})"


def run_comparators(timeout_s=420):
    """Library / reference-kernel comparators on cfg2-4 in a SUBPROCESS (scripts/comparators.py)."""
    import subprocess
    try:
        env = dict(os.environ, CMP_BUDGET_S="300")
        p = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "comparators.py")], capture_output=True, text=True,
                           timeout=timeout_s, env=env)
        for ln in p.stdout.splitlines():
            if ln.startswith("CMP "):
                return json.loads(ln[4:])
        return {"error": "no result", "rc": p.returncode, "stderr_tail": p.stderr[-400:]}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)[:300]}


def time_naive_python_cfg1():
    """BASELINE config 1 (B1 H2 S128 D64 fp32, no scale, no mask) through the reference's naive-Python path
    tiny_flash_attn.flash_attn_v2_multihead (flash_attention_py/tiny_flash_attn.py:137-196) when its unmodified copy
    travelled with baseline/_ref (kind "reference"); else the oracle's restatement of the same block algorithm
    (kind "port")."""
    import torch
    B_, H_, S_, D_ = 1, 2, 128, 64
    g = torch.Generator().manual_seed(20)
    q, k, v = (torch.empty(B_, H_, S_, D_).normal_(0, 0.5, generator=g) for _ in range(3))
    F = flops_effective(B_, H_, S_, D_)
    ref_dir = os.path.join(ROOT, "baseline", "_ref", "drivers", "py")
    if os.path.exists(os.path.join(ref_dir, "tiny_flash_attn.py")):
        sys.path.insert(0, ref_dir)
        try:
            import tiny_flash_attn as tfa_py
            torch.set_num_threads(1)
            fn = lambda: tfa_py.flash_attn_v2_multihead(q, k, v, device="cpu", BLOCK_M=4)
            kind, what = "reference", "tiny_flash_attn.flash_attn_v2_multihead(device='cpu', BLOCK_M=4), unmodified copy"
        finally:
            sys.path.remove(ref_dir)
    else:
        from oracle import oracle as orc
        fn = lambda: orc.flash_v2_blocks(q.numpy(), k.numpy(), v.numpy(), 4)
        kind, what = "port", "oracle.flash_v2_blocks (C restatement of tiny_flash_attn.py:137-196)"
    fn()
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    t = sorted(ts)[1]
    import torch as _t
    _t.set_num_threads(os.cpu_count() or 1)
    return {"tflops": F / t / 1e12, "seconds": t, "kind": kind, "cores": 1, "what": what,
            "config": "cfg1: B=1 H=2 S=128 D=64 fp32 non-causal, scale 1"}


def emit(line: dict) -> None:
    """Print THE one JSON line on the real stdout (everything else -- NCCL banners, torch.distributed chatter --
    was diverted to stderr in main())."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    # keep stdout clean for the driver: fd 1 -> stderr for the whole run, the JSON line goes to the saved fd
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-comparators", action="store_true")
    ap.add_argument("--exchange", default="fused", choices=["fused", "nccl"],
                    help="N>1: how O is gathered (fused peer stores in the kernel epilogue, or ncclAllGather)")
    ap.add_argument("--chunks", type=int, default=1, help="N>1: batch chunks per rank (gather/compute overlap)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's O and LSE at a fixed sample of query rows "
                         "as DIR/out.npy and DIR/lse.npy (float32)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
