#!/usr/bin/env python
"""bench.py -- the headline benchmark (BASELINE.json: "Q4_0 x Q8_1 GEMM ... HBM GB/s vs roofline;
M=1 GEMV us at Llama shapes").

One step = one decode token (M=1) pushed through every linear layer of a Llama-7B-shaped stack
with Q4_0 weights x Q8_1 activations: 32 layers x {wq,wk,wv,wo: 4096x4096, gate,up: 11008x4096,
down: 4096x11008} = 224 GEMV launches over 3.64 GB of distinct weight bytes (29x the 126 MB L2, so
every launch streams from HBM), replayed as one CUDA graph.

  value   = algorithmic bytes of all launches of all ranks / device time      [GB/s]
            (weights once + q8_1 activations + fp32 outputs; SURVEY.md section 8d)
  e2e     = the same step through the public python API (quant_gemm) with HOST buffers: pinned
            fp32 activations H2D, quantize_q8_1, 224 GEMVs, all outputs D2H -- inside the timed region
  N > 1   : weak scaling.  Decode shapes do not shard usefully (SURVEY.md 8e: "replicas only"), so by
            default every rank decodes its own copy of the stack with no data-path collective.
            --gather fused|nccl runs the tensor-parallel variant instead (every rank owns the rows of
            its shard of an N-times wider model, per-GEMV all-gather fused into the kernel or by NCCL).
            The shape that does shard, BASELINE configs[4] (M=4096 N=28672 K=8192 Q4_0, weight rows
            split over the ranks, all-gather of C), is timed as `extra.sharded_c5` at every N.
  --impl reference : the reference's own CPU implementation (oracle/_ref, all host threads) on
            a bounded sample (one layer = 7 GEMVs per step) of the same workload.

Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
_JSON_OUT = sys.stdout
for _p in (os.path.join(ROOT, "llama.cpp-quant-gemm_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "q4_0_q8_1_decode_gemv_hbm_gbs"
UNIT = "GB/s"
LLAMA7B = [("wq", 4096, 4096), ("wk", 4096, 4096), ("wv", 4096, 4096), ("wo", 4096, 4096),
           ("gate", 11008, 4096), ("up", 11008, 4096), ("down", 4096, 11008)]
WTYPE = 2  # Q4_0
GEMV_FLAGS = 0x10  # QGEMM_WEIGHTS_STATIC: model weights are never written while decoding
READY_FLAGS = 0x30  # + QGEMM_INPUTS_READY: wk/wv after wq and `up` after `gate` share an input that is already there
BS = {2: 18, 3: 20, 6: 22, 7: 24, 8: 34}


def algorithmic_bytes(wtype, T, F, K):
    nb = K // 32
    return F * nb * BS[wtype] + T * nb * 36 + 4 * T * F


def load_traffic():
    """Per-launch DRAM bytes of the dominant kernel from the committed ncu --set full capture."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["dram_bytes_per_launch_bench_average"], d["source"]
    return None, None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        import threading
        self.p, self.lines, self.first = None, [], threading.Event()
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "10"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return

        def pump():
            for line in self.p.stdout:
                self.lines.append((time.perf_counter(), line))
                self.first.set()
        self.t = threading.Thread(target=pump, daemon=True)
        self.t.start()
        self.first.wait(timeout=5.0)   # sampling is live before the timed region starts
        self.t_start = time.perf_counter()

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_stop = time.perf_counter()
        time.sleep(0.03)
        self.p.terminate()
        self.t.join(timeout=2.0)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            if ts < self.t_start or ts > t_stop + 0.02:   # only samples taken while the timed regions ran
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # the busiest half of the samples = "under load"
        sm.sort()
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU code on the host cores
# ------------------------------------------------------------------------------------------
def make_blocks_numpy(F, K, seed):
    import numpy as np
    import datagen
    return datagen.fuzz_weight_blocks(WTYPE, F, K // 32, seed=seed)


def cpu_reference_run(steps, warmup, sample_layers=1, budget_s=None):
    """Times the reference's cpu_gemm_q4_0_q8_1 (tests/unit/test_gemm_all_quants.cu:23-59, compiled
    unmodified into oracle/_ref) -- or the oracle port if that library is absent -- over
    `sample_layers` layers of the workload per step, all host threads (weight-row slabs)."""
    import numpy as np
    import datagen
    import qgemm_oracle as qo
    cores = os.cpu_count() or 1
    use_ref = qo.have_ref()
    R = qo.Reference() if use_ref else None
    O = qo.Oracle()
    mats = []
    for i, (_, F, K) in enumerate(LLAMA7B * sample_layers):
        w = make_blocks_numpy(F, K, seed=i)
        a = datagen.fuzz_act_blocks(1, K // 32, seed=i, const_ds=False)
        mats.append((F, K, w, a))
    step_bytes = sum(algorithmic_bytes(WTYPE, 1, F, K) for F, K, _, _ in mats)

    def one_step():
        for F, K, w, a in mats:
            if use_ref:
                R.cpu_gemm(WTYPE, w, a, threads=cores)
            else:
                # the oracle port, slabbed over weight rows with the same thread count
                import threading
                out = np.empty((F, 1), np.float32)
                slab = (F + cores - 1) // cores
                ths = []
                for c in range(cores):
                    f0, f1 = c * slab, min(F, (c + 1) * slab)
                    if f0 >= f1:
                        break
                    th = threading.Thread(target=lambda f0=f0, f1=f1: O.lib.qo_gemm(
                        WTYPE, a.ctypes.data, w[f0:f1].ctypes.data, out[f0:f1].ctypes.data, 1, f1 - f0, K, 1, 1, 0, 0, 1))
                    th.start()
                    ths.append(th)
                for th in ths:
                    th.join()

    for _ in range(warmup):
        one_step()
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        one_step()
        done += 1
        if budget_s and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": step_bytes * done / dt / 1e9, "unit": UNIT, "cores": cores,
            "kind": "reference" if use_ref else "port",
            "sample": f"{sample_layers} layer(s) = {7 * sample_layers} M=1 Q4_0 GEMVs per step "
                      f"({step_bytes / 1e6:.1f} MB), {done} steps, weight-row slabs over {cores} threads",
            "ms_per_step": dt / done * 1e3, "steps": done}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int8xint4->int32, fp32 fold", "data": "synthetic",
            "config": workload_config(args.gpus),
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), file=_JSON_OUT, flush=True)


def sharded_c5(torch, dist, quant_gemm, dev, world, rank, ctl, reps=3):
    """BASELINE configs[4]: Q4_0 M=4096 N=28672 K=8192, weight rows sharded over the ranks (strong scaling).
    Times (i) the local GEMM alone, (ii) GEMM + in-place NCCL all-gather, (iii) the GEMM whose tcgen05
    epilogue stores its tiles into every rank's gathered C over NVLink; device events, max over ranks."""
    from quant_gemm import sharded
    import bench_detail
    T, F, K = 4096, 28672, 8192
    f0, f1 = sharded.shard_rows(F, world, rank)
    w = bench_detail.make_weights(torch, WTYPE, f1 - f0, K, 1, dev, seed=99 + rank)[0]
    x = torch.randn((T, K), device=dev, generator=torch.Generator(device=dev).manual_seed(5))
    aq = quant_gemm.quantize_q8_1(x)
    del x
    out_full = torch.empty((F, T), device=dev)
    ops = 2.0 * T * F * K

    def timed(fn):
        best = 1e30
        for i in range(reps + 1):
            if world > 1:
                dist.barrier(group=ctl)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            if world > 1:
                t = torch.tensor([ms])
                dist.all_reduce(t, op=dist.ReduceOp.MAX, group=ctl)
                ms = float(t.item())
            if i > 0:
                best = min(best, ms)
        return best

    res = {"shape": "Q4_0 M=4096 N=28672 K=8192", "rows_per_rank": f1 - f0, "scaling": "strong",
           "note": "whole calls incl. operand prepass; best of %d; max over ranks" % reps}
    local = out_full[f0:f1]
    ms = timed(lambda: quant_gemm.gemm(w, aq, f1 - f0, T, K, WTYPE, GEMV_FLAGS, out=local))
    res["compute_only"] = {"ms": ms, "tops": ops / ms / 1e9}
    if world > 1:
        op_n = sharded.ShardedGemm(w, F, K, WTYPE, flags=GEMV_FLAGS)
        ms = timed(lambda: op_n(aq, out=out_full))
        res["nccl_all_gather"] = {"ms": ms, "tops": ops / ms / 1e9}
        def fused_variant(multicast):
            plan = sharded.PeerPlan(F * T, 1, dev, ctl_group=ctl, multicast=multicast)
            op_p = sharded.ShardedGemmP2P(w, F, K, WTYPE, T, plan, flags=GEMV_FLAGS)

            def fused():
                op_p(aq)
                plan.end_step()
            ms = timed(fused)
            return {"ms": ms, "tops": ops / ms / 1e9, "nvls_multicast": bool(plan.mc_ptr),
                    "equals_nccl_bitwise": bool(torch.equal(op_p.out, out_full))}
        res["fused_peer_stores"] = fused_variant(True)      # one store per value, replicated by the NVSwitch (if NVLS)
        if res["fused_peer_stores"]["nvls_multicast"]:
            res["fused_peer_stores_unicast"] = fused_variant(False)   # one store per value and rank
        res["fused_equals_nccl_bitwise"] = res["fused_peer_stores"]["equals_nccl_bitwise"]
    return res


def add_c5_efficiency(res, world):
    """Strong-scaling efficiency of the sharded shape against the single-GPU time of the same build (committed by the
    N=1 run of this round, profiles/r02_bench_n1.json); the N=1 run records its own time as the reference."""
    ref_ms = None
    p = os.path.join(ROOT, "profiles", "r02_bench_n1.json")
    if os.path.exists(p):
        try:
            ref_ms = json.load(open(p))["extra"]["sharded_c5"]["compute_only"]["ms"]
        except (KeyError, ValueError):
            ref_ms = None
    if world == 1:
        res["single_gpu_ms"] = res["compute_only"]["ms"]
        return
    if ref_ms is None:
        return
    res["single_gpu_ms"] = ref_ms
    res["single_gpu_source"] = "profiles/r02_bench_n1.json"
    for k in ("compute_only", "nccl_all_gather", "fused_peer_stores", "fused_peer_stores_unicast"):
        if k in res and isinstance(res[k], dict) and "ms" in res[k]:
            res[k]["speedup_vs_1gpu"] = ref_ms / res[k]["ms"]
            res[k]["efficiency"] = ref_ms / res[k]["ms"] / world
    res["baseline_it_beats"] = "nccl_all_gather (local GEMM, then ncclAllGather of C in place)"


def workload_config(n_gpus, tp=1):
    if n_gpus == 1:
        par = "1 GPU"
    elif tp == 1:
        par = f"{n_gpus} independent replicas, no data-path collective (SURVEY 8e: decode shapes do not shard)"
    else:
        par = f"weight rows (N) sharded x{n_gpus}, all-gather of C per GEMV"
    return {"workload": "Llama-7B decode GEMV stack: M=1, 32 layers x {4x 4096x4096, 2x 11008x4096, 1x 4096x11008}, "
                        "Q4_0 weights x Q8_1 activations (BASELINE configs[1])",
            "gemvs_per_step": 224, "weight_bytes_per_gpu": 32 * sum(F * (K // 32) * 18 for _, F, K in LLAMA7B),
            "l2_defeat": "inputs larger than L2: 3.64 GB of distinct weights per step vs 126 MB L2",
            "parallelism": par,
            "timing": "CUDA events on the launch stream around K graph replays, max over ranks"}


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layers", type=int, default=32)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--group", type=int, default=1, help="1 GPU: fuse q/k/v and gate/up into grouped launches")
    ap.add_argument("--chain", type=int, default=0,
                    help="1 GPU: layers per persistent chained launch (qgemm_gemv_chain: the grouped projections of `chain` layers "
                         "walked by one launch with device-side dependencies; every step still waits for its predecessor to "
                         "complete on the whole device).  0 (default): one launch per grouped projection -- measured faster: a "
                         "programmatic dependent launch costs less than a device-wide barrier inside a kernel "
                         "(profiles/r02_chain.md); the chained form is timed as extra.chained_launch_form")
    ap.add_argument("--d2h-chunk-layers", type=int, default=4,
                    help="e2e: copy the outputs back to the host every this many layers on a side stream, overlapped with the "
                         "following layers (0: one copy at the end of the step)")
    ap.add_argument("--prefetch", type=int, default=1, help="1: hint each GEMV with the next one's weights (L2 prefetch)")
    ap.add_argument("--prefetch-mb", type=int, default=12,
                    help="L2 prefetch window in MB, starting at the next launch's first matrix (0: exactly that matrix). "
                         "Measured on the decode stack: 0 -> 4057, 12 -> 4170, 16 -> 4130, 24 -> 3998, 40 -> 3832 GB/s")
    ap.add_argument("--gather", default="none", choices=["none", "fused", "nccl"],
                    help="N > 1: none = independent replicas (default); tensor-parallel decode with the all-gather "
                         "fused into the kernel (peer stores over NVLink) or by NCCL per GEMV")
    ap.add_argument("--sharded-extra", type=int, default=1, help="time BASELINE configs[4] sharded over the ranks")
    ap.add_argument("--detail", default=None, help="write a per-shape sweep (all formats, M=1..8, prefill) to this JSON file")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last step computed as DIR/<projection>.npy (float32, "
                         "[layers, rows]; rank 0's outputs).  Inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU decode stack's outputs; --impl reference times a CPU sample and keeps none")
    args.warmup = max(args.warmup, 3)
    # stdout carries exactly one JSON line: native libraries that print there (NCCL's version banner) go to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    global _JSON_OUT
    _JSON_OUT = os.fdopen(json_fd, "w")
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import quant_gemm

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ctl = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        # control-plane collectives (barriers, max over ranks) use gloo: eager NCCL calls on the communicator
        # that is also replayed from CUDA graphs hung on this stack
        ctl = dist.new_group(backend="gloo")
    quant_gemm._lib.lib()
    tp = world if args.gather != "none" else 1   # ranks one GEMV is sharded over

    # ---- synthetic weight pool: raw-block fuzz (all nibble values), sane fp16 scales
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    # one allocation, matrices back to back in launch order (like a model file mapped into HBM)
    sizes = [F * (K // 32) * 18 for _ in range(args.layers) for _, F, K in LLAMA7B]
    arena = torch.empty(sum((n + 255) // 256 * 256 for n in sizes), dtype=torch.uint8, device=dev)
    mats, off = [], 0
    for layer in range(args.layers):
        for name, F, K in LLAMA7B:
            nb = K // 32
            w = arena[off:off + F * nb * 18].view(F, nb, 18)
            off += (F * nb * 18 + 255) // 256 * 256
            w.copy_(torch.randint(0, 256, (F, nb, 18), dtype=torch.uint8, device=dev, generator=g))
            d = (torch.rand((F, nb), device=dev, generator=g) * 0.02 + 0.001).to(torch.float16)
            w[:, :, 0:2] = d.view(torch.uint8).view(F, nb, 2)
            mats.append((F, K, w))
    arena_end = arena.data_ptr() + arena.numel()

    def hint(w):   # the next launch's weights, and on into what follows them up to --prefetch-mb
        if args.prefetch_mb > 0:
            quant_gemm.hint_next_weights(w, min(args.prefetch_mb << 20, arena_end - w.data_ptr()))
        else:
            quant_gemm.hint_next_weights(w)
    # the step's two activation vectors (K = 4096 and K = 11008) live back to back in one pinned host buffer, one device
    # buffer and one q8_1 buffer: one host->device copy and one quantize_q8_1 launch per step, views per K
    KS = (4096, 11008)
    acts_host_all = torch.cat([torch.randn((1, K), generator=torch.Generator().manual_seed(7 + K)) for K in KS], dim=1).pin_memory()
    acts_dev_all = acts_host_all.to(dev)
    acts_q_all = quant_gemm.quantize_q8_1(acts_dev_all)            # [1, sum(K)/32, 36]
    acts_host, acts_dev, acts_q, k0 = {}, {}, {}, 0
    for K in KS:
        acts_host[K] = acts_host_all[:, k0:k0 + K]
        acts_dev[K] = acts_dev_all[:, k0:k0 + K]
        acts_q[K] = acts_q_all[:, k0 // 32:(k0 + K) // 32]            # block boundaries: same bytes as quantizing each vector alone
        k0 += K
    # gathered C of every GEMV, [F_total, T=1] each, carved out of one buffer so the step's result
    # goes back to the host in one copy
    total_out = sum(F * tp for F, K, _ in mats)
    out_all = torch.empty(total_out, device=dev)
    outs, off = [], 0
    for F, K, _ in mats:
        outs.append(out_all[off:off + F * tp].view(F * tp, 1))
        off += F * tp
    out_host = torch.empty(total_out + 64 * len(mats), dtype=torch.float32).pin_memory()  # + pool alignment padding
    step_bytes = sum(algorithmic_bytes(WTYPE, 1, F, K) for F, K, _ in mats)

    from quant_gemm import sharded
    # every rank owns rows [rank*F, (rank+1)*F) of an (N*F)-row matrix
    plan = None
    if tp > 1 and args.gather == "fused":
        # all-gather fused into the GEMV: the kernel stores its slice of C into every rank's gathered
        # buffer over NVLink (symmetric memory) and signals with device-side counters
        plan = sharded.PeerPlan(sum(F * tp for F, K, _ in mats), len(mats), dev, ctl_group=ctl)
        if args.group:
            # 4 launches per layer: [wq wk wv] fused, wo, [gate up] fused, down -- each waits for its predecessor
            plan.lps = 4 * args.layers
            ops, outs = [], []
            for l in range(args.layers):
                b = 7 * l
                for g in ([b, b + 1, b + 2], [b + 3], [b + 4, b + 5], [b + 6]):
                    K = mats[g[0]][1]
                    if len(g) == 1:
                        op = sharded.ShardedGemvP2P(mats[g[0]][2], mats[g[0]][0] * tp, K, WTYPE, 1, plan, flags=GEMV_FLAGS)
                        outs.append(op.out)
                    else:
                        op = sharded.ShardedGemvGroupP2P([mats[i][2] for i in g], [mats[i][0] * tp for i in g], K, WTYPE,
                                                         1, plan, flags=GEMV_FLAGS)
                        outs += op.outs
                    ops.append((op, K, g))
        else:
            # Llama dataflow: [wq wk wv] <- previous layer's down, wo <- wv, [gate up] <- wo, down <- up
            ops = []
            for i, (F, K, w) in enumerate(mats):
                j = i % 7
                wait = i - j if j < 3 else (i if j in (3, 4, 6) else i - 1)
                ops.append(sharded.ShardedGemvP2P(w, F * tp, K, WTYPE, 1, plan, wait_index=wait,
                                                  flags=READY_FLAGS if j in (1, 2, 5) else GEMV_FLAGS))
            outs = [op.out for op in ops]
    elif tp > 1:  # baseline: in-place NCCL all-gather after every GEMV
        # Llama dataflow: wk, wv read the same (already complete) input as wq, `up` the same as `gate`
        ops = [sharded.ShardedGemm(w, F * tp, K, WTYPE, flags=READY_FLAGS if (i % 7) in (1, 2, 5) else GEMV_FLAGS)
               for i, (F, K, w) in enumerate(mats)]

    # launch plan of one step.  Single GPU: the projections that share an input go out as ONE grouped
    # launch (fused q/k/v and gate/up, qgemm_gemm_group) -- 4 launches per layer instead of 7, the
    # same weights and the same 224 outputs.
    groups = []
    if tp == 1 and args.group:
        for l in range(args.layers):
            b = 7 * l
            groups += [[b, b + 1, b + 2], [b + 3], [b + 4, b + 5], [b + 6]]

    chains = []
    if groups and args.chain > 0:
        per = 4 * args.chain
        for c0 in range(0, len(groups), per):
            steps = []
            for g in groups[c0:c0 + per]:
                K = mats[g[0]][1]
                # stream-order semantics: no step is marked `ready`, each waits until its predecessor has completed
                steps.append({"weights": [mats[i][2] for i in g], "Ms": [mats[i][0] for i in g], "K": K,
                              "act_q": acts_q[K], "outs": [outs[i] for i in g]})
            chains.append((quant_gemm.GemvChain(steps, WTYPE, GEMV_FLAGS), mats[groups[c0][0]][2]))

    def gemv_all(after_layer=None):
        if chains:
            for ci, (ch, _) in enumerate(chains):
                if args.prefetch:   # the head of the next chain's weights
                    hint(chains[(ci + 1) % len(chains)][1])
                ch()
            return
        if plan is not None and args.group:
            for oi, (op, K, g) in enumerate(ops):
                if args.prefetch:
                    hint(mats[ops[(oi + 1) % len(ops)][2][0]][2])
                op(acts_q[K])
            plan.end_step()
            return
        if groups:
            for gi, g in enumerate(groups):
                nxt = groups[(gi + 1) % len(groups)]
                if args.prefetch:   # the next launch's first matrix is what HBM should be fetching in the bubble
                    hint(mats[nxt[0]][2])
                K = mats[g[0]][1]
                if len(g) == 1:
                    quant_gemm.gemm(mats[g[0]][2], acts_q[K], mats[g[0]][0], 1, K, WTYPE, GEMV_FLAGS, out=outs[g[0]])
                else:
                    quant_gemm.gemm_group([mats[i][2] for i in g], acts_q[K], [mats[i][0] for i in g], 1, K, WTYPE,
                                          GEMV_FLAGS, outs=[outs[i] for i in g])
                if after_layer is not None and gi % 4 == 3:
                    after_layer(gi // 4)
            return
        # a decode runtime knows its layer order: each launch pulls the next GEMV's weights into L2
        n = len(mats)
        for i, (F, K, w) in enumerate(mats):
            if args.prefetch:
                hint(mats[(i + 1) % n][2])
            if plan is not None:
                ops[i](acts_q[K])
            elif tp > 1:
                ops[i](acts_q[K], out=outs[i])
            else:
                quant_gemm.gemm(w, acts_q[K], F, 1, K, WTYPE, READY_FLAGS if (i % 7) in (1, 2, 5) else GEMV_FLAGS, out=outs[i])
        if plan is not None:
            plan.end_step()

    def e2e_step():
        acts_dev_all.copy_(acts_host_all, non_blocking=True)
        quant_gemm.quantize_q8_1(acts_dev_all, out=acts_q_all)     # the decode runtime's fixed activation buffers
        if groups and not chains and plan is None and args.d2h_chunk_layers > 0:
            # the step's results go back to the host as they are produced: every few layers a side stream copies the finished
            # slice of the output buffer while the next layers compute (same bytes, same pinned destination); the step ends
            # when the last slice has landed
            main = torch.cuda.current_stream()
            per_layer = sum(F for _, F, _ in LLAMA7B)
            sent = [0]

            def after_layer(l):
                if (l + 1) % args.d2h_chunk_layers == 0 or l == args.layers - 1:
                    lo, hi = sent[0], (l + 1) * per_layer
                    sent[0] = hi
                    d2h_stream.wait_stream(main)
                    with torch.cuda.stream(d2h_stream):
                        out_host[lo:hi].copy_(out_all[lo:hi], non_blocking=True)
            gemv_all(after_layer)
            main.wait_stream(d2h_stream)
            return
        gemv_all()
        if plan is not None:   # fused all-gather: the gathered outputs live in the symmetric pool
            out_host[:plan.cursor].copy_(plan.pool[:plan.cursor], non_blocking=True)
        else:
            out_host[:total_out].copy_(out_all, non_blocking=True)

    stream = torch.cuda.Stream(device=dev)
    d2h_stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(stream):
        gemv_all()  # warm: cudaFuncSetAttribute, NCCL channels
        e2e_step()
        stream.synchronize()
        quant_gemm.reset_launch_count()
        g_dev = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_dev, stream=stream):
            gemv_all()
        launches_per_step = quant_gemm.launch_count()
        g_e2e = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_e2e, stream=stream):
            e2e_step()
        launches_per_e2e = quant_gemm.launch_count() - launches_per_step

    def timed(graph, steps, warmup):
        with torch.cuda.stream(stream):
            for _ in range(warmup):
                graph.replay()
            stream.synchronize()
            if world > 1:
                dist.barrier(group=ctl)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                graph.replay()
            e1.record(stream)
            stream.synchronize()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier(group=ctl)
            ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms])
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=ctl)
            ms = float(t.item())
        return ms

    sampler = ClockSampler(local_rank) if rank == 0 else None   # samples through both timed regions
    ms_dev = timed(g_dev, args.steps, args.warmup)
    ms_e2e = timed(g_e2e, args.steps, args.warmup)
    clocks = sampler.stop() if sampler else None

    # correctness spot check of the timed path against the oracle (rank 0, a few rows)
    check = None
    if rank == 0:
        import qgemm_oracle as qo
        O = qo.Oracle()
        F, K, w = mats[4]
        rows = np.r_[0:4, F - 4:F]
        ref = O.gemm(WTYPE, acts_q[K].cpu().numpy(), w[torch.from_numpy(rows).to(dev)].cpu().numpy(), layout="FT")
        got = outs[4][(rank if tp > 1 else 0) * F:][:F].cpu().numpy()[rows]  # outs[] stays indexed by matrix in every mode
        check = qo.max_norm_err(got, ref)
        assert check <= 1e-5, f"timed path disagrees with the oracle: {check}"
        # before the extras below, which reuse the output buffers
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            layer_bytes = 4 * sum(outs[i].numel() for i in range(7))
            dump_layers = min(args.layers, (64 << 20) // layer_bytes)   # the first layers, at most 64 MB in all
            for j, (name, _, _) in enumerate(LLAMA7B):
                c = torch.stack([outs[7 * l + j].reshape(-1) for l in range(dump_layers)])
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), c.cpu().numpy().astype(np.float32))

    value = step_bytes * world * args.steps / (ms_dev * 1e-3) / 1e9
    e2e_value = step_bytes * world * args.steps / (ms_e2e * 1e-3) / 1e9
    peak, peak_src = load_peaks()
    n_launch = launches_per_step   # kernels of ours per step (grouped launches cover several matrices)
    per_launch_bytes = step_bytes / n_launch
    per_launch_us = ms_dev * 1e3 / (args.steps * n_launch)
    achieved = per_launch_bytes / (per_launch_us * 1e-6) / 1e9
    traffic, traffic_src = load_traffic()

    # prefill side of the metric ("Q4_0 x Q8_1 GEMM TOPS"): BASELINE configs[2], whole call, rank 0 only
    extra = {}
    if rank == 0 and world == 1:
        import bench_detail
        r = bench_detail.time_prefill(torch, quant_gemm, WTYPE, 512, 4096, 4096, reps=20)
        extra = {"prefill_q4_0_M512_N4096_K4096": {"us": r["us"], "tops": r["tops"], "path": r["path"],
                                                   "frac_of_nominal_int8_4500_tops": r["tops"] / 4500.0,
                                                   "note": "BASELINE configs[2]; whole qgemm_gemm call incl. the activation prepass "
                                                           "(weights are unpacked inside the kernel), L2 flushed between reps"}}
        r = bench_detail.time_prefill(torch, quant_gemm, 7, 2048, 14336, 4096, reps=8, fused_f32=True)
        extra["prefill_q5_1_M2048_N14336_K4096_incl_quantize"] = {
            "us": r["us"], "tops": r["tops"], "path": r["path"], "frac_of_nominal_int8_4500_tops": r["tops"] / 4500.0,
            "note": "BASELINE configs[3]; fp32 activations in, quantize_q8_1 inside the call (two launches), L2 flushed between reps"}
        if groups and not chains:
            # the same step as persistent chained launches (the last review's suggestion), for the record: it is slower
            try:
                forms = {}
                for L in (1, args.layers):
                    cs = []
                    for c0 in range(0, len(groups), 4 * L):
                        steps = [{"weights": [mats[i][2] for i in g], "Ms": [mats[i][0] for i in g], "K": mats[g[0]][1],
                                  "act_q": acts_q[mats[g[0]][1]], "outs": [outs[i] for i in g]} for g in groups[c0:c0 + 4 * L]]
                        cs.append(quant_gemm.GemvChain(steps, WTYPE, GEMV_FLAGS))
                    with torch.cuda.stream(stream):
                        for ch in cs:
                            ch()
                        stream.synchronize()
                        gch = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(gch, stream=stream):
                            for ch in cs:
                                ch()
                    ms = timed(gch, 10, 3)
                    forms[f"{L}_layer(s)_per_launch"] = {"ms_per_step": ms / 10, "gbs": step_bytes * 10 / (ms * 1e-3) / 1e9,
                                                         "launches_per_step": len(cs)}
                    del gch
                extra["chained_launch_form"] = dict(forms, note="qgemm_gemv_chain: one persistent launch walks the grouped projections "
                                                    "with device-side dependencies (stream-order semantics kept); bit-identical "
                                                    "outputs; slower than one PDL launch per projection, see profiles/r02_chain.md")
            except Exception as ex:  # noqa: BLE001 -- an extra, the headline stands
                extra["chained_launch_form"] = {"error": repr(ex)[:300]}
        extra["prefill_ceiling_note"] = ("the per-block scale fold runs on the CUDA cores: one I2FP + two packed FMAs per output pair and "
                                         "quantization block; profiles/microbench/epi_probe.cu measures 469 cycles per 128x128 block for "
                                         "that sequence alone (13.6 % of the int8 MMA rate), profiles/r02_prefill_knockouts.md")

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u4 x s8 -> s32 (dp4a), fp32 fold", "data": "synthetic",
        "config": workload_config(world, tp),     # the same object the reference arm prints
        "launch_form": (
            f"{len(chains)} persistent chained launches per step ({args.chain} layer(s) = {4 * args.chain} grouped projections each, "
            "qgemm_gemv_chain); every projection waits for its predecessor to complete on the whole device" if chains else
            f"{launches_per_step} launches per step, one per (grouped) projection"),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT,
                "h2d_bytes_per_step": sum(v.numel() * 4 for v in acts_host.values()),
                "d2h_bytes_per_step": total_out * 4, "ms_per_step": ms_e2e / args.steps,
                "d2h": (f"every {args.d2h_chunk_layers} layers on a side stream, overlapped with the following layers; the step "
                        "ends when the last slice has landed") if (groups and not chains and plan is None and args.d2h_chunk_layers > 0)
                       else "one copy at the end of the step",
                "api": "quant_gemm.quantize_q8_1 + quant_gemm.gemm (python mirror of the reference extension) "
                       "-> C ABI; weights resident in HBM like the reference API (device pointers)"},
        "gpu_launches": int(launches_per_step * args.steps),
        "gpu_launches_e2e": int(launches_per_e2e * args.steps),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "kernel": "gemv_chain_kernel<Q4_0>" if chains else "gemv_kernel<Q4_0,1>", "peak_source": peak_src,
                     "avg_launch_us": per_launch_us, "algorithmic_bytes_per_launch": per_launch_bytes,
                     "frac_of_nominal_8000": achieved / 8000.0},
        "oracle_check_max_norm_err": check,
        "extra": extra,
    }
    def emit():
        if rank == 0:
            print(json.dumps(line), file=_JSON_OUT, flush=True)

    # the shape that shards (configs[4]).  It comes after the headline measurement and under a watchdog: if a
    # collective wedges, the headline line still goes out and every rank leaves.
    if args.sharded_extra:
        import threading

        def bail():
            extra["sharded_c5"] = {"error": "timed out after 240 s"}
            emit()
            sys.stdout.flush()
            os._exit(0)
        wd = threading.Timer(240.0, bail)
        wd.daemon = True
        wd.start()
        try:
            extra["sharded_c5"] = sharded_c5(torch, dist, quant_gemm, dev, world, rank, ctl)
            add_c5_efficiency(extra["sharded_c5"], world)
        except Exception as ex:  # noqa: BLE001 -- reported, the headline stands
            extra["sharded_c5"] = {"error": repr(ex)[:300]}
        wd.cancel()
    if world > 1:
        dist.barrier(group=ctl)
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_reference_run(steps=10 ** 6, warmup=1, sample_layers=1, budget_s=12.0)
            line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        if args.detail:
            import bench_detail
            bench_detail.run(args.detail)
    emit()
    if world > 1:
        dist.barrier(group=ctl)
        sys.stdout.flush()
        os._exit(0)  # skip NCCL teardown: communicators that were captured into graphs can hang in destroy


if __name__ == "__main__":
    main()
