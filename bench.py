#!/usr/bin/env python
"""bench.py -- FP4 x BF16 GEMM benchmark (BASELINE.json metric) for the B200 build.

Workload (config.workload): the four NVFP4 GEMMs of one Llama-3.3-70B decoder layer
(qkv 10240x8192, o 8192x8192, gate_up 57344x8192, down 8192x28672) at M = 16 decode
tokens, bf16 activations -- BASELINE.json configs[1].  One "step" = one pass over the
layer set.  With --gpus N > 1 the layer is tensor-parallel over N ranks exactly as
Llama TP shards it (qkv/gate_up N-split, no collective; o/down K-split + one NCCL
all-reduce each), so total work is fixed ("strong" scaling).

value  = algorithmic bytes of the whole (unsharded) layer set per second, inputs
         resident in HBM, CUDA-event timed, max over ranks.
e2e    = same, through the public petit_kernel Python API with the activations coming
         from pinned host memory and the outputs copied back, every step.
roofline / cpu_baseline / clocks / details: see DESIGN.md "Measurement".

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--m M]
                  [--dump-outputs DIR]

--dump-outputs DIR writes the outputs of the last timed step as DIR/<gemm>.npy (float32) so
that two builds can be compared output for output: the inputs depend only on the arguments.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "petit-kernel_b200"))
sys.path.insert(0, ROOT)

LAYER = [("qkv", 10240, 8192, "column"), ("o", 8192, 8192, "row"),
         ("gate_up", 57344, 8192, "column"), ("down", 8192, 28672, "row")]
METRIC = "FP4xBF16 GEMM algorithmic HBM GB/s, Llama-3.3-70B decoder-layer GEMM set (NVFP4, M=16)"
DUMP_LIMIT = 64 << 20  # bytes written by --dump-outputs, per run


def dump_outputs(dirname, named, limit=DUMP_LIMIT, suffix=""):
    """Write each [m, n] output of `named` ((name, tensor) pairs) as DIR/<name><suffix>.npy in
    float32.  Above `limit` bytes in all, the same seeded sample of rows is kept from each."""
    import numpy as np

    os.makedirs(dirname, exist_ok=True)
    m = named[0][1].shape[0]
    row_bytes = sum(c[0].numel() for _, c in named) * 4
    rows = None
    if m * row_bytes > limit:
        keep = max(1, limit // row_bytes)
        rows = torch.from_numpy(np.sort(np.random.RandomState(0).choice(m, keep, replace=False)))
    for name, c in named:
        if rows is not None:
            c = c[rows.to(c.device)]
        np.save(os.path.join(dirname, name + suffix + ".npy"), c.float().cpu().numpy())


def algo_bytes(m, n, k, group=16):
    # SURVEY.md 8(d): fp4 + scales + A + C + global scale
    return n * k // 2 + n * k // group + 2 * m * k + 2 * m * n + 4


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p["bf16_tflops"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([x.strip() for x in line.split(",")])

    def wait_started(self, timeout=5.0):
        t0 = time.time()
        while self.proc and not self.samples and time.time() - t0 < timeout:
            time.sleep(0.02)

    def mark(self):
        return len(self.samples)

    def stop(self, lo=0, hi=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        window = self.samples[lo:hi] or self.samples
        self.samples = window
        mhz = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for nm, v in zip(names, s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        mx = next((int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()), None)
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(mhz)}


# ------------------------------------------------------------------ CPU reference arm
def cpu_case(g, m, n, k):
    """One seeded NVFP4 problem for the CPU arm: activations, packed weights, scales, global scale."""
    a = torch.randn((m, k), generator=g).to(torch.bfloat16)
    q = torch.randint(0, 256, (n, k // 2), generator=g, dtype=torch.uint8)
    s = (torch.rand((n, k // 16), generator=g) * 3.5 + 0.25).to(torch.float8_e4m3fn)
    return a, q, s, torch.ones(1)


def cpu_reference_rate(m, shapes, reps):
    """The reference's CPU path (torch dequantise + fp32 matmul,
    tests/ops/test_fp4_gemm_quark.py:9-24) restated in oracle/, on the host cores."""
    from oracle import petit_oracle as orc

    g = torch.Generator().manual_seed(0)
    total_bytes, total_s, last = 0, 0.0, []
    for (nm, n, k, _) in shapes:
        a, q, s, gs = cpu_case(g, m, n, k)
        orc.nvfp4_gemm_ref_torch(a[:, :256], q[:64, :128], s[:64, :16], gs)  # warm torch
        t0 = time.perf_counter()
        for _ in range(reps):
            c = orc.nvfp4_gemm_ref_torch(a, q, s, gs)
        total_s += time.perf_counter() - t0
        total_bytes += reps * algo_bytes(m, n, k)
        last.append((nm, c))
    return total_bytes / total_s / 1e9, total_s, last


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to every rank: the CPU arm uses all host cores at
    # every N, so its value does not depend on how it was launched
    torch.set_num_threads(os.cpu_count() or 1)
    shapes = [LAYER[1]]  # o_proj 8192 x 8192: bounded sample of the layer set
    steps = args.steps
    for _ in range(min(args.warmup, 1)):
        cpu_reference_rate(args.m, shapes, 1)
    t0 = time.perf_counter()
    gbs, secs, last = cpu_reference_rate(args.m, shapes, steps)
    wall = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    out = {
        "impl": "reference", "metric": METRIC, "value": gbs, "unit": "GB/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1),
        "ms_per_step": secs / steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": torch.get_num_threads(),
                         "kind": "port",
                         "sample": f"o_proj 8192x8192 NVFP4 M={args.m}, {steps} passes of torch "
                                   f"dequant+fp32 matmul (oracle/petit_oracle.py), {wall:.1f} s"},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


def workload_config(args, world):
    return {"workload": f"Llama-3.3-70B decoder-layer GEMM set qkv/o/gate_up/down, NVFP4 weights, "
                        f"bf16 activations, M={args.m}",
            "m": args.m, "shapes": {n: [a, b] for n, a, b, _ in LAYER},
            "parallelism": f"tp{world}" if world > 1 else "single",
            "allreduce": getattr(args, "allreduce_kind", "none"),
            "launch": "cuda-graph per layer step" if getattr(args, "graph", False)
            else "eager launches on one stream, programmatic dependent launch between GEMMs",
            "l2": "weights rotate over distinct copies > 2x L2 (126 MB) between reuses"}


# ------------------------------------------------------------------ GPU arm
def make_inputs(pk, shard, m, dev, rank):
    """Seeded inputs of the GPU arm: `copies` distinct packed copies of the (sharded) layer set,
    together larger than L2, the global scale and one activation per K.  The same arguments
    always give the same inputs.  Returns them with the generator, which later code draws on."""
    set_bytes = sum(n * k // 2 + n * k // 16 for _, n, k, _ in shard)
    copies = max(2, int(300e6 // set_bytes) + 2)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    layers = []
    for _ in range(copies):
        one = []
        for nm, n, k, kind in shard:
            q = torch.randint(0, 256, (n, k // 2), generator=g, dtype=torch.uint8, device=dev)
            s = (torch.rand((n, k // 16), generator=g, device=dev) * 3.5 + 0.25).to(torch.float8_e4m3fn)
            b = pk.repack_nvfp4(q.view(torch.int32), n, k)
            sp = pk.process_nvfp4_scales(s, n, k)
            one.append((nm, n, k, kind, b, sp))
            del q, s
        layers.append(one)
    gs = torch.rand(1, generator=g, device=dev) * 1.5 + 0.5
    acts = {k: torch.randn((m, k), generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)
            for k in {k for _, _, k, _ in shard}}
    return layers, copies, gs, acts, g


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500,
                    help="timed steps.  With --impl reference every step is a host-CPU pass of the "
                         "o_proj dequantise + fp32 matmul (about 0.3 s on an 8-core x86 host), so "
                         "the default of 500 takes minutes there")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--m", type=int, default=16)
    ap.add_argument("--no-details", action="store_true")
    ap.add_argument("--no-competitors", action="store_true",
                    help="skip the cuBLAS / vLLM Marlin comparator rows of `details`")
    ap.add_argument("--graph", action="store_true",
                    help="replay one captured CUDA graph per layer step instead of eager launches")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<gemm>.npy (float32; "
                         "a seeded sample of rows when they exceed 64 MB; one file per rank "
                         "with --gpus > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import petit_kernel as pk  # fails loudly without the CUDA extension
    import petit_tp

    dev = torch.device("cuda", local)
    m = args.m
    hbm_peak, tf_peak, peak_src = peaks()

    # ---- build the (sharded) layer set, several distinct copies to defeat L2
    shard = [(nm,) + petit_tp.shard_shape(n, k, kind, world) + (kind,) for nm, n, k, kind in LAYER]
    layers, copies, gs, acts, g = make_inputs(pk, shard, m, dev, rank)

    # row-parallel outputs (o, down): PETIT_TP_ALLREDUCE = fused (default) | peer | nccl | symm
    #   fused: ONE kernel per rank computes the K-split GEMM and all-reduces its output -- the
    #         CTA that finishes a tile pushes its partial to the peers over NVLink and sums
    #         theirs (csrc/fp4_gemm.cu "fused all-reduce", petit_tp.FusedAllReduce);
    #   peer: the GEMM writes into a peer-mapped buffer and this package's one-shot
    #         all-reduce kernel (csrc/allreduce.cu) sums all ranks' buffers over NVLink --
    #         one PDL-chained launch, ~5 us of host time;
    #   nccl: dist.all_reduce; symm: torch.ops.symm_mem.one_shot_all_reduce.
    symm = None
    peer = None
    fused = None
    allreduce_kind = "none" if world == 1 else "nccl"
    want_ar = os.environ.get("PETIT_TP_ALLREDUCE", "fused")
    if world > 1 and want_ar == "fused" and m <= 64:
        try:
            fused = petit_tp.FusedAllReduce()
            for j, (nm, n, k, kind) in enumerate(shard):
                if kind == "row":
                    fused._context(n, dev, j)
            torch.cuda.synchronize()
            allreduce_kind = "fused into the row-parallel GEMM (packets over NVLink peer memory)"
        except Exception as exc:  # fall back to NCCL, loudly
            if rank == 0:
                print(f"[bench] fused all-reduce unavailable ({exc}); using NCCL", file=sys.stderr)
            fused = None
    if world > 1 and want_ar == "peer":
        try:
            peer = petit_tp.PeerAllReduce()
            for j, (nm, n, k, kind) in enumerate(shard):
                if kind == "row":
                    buf = peer.buffer(m, n, torch.bfloat16, dev, j)
                    buf.zero_()
                    peer.reduce(buf)
            torch.cuda.synchronize()
            allreduce_kind = "petit one-shot peer-memory all-reduce kernel (NVLink P2P)"
        except Exception as exc:  # fall back to NCCL, loudly
            if rank == 0:
                print(f"[bench] peer-memory all-reduce unavailable ({exc}); using NCCL",
                      file=sys.stderr)
            peer = None
    if world > 1 and want_ar == "symm":
        try:
            symm = petit_tp.SymmAllReduce()
            for j, (nm, n, k, kind) in enumerate(shard):
                if kind == "row":
                    symm.reduce(symm.buffer(m, n, torch.bfloat16, dev, j).zero_())
            torch.cuda.synchronize()
            allreduce_kind = "symm_mem.one_shot_all_reduce"
        except Exception as exc:  # fall back to NCCL, loudly
            if rank == 0:
                print(f"[bench] symmetric-memory all-reduce unavailable ({exc}); using NCCL",
                      file=sys.stderr)
            symm = None

    def layer_step(i, a_by_k=acts, collective=True):
        outs = []
        for j, (nm, n, k, kind, b, sp) in enumerate(layers[i % copies]):
            if kind == "row" and world > 1 and collective and fused is not None:
                c = fused.matmul(a_by_k[k], b, sp, gs, n, k, slot=j)
            elif kind == "row" and world > 1 and collective and peer is not None:
                buf = peer.buffer(m, n, torch.bfloat16, dev, j)
                pk.ops.mul_nvfp4_a16_out(buf, a_by_k[k], b, sp, gs, m, n, k, -1)
                c = peer.reduce(buf)
            elif kind == "row" and world > 1 and collective and symm is not None:
                buf = symm.buffer(m, n, torch.bfloat16, dev, j)
                pk.ops.mul_nvfp4_a16_out(buf, a_by_k[k], b, sp, gs, m, n, k, -1)
                c = symm.reduce(buf)
            else:
                c = pk.mul_nvfp4_a16(a_by_k[k], b, sp, gs, m, n, k, -1)
                if kind == "row" and world > 1 and collective:
                    dist.all_reduce(c)
            outs.append(c)
        return outs

    args.allreduce_kind = allreduce_kind

    # ---- TP outputs checked once before anything is timed: the row-parallel results of the
    # data plane that is about to be measured against ncclAllReduce of the same partials
    tp_check = None
    if world > 1:
        outs = layer_step(0)
        parts = layer_step(0, collective=False)
        max_abs, max_ref, identical = 0.0, 0.0, True
        for (nm, n, k, kind, _, _), got, part in zip(layers[0], outs, parts):
            if kind != "row":
                continue
            ref = part.clone()
            dist.all_reduce(ref)
            max_abs = max(max_abs, (got.float() - ref.float()).abs().max().item())
            max_ref = max(max_ref, ref.float().abs().max().item())
            gathered = [torch.empty_like(got) for _ in range(world)]
            dist.all_gather(gathered, got.contiguous())
            identical = identical and all(torch.equal(gathered[0], x) for x in gathered)
        tp_check = {"vs": "ncclAllReduce of the same bf16 partials", "max_abs_diff": max_abs,
                    "max_abs_ref": max_ref, "identical_across_ranks": identical,
                    # NCCL rounds to bf16 per hop, the one-shot kernel once: one bf16 ulp of max
                    "ok": bool(max_abs <= max_ref * 2 ** -6 and identical)}
        if not tp_check["ok"]:
            raise RuntimeError(f"TP output check failed: {tp_check}")

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    full_bytes = sum(algo_bytes(m, n, k) for _, n, k, _ in LAYER)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    # ---- optional CUDA graphs (--graph): one captured layer step per weight copy.  Not the
    # default: with PDL the eager stream is as fast at TP1 (129 vs 127 us/step measured)
    # and capturing NCCL collectives hung at TP2 on this stack.
    use_graph = args.graph
    graphs = None
    graph_outs = []
    if use_graph:
        try:
            for i in range(copies):  # warm every path (workspace, NCCL) before capture
                layer_step(i)
            sync()
            graphs = []
            side = torch.cuda.Stream()
            for i in range(copies):
                gph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gph, stream=side):
                    graph_outs.append(layer_step(i))
                graphs.append(gph)
            sync()
        except Exception as exc:
            if rank == 0:
                print(f"[bench] CUDA graph capture failed ({exc}); timing eager launches",
                      file=sys.stderr)
            graphs = None
    eager_step = layer_step

    def timed_step(i):
        if graphs is not None:
            graphs[i % copies].replay()
            return graph_outs[i % copies]
        return eager_step(i)

    # ---- device-resident timing
    for i in range(args.warmup):
        timed_step(i)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_started()
    sync()
    lo = sampler.mark()
    e0.record()
    for i in range(args.steps - 1):
        timed_step(i)
    # only the last step's outputs are kept (--dump-outputs): every earlier step drops its
    # own before the next allocates, so the allocator hands out the same blocks each step
    last = timed_step(args.steps - 1)
    e1.record()
    sync()
    ms = e0.elapsed_time(e1)
    hi = sampler.mark()
    if hi - lo < 3:
        # timed region shorter than the 20 ms sampling period: keep the same load
        # running (untimed) until a few samples exist
        t_end = time.time() + 0.25
        i = 0
        while time.time() < t_end:
            layer_step(i, collective=False)  # rank-local load only: no unmatched collectives
            i += 1
        torch.cuda.synchronize()
        hi = sampler.mark()
    clocks = sampler.stop(lo, hi) if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "timed region" if hi - lo >= 3 else "timed region + same load repeated"
    if args.dump_outputs:
        # (the untimed filler load above allocates its own outputs: `last` is untouched)
        dump_outputs(args.dump_outputs, [(x[0], c) for x, c in zip(shard, last)],
                     DUMP_LIMIT // world, f"_rank{rank}" if world > 1 else "")
    del last
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = t.item() / args.steps
    value = full_bytes / (ms_step * 1e-3) / 1e9

    # ---- end to end: host activations in, host outputs out, every step.
    # Three streams, double buffered: the H2D copy of step i+1 and the D2H copy of step
    # i-1 run beside the GEMMs of step i (PCIe moves ~4 MB per step = 70 us if serialised
    # on the compute stream, more than half a step).  Every step still copies its own
    # inputs from pinned host memory and its own outputs back; the timed region ends
    # only after the last D2H copy has finished.
    host_a = {k: v.cpu().pin_memory() for k, v in acts.items()}
    nbuf = 2
    dev_a = [{k: torch.empty_like(v) for k, v in acts.items()} for _ in range(nbuf)]
    dev_c = [[torch.empty((m, n), dtype=torch.bfloat16, device=dev) for _, n, _, _ in shard]
             for _ in range(nbuf)]
    host_c = [[torch.empty((m, n), dtype=torch.bfloat16).pin_memory() for _, n, _, _ in shard]
              for _ in range(nbuf)]
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    ev_in = [torch.cuda.Event() for _ in range(nbuf)]
    ev_cmp = [torch.cuda.Event() for _ in range(nbuf)]
    ev_out = [torch.cuda.Event() for _ in range(nbuf)]
    for ev in ev_cmp + ev_out:
        ev.record()

    def layer_step_out(i, a_by_k, outs):
        for j, (nm, n, k, kind, b, sp) in enumerate(layers[i % copies]):
            if kind == "row" and world > 1 and fused is not None:
                fused.matmul(a_by_k[k], b, sp, gs, n, k, out=outs[j], slot=j)
                continue
            if kind == "row" and world > 1 and peer is not None:
                buf = peer.buffer(m, n, torch.bfloat16, dev, j)
                pk.ops.mul_nvfp4_a16_out(buf, a_by_k[k], b, sp, gs, m, n, k, -1)
                peer.reduce(buf, out=outs[j])
                continue
            pk.ops.mul_nvfp4_a16_out(outs[j], a_by_k[k], b, sp, gs, m, n, k, -1)
            if kind == "row" and world > 1:
                if symm is not None:
                    buf = symm.buffer(m, n, torch.bfloat16, dev, j)
                    buf.copy_(outs[j])
                    outs[j].copy_(symm.reduce(buf))
                else:
                    dist.all_reduce(outs[j])

    def e2e_step(i):
        b = i % nbuf
        cur = torch.cuda.current_stream()
        s_in.wait_event(ev_cmp[b])   # the GEMMs of step i-2 have consumed dev_a[b]
        with torch.cuda.stream(s_in):
            for k in dev_a[b]:
                dev_a[b][k].copy_(host_a[k], non_blocking=True)
            ev_in[b].record(s_in)
        cur.wait_event(ev_in[b])
        cur.wait_event(ev_out[b])    # the D2H copies of step i-2 have drained dev_c[b]
        layer_step_out(i, dev_a[b], dev_c[b])
        ev_cmp[b].record(cur)
        s_out.wait_event(ev_cmp[b])
        with torch.cuda.stream(s_out):
            for h, c in zip(host_c[b], dev_c[b]):
                h.copy_(c, non_blocking=True)
            ev_out[b].record(s_out)

    def e2e_drain():
        cur = torch.cuda.current_stream()
        for ev in ev_out:
            cur.wait_event(ev)

    # (the e2e leg is always eager: its cross-stream events are not capturable as is)
    e2e_timed = e2e_step

    for i in range(args.warmup):
        e2e_timed(i)
    sync()
    e0.record()
    for i in range(args.steps):
        e2e_timed(i)
    e2e_drain()
    e1.record()
    sync()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = full_bytes / (t.item() / args.steps * 1e-3) / 1e9
    h2d = sum(v.numel() * 2 for v in host_a.values())
    d2h = sum(h.numel() * 2 for h in host_c[0])

    # ---- roofline of the dominant kernel (the stream-K GEMM), per launch, live
    per_launch = []
    names0 = [x[0] for x in layers[0]]
    for j, (nm, n, k, kind, _, _) in enumerate(layers[0]):
        # row-parallel layers under TP: the launch that is timed is the fused GEMM + all-reduce
        # (every rank runs the same loop, so the calls match up); the max over ranks is kept
        with_ar = kind == "row" and world > 1 and fused is not None

        def one(i):
            b, sp = layers[i % copies][names0.index(nm)][4:6]
            if with_ar:
                fused.matmul(acts[k], b, sp, gs, n, k, slot=j)
            else:
                pk.mul_nvfp4_a16(acts[k], b, sp, gs, m, n, k, -1)

        def timed_us(fn, reps=20):
            for i in range(3):
                fn(i)
            sync()
            e0.record()
            for i in range(reps):
                fn(i)
            e1.record()
            torch.cuda.synchronize()
            tl = torch.tensor([e0.elapsed_time(e1) / reps * 1e3], device=dev)
            if world > 1:
                dist.all_reduce(tl, op=dist.ReduceOp.MAX)
            return tl.item()

        us = timed_us(one)
        row = {"gemm": nm, "n": n, "k": k, "us": round(us, 2),
               "gbs": round(algo_bytes(m, n, k) / us * 1e-3, 1),
               "frac_hbm": round(algo_bytes(m, n, k) / us * 1e-3 / hbm_peak, 4),
               "includes_allreduce": bool(with_ar)}
        if with_ar:
            # the same shard GEMM without the exchange: what the fused all-reduce adds
            def plain(i):
                b, sp = layers[i % copies][names0.index(nm)][4:6]
                pk.mul_nvfp4_a16(acts[k], b, sp, gs, m, n, k, -1)

            row["gemm_only_us"] = round(timed_us(plain), 2)
        per_launch.append(row)
    tp_breakdown = None
    if world > 1:
        col = sum(p["us"] for p in per_launch if not p["includes_allreduce"])
        row_fused = sum(p["us"] for p in per_launch if p["includes_allreduce"])
        row_plain = sum(p.get("gemm_only_us", 0.0) for p in per_launch if p["includes_allreduce"])
        tp_breakdown = {"column_parallel_gemm_us": round(col, 2), "row_parallel_gemm_only_us": round(row_plain, 2),
                        "row_parallel_with_allreduce_us": round(row_fused, 2),
                        "allreduce_extra_us": round(row_fused - row_plain, 2) if row_plain else None,
                        "note": "per-launch event times, max over ranks; the step overlaps neighbours by PDL"}
    shard_bytes = sum(algo_bytes(m, n, k) for _, n, k, _ in shard)
    avg_launch_us = sum(p["us"] for p in per_launch) / len(per_launch)
    achieved = (shard_bytes / len(shard)) / avg_launch_us * 1e-3
    # dram__bytes_read+write per launch comes from an ncu capture of the unsharded layer set
    # (profiles/): it only describes the N=1 workload
    traffic = None
    if world == 1:
        for name in ("r02_dram_traffic.json", "r01_dram_traffic.json"):
            try:
                with open(os.path.join(ROOT, "profiles", name)) as f:
                    traffic = json.load(f).get("avg_bytes_per_launch_m16")
                break
            except Exception:
                pass
    roofline = {"bound": "hbm", "achieved": round(achieved, 1), "peak": hbm_peak, "unit": "GB/s",
                "frac": round(achieved / hbm_peak, 4), "traffic": traffic,
                "peak_source": peak_src, "kernel": "fp4_gemm_kernel<nvfp4,bf16,tok16> (stream-K tcgen05)",
                "per_launch": per_launch}

    # ---- TP only: the same sharded layer step at the other ends of config 5's M range
    tp_m_sweep = None
    if world > 1:
        tp_m_sweep = []
        for mm in (1, 64):
            acts_mm = {k: torch.randn((mm, k), generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)
                       for k in acts}

            def step_mm(i):
                for j, (nm, n, k, kind, b, sp) in enumerate(layers[i % copies]):
                    if kind == "row" and fused is not None:
                        fused.matmul(acts_mm[k], b, sp, gs, n, k, slot=j)
                    else:
                        c = pk.mul_nvfp4_a16(acts_mm[k], b, sp, gs, mm, n, k, -1)
                        if kind == "row":
                            if peer is not None:
                                buf = peer.buffer(mm, n, torch.bfloat16, dev, 8 + j)
                                buf.copy_(c)
                                peer.reduce(buf)
                            else:
                                dist.all_reduce(c)

            for i in range(5):
                step_mm(i)
            sync()
            e0.record()
            for i in range(100):
                step_mm(i)
            e1.record()
            sync()
            tm = torch.tensor([e0.elapsed_time(e1) / 100], device=dev)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            by = sum(algo_bytes(mm, n, k) for _, n, k, _ in LAYER)
            tp_m_sweep.append({"m": mm, "us_per_step": round(tm.item() * 1e3, 2),
                               "gbs": round(by / (tm.item() * 1e-3) / 1e9, 1)})

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    details = None
    if world == 1 and not args.no_details:
        details = sweep_details(pk, layers, copies, gs, dev, hbm_peak, tf_peak,
                                with_competitors=not args.no_competitors)

    torch.set_num_threads(os.cpu_count() or 1)  # torchrun pins OMP_NUM_THREADS=1
    cores = torch.get_num_threads()
    t0 = time.perf_counter()
    cpu_gbs, cpu_s, _ = cpu_reference_rate(m, [LAYER[1]], 2)
    cpu = {"value": round(cpu_gbs, 3), "unit": "GB/s", "cores": cores, "kind": "port",
           "sample": f"o_proj 8192x8192 NVFP4 M={m}, 2 passes of the torch dequant+fp32-matmul "
                     f"oracle on the host ({time.perf_counter() - t0:.1f} s)"}

    out = {
        "metric": METRIC, "value": round(value, 1), "unit": "GB/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 5),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic", "config": workload_config(args, world),
        "e2e": {"value": round(e2e_value, 1), "unit": "GB/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h},
        # our own kernels in the timed region: the GEMMs, plus the peer all-reduce launches
        "gpu_launches": args.steps * (len(shard) + (sum(1 for x in shard if x[3] == "row")
                                                    if (world > 1 and peer is not None) else 0)),
        "launches_per_step": {"gemm": len(shard),
                              "allreduce": (0 if (world == 1 or fused is not None)
                                            else sum(1 for x in shard if x[3] == "row"))},
        "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
        "frac_of_hbm_peak_layer_set": round(value / (hbm_peak * world), 4),
    }
    if tp_check is not None:
        out["tp_check"] = tp_check
    if tp_m_sweep is not None:
        out["tp_m_sweep"] = tp_m_sweep
    if tp_breakdown is not None:
        out["tp_breakdown"] = tp_breakdown
    if details:
        out["details"] = details
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def _timed(fn, reps, e0, e1):
    for i in range(3):
        fn(i)
    torch.cuda.synchronize()
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


def moe_grouped(pk, dev, hbm_peak, e0, e1):
    rows = []
    g = torch.Generator(device=dev).manual_seed(11)
    for name, n, k, counts in (("w13 8 experts", 28672, 4096, [4, 5, 3, 4, 6, 2, 4, 4]),
                               ("w2 8 experts", 4096, 14336, [4, 5, 3, 4, 6, 2, 4, 4]),
                               ("w13 8 experts", 28672, 4096, [16, 20, 12, 16, 24, 8, 16, 16]),
                               ("64 experts 2048x2048", 2048, 2048, [2] * 64)):
        e = len(counts)
        stacks = []
        for _ in range(2):  # two stacks of experts in rotation: > 2x L2 between reuses
            b = torch.randint(-2 ** 31, 2 ** 31 - 1, (e, n // 16, 2 * k), dtype=torch.int32, device=dev, generator=g)
            sc = torch.randint(0x30, 0x50, (e, n, k // 16), dtype=torch.uint8, device=dev,
                               generator=g).view(torch.float8_e4m3fn)
            stacks.append((b, sc))
        gs = torch.ones(e, dtype=torch.float32, device=dev)
        offsets = [0]
        for c in counts:
            offsets.append(offsets[-1] + c)
        a = torch.randn((offsets[-1], k), generator=g, device=dev).to(torch.bfloat16)
        out = torch.empty((offsets[-1], n), dtype=torch.bfloat16, device=dev)
        by = sum(1 for c in counts if c) * (n * k // 2 + n * k // 16) + offsets[-1] * (k + n) * 2
        row = {"case": name, "n": n, "k": k, "tokens_per_expert": counts if e <= 8 else f"{counts[0]} x {e}"}
        for key, env in (("single_launch", "1"), ("one_by_one", "0")):
            os.environ["PETIT_GROUPED_SINGLE"] = env
            us = _timed(lambda i: pk.ops.mul_fp4_a16_grouped_out(out, a, stacks[i % 2][0], stacks[i % 2][1], gs,
                                                                 offsets, n, k, -1, False), 20, e0, e1)
            row[key] = {"us": round(us, 2), "gbs": round(by / us * 1e-3), "frac_hbm": round(by / us * 1e-3 / hbm_peak, 3)}
        os.environ.pop("PETIT_GROUPED_SINGLE", None)
        rows.append(row)
        del stacks
        torch.cuda.empty_cache()
    return rows


def competitors(pk, layers, copies, gs, dev, hbm_peak, tf_peak):
    """Same-box library comparators (BASELINE.md section 4; the role of the reference bench's
    hipBLASLt backend, tools/benchmarks/matmul/rocm/matmul_hipblaslt.cc:220-263), same CUDA
    event method and weight rotation as the rest of this file:
      * cuBLAS bf16 (torch.matmul) on weights dequantised ahead of time -- 4x the weight bytes;
      * vLLM 0.22's Marlin FP4 W4A16 kernel (mma.sync path) on the same NVFP4 tensors.
    Reported per shape and M; `vs_ours` = their us / our us on the same box."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g = torch.Generator(device=dev).manual_seed(11)
    out = {"cublas_bf16_dense": [], "vllm_marlin_fp4": [], "notes": []}
    names = [x[0] for x in layers[0]]
    ms = (1, 16, 64, 1024)
    ours = {}
    for nm, n, k, _, _, _ in layers[0]:
        idx = names.index(nm)
        for m in ms:
            a = torch.randn((m, k), generator=g, device=dev).to(torch.bfloat16)
            ours[(nm, m)] = _timed(lambda i: pk.mul_nvfp4_a16(a, layers[i % copies][idx][4],
                                                               layers[i % copies][idx][5], gs, m, n, k, -1),
                                   20 if m <= 64 else 5, e0, e1)
    # ---- cuBLAS bf16 on pre-dequantised weights (distinct dense copies > L2)
    for nm, n, k, _, _, _ in layers[0]:
        idx = names.index(nm)
        ncopy = max(2, min(copies, int(400e6 // (n * k * 2)) + 1))
        dense = [pk.ops.dequant_dense(layers[c % copies][idx][4], layers[c % copies][idx][5], 1.0,
                                      torch.bfloat16, n, k, False, True) for c in range(ncopy)]
        for m in ms:
            a = torch.randn((m, k), generator=g, device=dev).to(torch.bfloat16)
            us = _timed(lambda i: torch.matmul(a, dense[i % ncopy].t()), 20 if m <= 64 else 5, e0, e1)
            by = 2 * n * k + 2 * m * k + 2 * m * n
            out["cublas_bf16_dense"].append({
                "gemm": nm, "m": m, "us": round(us, 2), "ours_us": round(ours[(nm, m)], 2),
                "vs_ours": round(us / ours[(nm, m)], 2), "bytes": by,
                "frac_hbm_own_bytes": round(by / us * 1e-3 / hbm_peak, 3),
                "tflops": round(2.0 * m * n * k / us * 1e-6, 1)})
        del dense
        torch.cuda.empty_cache()
    # ---- vLLM Marlin FP4 (W4A16, NVFP4 weights)
    try:
        from vllm.model_executor.layers.quantization.utils import marlin_utils_fp4 as mfp4

        class _L(torch.nn.Module):
            pass

        for nm, n, k, _, _, _ in layers[0]:
            lays = []
            for c in range(2):
                q = torch.randint(0, 256, (n, k // 2), generator=g, dtype=torch.uint8, device=dev)
                sc = (torch.rand((n, k // 16), generator=g, device=dev) * 3.5 + 0.25).to(torch.float8_e4m3fn)
                lay = _L()
                lay.output_size_per_partition, lay.input_size_per_partition = n, k
                lay.params_dtype = torch.bfloat16
                lay.weight = torch.nn.Parameter(q, requires_grad=False)
                lay.weight_scale = torch.nn.Parameter(sc, requires_grad=False)
                lay.weight_global_scale = torch.nn.Parameter(torch.ones(1, device=dev), requires_grad=False)
                mfp4.prepare_fp4_layer_for_marlin(lay)
                lays.append(lay)
            for m in ms:
                a = torch.randn((m, k), generator=g, device=dev).to(torch.bfloat16)

                def run(i, lays=lays, a=a, n=n, k=k):
                    lay = lays[i % 2]
                    return mfp4.apply_fp4_marlin_linear(a, lay.weight, lay.weight_scale,
                                                        lay.weight_global_scale, lay.workspace, n, k)

                us = _timed(run, 20 if m <= 64 else 5, e0, e1)
                out["vllm_marlin_fp4"].append({
                    "gemm": nm, "m": m, "us": round(us, 2), "ours_us": round(ours[(nm, m)], 2),
                    "vs_ours": round(us / ours[(nm, m)], 2),
                    "frac_hbm": round(algo_bytes(m, n, k) / us * 1e-3 / hbm_peak, 3),
                    "tflops": round(2.0 * m * n * k / us * 1e-6, 1)})
            del lays
            torch.cuda.empty_cache()
        out["notes"].append("vLLM Marlin: 2 weight copies per shape (qkv / o fit in L2 between reuses: "
                            "an upper bound on its speed for those two)")
    except Exception as exc:  # not fatal: the comparator is a library outside this repo
        out["vllm_marlin_fp4"] = None
        out["notes"].append(f"vLLM Marlin FP4 unavailable on this box: {type(exc).__name__}: {str(exc)[:200]}")
    return out


def sweep_details(pk, layers, copies, gs, dev, hbm_peak, tf_peak, with_competitors=True):
    """BASELINE metric in full: us / GB/s / % HBM at M = 1..16 (NVFP4 bf16 + fp16, MXFP4), the
    mid-M points, TFLOPS / % peak at M = 256..8192, per shape.  Outside the headline timed region."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {"decode_nvfp4_bf16": [], "decode_nvfp4_fp16": [], "decode_mxfp4_bf16": [],
           "mid_m_nvfp4_bf16": [], "prefill_nvfp4_bf16": []}
    g = torch.Generator(device=dev).manual_seed(7)
    names = [x[0] for x in layers[0]]

    def hbm_row(nm, m, us, group=16):
        n, k = [(x[1], x[2]) for x in layers[0] if x[0] == nm][0]
        by = algo_bytes(m, n, k, group)
        return {"gemm": nm, "m": m, "us": round(us, 2), "gbs": round(by / us * 1e-3),
                "frac_hbm": round(by / us * 1e-3 / hbm_peak, 3)}

    for nm, n, k, _, _, _ in layers[0]:
        idx = names.index(nm)
        for m in (1, 4, 8, 16):
            a = torch.randn((m, k), generator=g, device=dev).to(torch.bfloat16)
            us = _timed(lambda i: pk.mul_nvfp4_a16(a, layers[i % copies][idx][4], layers[i % copies][idx][5],
                                                   gs, m, n, k, -1), 20, e0, e1)
            res["decode_nvfp4_bf16"].append(hbm_row(nm, m, us))
        for m in (32, 64):
            a = torch.randn((m, k), generator=g, device=dev).to(torch.bfloat16)
            us = _timed(lambda i: pk.mul_nvfp4_a16(a, layers[i % copies][idx][4], layers[i % copies][idx][5],
                                                   gs, m, n, k, -1), 20, e0, e1)
            row = hbm_row(nm, m, us)
            row["tflops"] = round(2.0 * m * n * k / us * 1e-6, 1)
            res["mid_m_nvfp4_bf16"].append(row)
        a = torch.randn((16, k), generator=g, device=dev).to(torch.float16)
        us = _timed(lambda i: pk.mul_nvfp4_a16(a, layers[i % copies][idx][4], layers[i % copies][idx][5],
                                               gs, 16, n, k, -1), 20, e0, e1)
        row = hbm_row(nm, 16, us)
        row["weight_layout"] = "default (bf16-native)"
        res["decode_nvfp4_fp16"].append(row)
    # fp16 activations on weights repacked for them (petit_utils.repack_nvfp4_for(..., float16))
    from petit_kernel import petit_utils as pu
    for nm, n, k, _, _, _ in layers[0]:
        ncopy = max(2, int(300e6 // (n * k // 2 + n * k // 16)) + 1)
        packs = []
        for _ in range(ncopy):
            q = torch.randint(0, 256, (n, k // 2), generator=g, dtype=torch.uint8, device=dev)
            s = (torch.rand((n, k // 16), generator=g, device=dev) * 3.5 + 0.25).to(torch.float8_e4m3fn)
            packs.append((pu.repack_nvfp4_for(q.view(torch.int32), n, k, torch.float16),
                          pk.process_nvfp4_scales(s, n, k)))
            del q, s
        for m in (1, 16):
            a = torch.randn((m, k), generator=g, device=dev).to(torch.float16)
            us = _timed(lambda i: pk.mul_nvfp4_a16(a, packs[i % ncopy][0], packs[i % ncopy][1], gs, m, n, k, -1),
                        20, e0, e1)
            row = hbm_row(nm, m, us)
            row["weight_layout"] = "fp16-native"
            res["decode_nvfp4_fp16"].append(row)
        del packs
        torch.cuda.empty_cache()
    # MXFP4 (config 3): all four shapes, M = 1, 4, 8, 16
    for nm, n, k, _, _, _ in layers[0]:
        ncopy = max(2, int(300e6 // (n * k // 2 + n * k // 32)) + 1)
        packs = []
        for _ in range(ncopy):
            q = torch.randint(0, 256, (n, k // 2), generator=g, dtype=torch.uint8, device=dev)
            s = torch.randint(108, 125, (n, k // 32), generator=g, dtype=torch.uint8, device=dev)  # 2^-19..2^-3, typical of MX weights
            packs.append((pk.repack_mxfp4(q.view(torch.int32), n, k), pk.process_mxfp4_scales(s, n, k)))
            del q, s
        for m in (1, 4, 8, 16):
            a = torch.randn((m, k), generator=g, device=dev).to(torch.bfloat16)
            us = _timed(lambda i: pk.mul_mxfp4_a16(a, packs[i % ncopy][0], packs[i % ncopy][1], gs, m, n, k, -1),
                        20, e0, e1)
            res["decode_mxfp4_bf16"].append(hbm_row(nm, m, us, 32))
        del packs
        torch.cuda.empty_cache()
    # grouped (MoE) GEMM, SURVEY section 8 row f4: Mixtral-8x7B-size experts, a decode step's tokens
    # spread over the experts; one launch for all experts against the experts issued one by one
    res["moe_grouped_nvfp4_bf16"] = moe_grouped(pk, dev, hbm_peak, e0, e1)
    # prefill after the decode rows: it power-caps the part, and the decode kernels are
    # issue-bound (clock-sensitive).  The denominator is the BURST bf16 peak, so every shape
    # starts from an idle part (1 s pause): back to back the sweep runs into the 1 kW power cap
    # and measures the sustained clock instead (down M=2048: 58 % vs 83 % in isolation).
    for nm, n, k, _, _, _ in layers[0]:
        idx = names.index(nm)
        torch.cuda.synchronize()
        time.sleep(1.0)
        for m in (256, 512, 1024, 2048, 4096, 8192):
            a = torch.randn((m, k), generator=g, device=dev).to(torch.bfloat16)
            us = _timed(lambda i: pk.mul_nvfp4_a16(a, layers[i % copies][idx][4], layers[i % copies][idx][5],
                                                   gs, m, n, k, -1), 5, e0, e1)
            tf = 2.0 * m * n * k / us * 1e-6
            res["prefill_nvfp4_bf16"].append({"gemm": nm, "m": m, "us": round(us, 1),
                                              "tflops": round(tf, 1), "frac_bf16_peak": round(tf / tf_peak, 3)})
    if with_competitors:
        time.sleep(1.0)
        res["competitors"] = competitors(pk, layers, copies, gs, dev, hbm_peak, tf_peak)
    return res


if __name__ == "__main__":
    main()
