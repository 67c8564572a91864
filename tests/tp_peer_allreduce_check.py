"""Run under torchrun (world >= 2, one GPU per rank): petit_tp.PeerAllReduce against
ncclAllReduce on a row-parallel NVFP4 layer, then a stress loop with data that changes every
call (a stale read of a peer buffer or a lost flag shows up as a mismatch against NCCL).
Launched by tests/test_gpu_parity.py and tools/exp_tp_check.sh.

  torchrun --nproc-per-node N tests/tp_peer_allreduce_check.py [iters] [out.json]
"""
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "petit-kernel_b200"))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import petit_kernel as pk  # noqa: E402
import petit_tp  # noqa: E402
from oracle import petit_oracle as orc  # noqa: E402  (checker only)


def gemm_case(rank, world):
    m, n, k = 16, 1024, 2048
    a, q, s, gs = orc.make_nvfp4_case(m, n, k, 77)
    # K-split (row parallel): every rank owns k / world columns
    qs, ss = petit_tp.row_shard(q, s, world, rank)
    a_s = petit_tp.row_shard_activation(a, world, rank).cuda()
    ks = k // world
    b = pk.repack_nvfp4(qs.cuda().contiguous().view(torch.int32), n, ks)
    sp = pk.process_nvfp4_scales(ss.cuda().contiguous(), n, ks)
    gsc = gs.cuda()
    par = petit_tp.PeerAllReduce()
    for it in range(5):
        ref = pk.mul_nvfp4_a16(a_s, b, sp, gsc, m, n, ks, -1)
        mine_in = par.buffer(m, n, torch.bfloat16, a_s.device, 0)
        pk.ops.mul_nvfp4_a16_out(mine_in, a_s, b, sp, gsc, m, n, ks, -1)
        got = par.reduce(mine_in)
        dist.all_reduce(ref)
        torch.cuda.synchronize()
        # same partials, both summed in fp32?  NCCL rounds per hop; allow one bf16 ulp of the max
        err = (got.float() - ref.float()).abs().max().item()
        scale = ref.float().abs().max().item()
        assert err <= scale * 2 ** -7, (it, err, scale)
        # identical on every rank
        gathered = [torch.empty_like(got) for _ in range(world)]
        dist.all_gather(gathered, got)
        assert all(torch.equal(gathered[0], x) for x in gathered)
    full = orc.nvfp4_gemm_ref_torch(a, q, s, gs)
    assert orc.max_rel_err(got.float().cpu(), full) <= 1e-2
    assert par.status() == 0


FUSED_FORMATS = (("nvfp4", torch.bfloat16), ("nvfp4", torch.float16), ("mxfp4", torch.bfloat16))


def fused_case(rank, world, calls):
    """petit_tp.FusedAllReduce (GEMM + all-reduce in one kernel) on exact cases
    (oracle.make_exact_case, K split over the ranks), NVFP4 x bf16 / fp16 and MXFP4 x bf16, on
    shapes where tiles are whole and where stream-K splits them: `calls` calls per shape with
    inputs that change on every call, each output bit for bit oracle.rank_order_sum of the
    ranks' exact partials (the epoch / buffer-parity protocol has to hold)."""
    from test_gemm_exact import assert_bits

    far = petit_tp.FusedAllReduce()
    dev = torch.device("cuda", torch.cuda.current_device())
    checked = []
    for fmt, dt in FUSED_FORMATS:
        # (m, n, k per rank)
        for m, n, ks in ((16, 1024, 2048), (1, 8192, 1024), (33, 2048, 512), (64, 8192, 256), (16, 2048, 3584)):
            k = ks * world
            a, q, s, gs, w, _ = orc.make_exact_case(fmt, dt, m * calls, n, k, 99 + m)
            qs, ss = petit_tp.row_shard(q, s, world, rank)
            a_s = petit_tp.row_shard_activation(a, world, rank).to(dev)  # every call's rows, staged
            qw = qs.to(dev).contiguous().view(torch.int32)
            if fmt == "nvfp4":
                b, sp = pk.repack_nvfp4(qw, n, ks), pk.process_nvfp4_scales(ss.to(dev).contiguous(), n, ks)
            else:
                b, sp = pk.repack_mxfp4(qw, n, ks), pk.process_mxfp4_scales(ss.to(dev).contiguous(), n, ks)
            gsc = gs.to(dev)
            torch.cuda.synchronize()
            outs = [far.matmul(a_s[i * m:(i + 1) * m], b, sp, gsc, n, ks, fmt) for i in range(calls)]
            torch.cuda.synchronize()
            a_dev = a.to(dev)
            parts = [orc.exact_ref(a_dev[:, r * ks:(r + 1) * ks], np.ascontiguousarray(w[:, r * ks:(r + 1) * ks]),
                                   gs.item(), dt) for r in range(world)]
            want = orc.rank_order_sum(parts, dt)
            for i in range(calls):
                assert_bits(outs[i], want[i * m:(i + 1) * m], f"rank {rank} {fmt} {dt} m={m} n={n} k={k} call {i}")
            checked.append([fmt, str(dt), m, n, k])
    assert far.status() == 0
    return checked


def stress(rank, world, iters, end_barrier, fenced, m=16, n=8192):
    """Integer-valued bf16 data that changes every call: the exact sum is representable, so
    the peer kernel must match the closed form bit for bit (any stale 16-byte vector from a
    previous call, a torn read or a missed flag is a mismatch).  A device-side check every
    call, one host sync per 256 calls."""
    dev = torch.device("cuda", torch.cuda.current_device())
    par = petit_tp.PeerAllReduce(end_barrier=end_barrier, fenced=fenced)
    idx = (torch.arange(m * n, device=dev, dtype=torch.int32) % 7).view(m, n)
    bad = torch.zeros((), dtype=torch.int32, device=dev)
    out = torch.empty((m, n), dtype=torch.bfloat16, device=dev)
    t0 = time.time()
    for it in range(iters):
        buf = par.buffer(m, n, torch.bfloat16, dev, 1)
        # rank r contributes (idx + it + r) % 13 - 6  (|.| <= 6, sums <= 48: exact in bf16)
        buf.copy_(((idx + (it + rank)) % 13 - 6).to(torch.bfloat16))
        par.reduce(buf, out=out)
        want = sum(((idx + (it + r)) % 13 - 6) for r in range(world)).to(torch.bfloat16)
        bad += (out != want).any().to(torch.int32)
        if it % 256 == 255:
            assert bad.item() == 0, f"rank {rank}: mismatch by iteration {it}"
    torch.cuda.synchronize()
    assert bad.item() == 0, f"rank {rank}: mismatch"
    assert par.status() == 0
    return time.time() - t0


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl")
    iters = int(sys.argv[1]) if len(sys.argv) > 1 else 300
    gemm_case(rank, world)
    res = {"world": world, "iters": iters, "modes": []}
    res["fused_gemm_allreduce"] = {"shapes": fused_case(rank, world, 6), "ok": True,
                                   "two_shot_env": os.environ.get("PETIT_AR_TWO_SHOT")}
    for end_barrier in (False, True):
        for fenced in (False, True):
            secs = stress(rank, world, iters, end_barrier, fenced)
            res["modes"].append({"end_barrier": end_barrier, "fenced": fenced, "ok": True,
                                 "seconds": round(secs, 2)})
    dist.barrier()
    if rank == 0:
        print("PEER_ALLREDUCE_OK", json.dumps(res))
        if len(sys.argv) > 2:
            with open(sys.argv[2], "w") as f:
                json.dump(res, f)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
