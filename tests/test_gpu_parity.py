"""GPU parity tests (run on the B200 box): the CUDA path, called through the public
Python ops -> torch extension -> C ABI (libpetit_b200.so), against the oracle and the
committed golden vectors.  Bars: bit-exact for repack round trips and dequantised
weights; GEMM max rel err <= 1e-2 vs fp32 accumulation of the dequantised weights
(BASELINE.json north_star), plus the reference's own assert_close(2e-2, 2e-2)
(tests/ops/test_fp4_gemm_quark.py:54) and its C++ matcher on the reference's sizes."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import ROOT, bits16, from_bits16, golden, orc, pack_mxfp4, pack_nvfp4

pytestmark = pytest.mark.gpu

NVFP4_CASES = [(64, 128, 256, 1234), (96, 64, 512, 2026)]
MXFP4_CASES = [(64, 128, 256, 1234), (96, 96, 512, 2026)]
GEMM_TOL = 1e-2  # north_star: max |c - ref| / max |ref|


@pytest.fixture(scope="module")
def pk():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import petit_kernel  # fails loudly if the extension is missing

    assert torch.cuda.get_device_capability()[0] == 10, "sm_100 required"
    return petit_kernel


def gpu_ref_f32(pk, a, b, s, gs, n, k, mx):
    """fp32 accumulation of the (bit-exact-verified) dequantised weights, on the GPU."""
    w = pk.ops.dequant_dense(b, s, 1.0, torch.bfloat16, n, k, mx, True).float()
    return (a.float() @ w.t()) * gs.item()


# ------------------------------------------------------------------ reference cases
@pytest.mark.parametrize("m,n,k,seed", NVFP4_CASES)
def test_nvfp4_reference_cases(pk, m, n, k, seed):
    a, q, s, gs = orc.make_nvfp4_case(m, n, k, seed)
    b, sp = pack_nvfp4(pk, q, s, n, k)
    c = pk.mul_nvfp4_a16(a.cuda(), b, sp, gs.cuda(), m, n, k, -1)
    assert c.shape == (m, n) and c.dtype == torch.bfloat16 and c.is_cuda
    c_ref = orc.nvfp4_gemm_ref(a, q, s, gs)
    torch.testing.assert_close(c.cpu(), c_ref, rtol=2e-2, atol=2e-2)
    c_gold = from_bits16(golden("nvfp4_gemm_cases.npz")[f"m{m}_n{n}_k{k}_s{seed}_c"], torch.bfloat16)
    torch.testing.assert_close(c.cpu(), c_gold, rtol=2e-2, atol=2e-2)
    assert orc.is_near_cpp(c, c_ref).all()
    ref32 = (a.float() @ torch.from_numpy(
        orc.dequant_nvfp4(q.numpy(), s.view(torch.uint8).numpy())).t()) * gs.item()
    assert orc.max_rel_err(c, ref32) <= GEMM_TOL


@pytest.mark.parametrize("m,n,k,seed", MXFP4_CASES)
def test_mxfp4_reference_cases(pk, m, n, k, seed):
    a, q, s, gs = orc.make_mxfp4_case(m, n, k, seed)
    b, sp = pack_mxfp4(pk, q, s, n, k)
    assert tuple(b.shape) == (n // 16, 2 * k) and tuple(sp.shape) == (n // 32, k)
    c = pk.mul_mxfp4_a16(a.cuda(), b, sp, gs.cuda(), m, n, k, -1)
    c_ref = orc.mxfp4_gemm_ref(a, q, s, gs)
    # scales span 2^-126..2^110: compare relative to the output scale
    scale = c_ref.float().abs().max().item()
    torch.testing.assert_close(c.cpu().float() / scale, c_ref.float() / scale, rtol=2e-2, atol=2e-2)
    ref32 = (a.float() @ torch.from_numpy(orc.dequant_mxfp4(q.numpy(), s.numpy())).t()) * gs.item()
    assert orc.max_rel_err(c, ref32) <= GEMM_TOL
    c_gold = from_bits16(golden("mxfp4_cases.npz")[f"m{m}_n{n}_k{k}_s{seed}_c"], torch.bfloat16)
    assert orc.max_rel_err(c, c_gold.float()) <= GEMM_TOL
    # vectors built WITHOUT the oracle (torch e8m0 dtype x compressed-tensors e2m1 decoder,
    # tests/golden/make_golden_mx.py): dequantised weights bit-exact, GEMM within tolerance
    ind = golden("mxfp4_independent.npz")
    tag = f"m{m}_n{n}_k{k}_s{seed}"
    dense = pk.ops.dequant_dense(b, sp, 1.0, torch.bfloat16, n, k, True, True)
    assert np.array_equal(bits16(dense), ind[f"{tag}_w"])
    c_ind = from_bits16(ind[f"{tag}_c"], torch.bfloat16)
    assert orc.max_rel_err(c, c_ind.float()) <= GEMM_TOL
    torch.testing.assert_close(c.cpu().float() / scale, c_ind.float() / scale, rtol=2e-2, atol=2e-2)


# ------------------------------------------------------------------ exhaustive dequant
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_nvfp4_dequant_exhaustive_bit_exact(pk, dtype):
    """All 16 codes x all positive e4m3 0x01..0x7E (ExhaustiveFp4DequantTest,
    quantization_utils_fp4_test.cc:344-365,388-394); +-0 compare equal."""
    sb = golden("nvfp4_exhaustive.npz")["scale_bits"]
    n, k = 128, 2048  # rows cycle through the 16 codes, 128 groups cover the 126 scales
    q = torch.from_numpy(np.repeat(((np.arange(n) % 16).astype(np.uint8) * 0x11)[:, None], k // 2, axis=1).copy())
    sc = np.tile(np.resize(sb, k // 16), (n, 1))
    s = torch.from_numpy(sc.copy()).view(torch.float8_e4m3fn)
    expect = torch.from_numpy(orc.dequant_nvfp4(q.numpy(), sc)).to(dtype)
    b, sp = pack_nvfp4(pk, q, s, n, k)
    got_packed = pk.ops.dequant_dense(b, sp, 1.0, dtype, n, k, False, True)
    got_native = pk.ops.dequant_dense(q.cuda().view(torch.int32), s.cuda(), 1.0, dtype, n, k, False, False)
    assert orc.bits_equal_pm0(got_packed, expect)
    assert orc.bits_equal_pm0(got_native, expect)
    # golden table produced by the reference's own _dequant_nvfp4
    table = torch.from_numpy(golden("nvfp4_exhaustive.npz")["table"].copy()).to(dtype)
    assert orc.bits_equal_pm0(got_packed[:16, :126 * 16:16].cpu(), table)


def test_mxfp4_dequant_exhaustive_bit_exact(pk):
    """All 16 codes x e8m0 1..237 with the row/col mixing pattern of MxFp4DequantTest
    (quantization_utils_fp4_test.cc:273-278,311-342)."""
    n, k = 256, 256 * 32 // 32 * 8  # 64 groups per row
    k = 2048
    rows = np.arange(n)[:, None]
    cols = np.arange(k // 32)[None, :]
    sc = (1 + (cols + 29 * rows) % 237).astype(np.uint8)
    q = torch.from_numpy(np.repeat(((np.arange(n) % 16).astype(np.uint8) * 0x11)[:, None], k // 2, axis=1).copy())
    s = torch.from_numpy(sc.copy())
    expect = torch.from_numpy(orc.dequant_mxfp4(q.numpy(), sc)).to(torch.bfloat16)
    b, sp = pack_mxfp4(pk, q, s, n, k)
    got_packed = pk.ops.dequant_dense(b, sp, 1.0, torch.bfloat16, n, k, True, True)
    got_native = pk.ops.dequant_dense(q.cuda().view(torch.int32), s.cuda(), 1.0, torch.bfloat16, n, k, True, False)
    assert orc.bits_equal_pm0(got_packed, expect)
    assert orc.bits_equal_pm0(got_native, got_packed)
    with pytest.raises(RuntimeError):  # MXFP4 is bf16 only (gemm_fp4.h:19-21 -> -1)
        pk.ops.dequant_dense(b, sp, 1.0, torch.float16, n, k, True, True)
    # the same two tables from implementations the oracle did not write
    # (tests/golden/make_golden_mx.py): 16 codes x e8m0 1..237, and the mixing pattern slab
    ind = golden("mxfp4_independent.npz")
    sb = np.arange(1, 238, dtype=np.uint8)
    n2, k2 = 128, 256 * 32          # 256 groups per row >= 237 scales
    q2 = torch.from_numpy(np.repeat(((np.arange(n2) % 16).astype(np.uint8) * 0x11)[:, None], k2 // 2, axis=1).copy())
    s2 = torch.from_numpy(np.tile(np.resize(sb, k2 // 32), (n2, 1)).copy())
    b2, sp2 = pack_mxfp4(pk, q2, s2, n2, k2)
    got = pk.ops.dequant_dense(b2, sp2, 1.0, torch.bfloat16, n2, k2, True, True)
    assert np.array_equal(bits16(got[:16, :237 * 32:32]), ind["exhaustive_bf16_bits"])
    qm, sm = torch.from_numpy(ind["mix_q"].copy()), torch.from_numpy(ind["mix_s"].copy())
    bm, spm = pack_mxfp4(pk, qm, sm, 64, 512)
    gm = pk.ops.dequant_dense(bm, spm, 1.0, torch.bfloat16, 64, 512, True, True)
    assert np.array_equal(bits16(gm), ind["mix_w_bits"])


def test_scale_edge_cases_documented(pk):
    """Outside the reference's tested domain: e4m3 0x00 -> weights 0; e8m0 0 -> 2^-127
    (OCP; the reference's bf16 shift gives 0), checked through the GEMM-exact hook."""
    n, k = 32, 256
    q = torch.full((n, k // 2), 0x77, dtype=torch.uint8)  # all +6
    s = torch.zeros((n, k // 16), dtype=torch.uint8).view(torch.float8_e4m3fn)
    b, sp = pack_nvfp4(pk, q, s, n, k)
    for dt in (torch.bfloat16, torch.float16):
        assert pk.ops.dequant_dense(b, sp, 1.0, dt, n, k, False, True).abs().max().item() == 0
    smx = torch.zeros((n, k // 32), dtype=torch.uint8)
    smx[:, 1] = 1
    b, sp = pack_mxfp4(pk, q, smx, n, k)
    w = pk.ops.dequant_dense(b, sp, 1.0, torch.bfloat16, n, k, True, True).float()
    assert torch.all(w[:, 32:64] == 6 * 2.0 ** -126)
    assert torch.all(w[:, 0:32] == 6 * 2.0 ** -127)


# ------------------------------------------------------------------ repack round trip
@pytest.mark.parametrize("n,k", [(512, 512), (96, 256), (1040, 768), (10240, 8192)])
def test_repack_round_trip_bit_exact(pk, n, k):
    """unpack(repack(q)) == q; dense(native) == dense(repacked) (NvFp4ToPetitFp4Test,
    quantization_utils_fp4_test.cc:103-133).  No -0 canonicalisation is applied."""
    _, q, s, _ = orc.make_gtest_style_case(1, n, k, "nvfp4")
    qw = q.cuda().contiguous().view(torch.int32)
    b = pk.repack_nvfp4(qw, n, k)
    assert tuple(b.shape) == (n // 16, 2 * k) and b.dtype == torch.int32
    assert torch.equal(pk.ops.unpack_fp4(b, n, k), qw)
    sp = pk.process_nvfp4_scales(s.cuda(), n, k)
    assert sp.shape == s.shape and sp.dtype == torch.float8_e4m3fn
    for dt in (torch.bfloat16, torch.float16):
        d_native = pk.ops.dequant_dense(qw, s.cuda(), 1.0, dt, n, k, False, False)
        d_packed = pk.ops.dequant_dense(b, sp, 1.0, dt, n, k, False, True)
        assert torch.equal(d_native.view(torch.int16), d_packed.view(torch.int16))
        if n * k <= 1 << 20:
            expect = torch.from_numpy(orc.dequant_nvfp4(q.numpy(), s.view(torch.uint8).numpy())).to(dt)
            assert orc.bits_equal_pm0(d_packed, expect)
    assert pk.ops.packed_layout_version() == 2


# ------------------------------------------------------------------ GEMM shapes
def run_gemm_case(pk, fmt, dtype, m, n, k, solution_id=-1, seed=42):
    a, q, s, gs = orc.make_gtest_style_case(m, n, k, fmt, dtype, seed)
    if fmt == "mxfp4":
        s = (s % 24 + 112).to(torch.uint8)  # keep outputs inside the 16-bit range
    gs = torch.tensor([1.0 / 64 if dtype == torch.float16 else 1.0])
    mx = fmt == "mxfp4"
    b, sp = (pack_mxfp4 if mx else pack_nvfp4)(pk, q, s, n, k)
    mul = pk.mul_mxfp4_a16 if mx else pk.mul_nvfp4_a16
    c = mul(a.cuda(), b, sp, gs.cuda(), m, n, k, solution_id)
    ref = gpu_ref_f32(pk, a.cuda(), b, sp, gs, n, k, mx)
    err = orc.max_rel_err(c, ref)
    assert err <= GEMM_TOL, f"{fmt} {dtype} m={m} n={n} k={k} sol={solution_id}: max rel err {err}"
    # per element, against the oracle's own dequantisation (sampled rows of large weights)
    rows = np.arange(n) if n * k <= 1 << 26 else np.unique(np.concatenate(
        [np.arange(128), np.arange(n - 128, n), np.random.RandomState(0).choice(n, 256, replace=False)]))
    sb = s.numpy() if mx else s.view(torch.uint8).numpy()
    w = (orc.dequant_mxfp4 if mx else orc.dequant_nvfp4)(q.numpy()[rows], sb[rows])
    assert orc.elementwise_ok(c[:, torch.from_numpy(rows).cuda()], a.cuda(), w, gs.item(), dtype), \
        f"{fmt} {dtype} m={m} n={n} k={k} sol={solution_id}: elementwise"
    return c


@pytest.mark.parametrize("m", [1, 2, 3, 4, 7, 8, 15, 16, 17, 44, 63, 64, 96, 566, 1003])
def test_gemm_m_sweep(pk, m):
    # odd M values from the reference's real-traffic list (tools/benchmarks/matmul.py:9-90)
    run_gemm_case(pk, "nvfp4", torch.bfloat16, m, 1280, 1024)


@pytest.mark.parametrize("n,k", [(64, 256), (1280, 3584), (10240, 1024), (2048, 8192)])
@pytest.mark.parametrize("fmt,dtype", [("nvfp4", torch.bfloat16), ("nvfp4", torch.float16), ("mxfp4", torch.bfloat16)])
def test_gemm_shape_sweep(pk, fmt, dtype, n, k):
    if fmt == "mxfp4" and n % 32:
        pytest.skip("MXFP4 scales need N % 32")
    run_gemm_case(pk, fmt, dtype, 16, n, k)
    run_gemm_case(pk, fmt, dtype, 130, n, k)


@pytest.mark.parametrize("k", [512, 768, 1024])  # pipeline-depth cases, rocm_test.cc:383-401
@pytest.mark.parametrize("fmt,dtype", [("nvfp4", torch.bfloat16), ("nvfp4", torch.float16), ("mxfp4", torch.bfloat16)])
def test_every_solution_id(pk, fmt, dtype, k):
    m, n = 96, 320
    b_type = pk.ops.kDataTypeMxFp4e2m1 if fmt == "mxfp4" else pk.ops.kDataTypeFp4e2m1
    sols = pk.ops.get_fp4_solutions(m, n, k, dtype, dtype, b_type=int(b_type))
    assert len(sols) == 5
    outs = [run_gemm_case(pk, fmt, dtype, m, n, k, sid) for sid in sols]
    for o in outs[1:]:
        assert orc.max_rel_err(o, outs[0].float()) <= GEMM_TOL


def test_gemm_matches_cpp_matcher_on_reference_sizes(pk):
    # TEST_BF16 sizes: M = tile_m*16, N = lcm(tile_n*16, 32), K = lcm(tile_k*16, 256)
    for (m, n, k) in [(16, 32, 256), (64, 64, 256), (128, 128, 256), (256, 256, 256), (32, 32, 512)]:
        a, q, s, gs = orc.make_gtest_style_case(m, n, k, "nvfp4", torch.bfloat16)
        b, sp = pack_nvfp4(pk, q, s, n, k)
        c = pk.mul_nvfp4_a16(a.cuda(), b, sp, gs.cuda(), m, n, k, -1)
        w = torch.from_numpy(orc.dequant_nvfp4(q.numpy(), s.view(torch.uint8).numpy()))
        ref = (a.float() @ w.t()).to(torch.bfloat16)  # fp32-compute reference, rocm_test.cc:120-164
        assert orc.is_near_cpp(c, ref).all()


# ------------------------------------------------------------------ API behaviour
def test_api_errors_and_checks(pk):
    m, n, k = 16, 128, 256
    a, q, s, gs = orc.make_nvfp4_case(m, n, k, 1)
    b, sp = pack_nvfp4(pk, q, s, n, k)
    ac, gsc = a.cuda(), gs.cuda()
    with pytest.raises(RuntimeError, match="No kernel implementation for solution_id=12345"):
        pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, 12345)
    with pytest.raises(RuntimeError, match="Only groupsize = 16"):
        pk.mul_nvfp4_a16(ac, b, sp[:, :8].contiguous(), gsc, m, n, k, -1)
    with pytest.raises(RuntimeError, match="bfloat16 or float16"):
        pk.mul_nvfp4_a16(ac.float(), b, sp, gsc, m, n, k, -1)
    with pytest.raises(RuntimeError, match="not contiguous"):
        pk.mul_nvfp4_a16(torch.zeros((m, 2 * k), dtype=torch.bfloat16, device="cuda")[:, ::2], b, sp, gsc, m, n, k, -1)
    with pytest.raises(RuntimeError, match="not contiguous"):
        pk.repack_nvfp4(torch.zeros((n, k // 4), dtype=torch.int32, device="cuda")[:, ::2], n, k)
    with pytest.raises(RuntimeError, match="kInt"):
        pk.repack_nvfp4(torch.zeros((n, k // 8), dtype=torch.float32, device="cuda"), n, k)
    # MXFP4 x fp16 has no kernel (gemm_fp4_fp16_grid.cc:60-63)
    _, qm, sm, _ = orc.make_mxfp4_case(m, n, k, 1)
    bm, spm = pack_mxfp4(pk, qm, sm, n, k)
    with pytest.raises(RuntimeError, match="No kernel implementation"):
        pk.mul_mxfp4_a16(ac.half(), bm, spm, gsc, m, n, k, -1)
    with pytest.raises(RuntimeError, match="is not size_n / 32"):
        pk.mul_mxfp4_a16(ac, bm, spm.view(n // 16, -1), gsc, m, n, k, -1)
    # keyword call, as SGLang/vLLM do
    c = pk.mul_nvfp4_a16(a=ac, b=b, s=sp, global_scale=gsc, size_m=m, size_n=n, size_k=k, solution_id=-1)
    assert c.shape == (m, n)
    # an explicit id of the wrong activation type is rejected
    sol_bf16 = pk.get_fp4_solutions(m, n, k, torch.bfloat16, torch.bfloat16)[0]
    with pytest.raises(RuntimeError, match="No kernel implementation"):
        pk.mul_nvfp4_a16(ac.half(), b, sp, gsc, m, n, k, sol_bf16)


def test_deterministic_and_stream_ordered(pk):
    m, n, k = 16, 2048, 4096   # stream-K splits every tile here
    a, q, s, gs = orc.make_nvfp4_case(m, n, k, 3)
    b, sp = pack_nvfp4(pk, q, s, n, k)
    ac, gsc = a.cuda(), gs.cuda()
    c0 = pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1)
    for _ in range(5):
        assert torch.equal(pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1), c0)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        c1 = pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1)
    st.synchronize()
    assert torch.equal(c1, c0)


def test_cuda_graph_capture_reads_global_scale_on_device(pk):
    """global_scale is dereferenced inside the kernel (gemm_fp4_fp16_grid.cuh:469-470):
    no host sync, so the op is graph-capturable and sees later updates of the scale."""
    m, n, k = 8, 1024, 2048
    a, q, s, gs = orc.make_nvfp4_case(m, n, k, 5)
    b, sp = pack_nvfp4(pk, q, s, n, k)
    ac, gsc = a.cuda(), torch.ones(1, device="cuda")
    pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1)  # warm-up allocates the stream-K workspace
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c = pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1)
    g.replay()
    torch.cuda.synchronize()
    c1 = c.clone()
    gsc.fill_(2.0)
    g.replay()
    torch.cuda.synchronize()
    torch.testing.assert_close(c.float(), 2 * c1.float(), rtol=1e-2, atol=1e-2)


def test_two_graphs_captured_on_a_fresh_stream_replay_in_any_order(pk):
    """The stream-K workspace of a stream is created lazily; when the first GEMM on a stream
    runs inside graph capture its counters must still be zeroed eagerly, not as a node of that
    one graph (ADVICE r1): capture two graphs on a fresh stream, replay the SECOND first."""
    m, n, k = 16, 2048, 4096   # stream-K splits every tile here
    a, q, s, gs = orc.make_nvfp4_case(m, n, k, 11)
    b, sp = pack_nvfp4(pk, q, s, n, k)
    ac, gsc = a.cuda(), gs.cuda()
    want = pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    outs, graphs = [], []
    for _ in range(2):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            outs.append(pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1))
        graphs.append(g)
    for o in outs:
        o.zero_()
    torch.cuda.synchronize()
    graphs[1].replay()
    torch.cuda.synchronize()
    assert torch.equal(outs[1], want)
    graphs[0].replay()
    graphs[1].replay()
    torch.cuda.synchronize()
    assert torch.equal(outs[0], want) and torch.equal(outs[1], want)


def test_concurrent_streams_split_tile_gemms(pk):
    """Stream-K GEMMs (every tile split between CTAs) issued concurrently from three streams,
    one of them high priority, 300 rounds: bit-identical results, no watchdog report.
    (petit.h documents why equal-priority streams always make progress and what the
    watchdog does otherwise.)"""
    m, n, k = 16, 2048, 4096
    cases = []
    for seed in (21, 22, 23):
        a, q, s, gs = orc.make_nvfp4_case(m, n, k, seed)
        b, sp = pack_nvfp4(pk, q, s, n, k)
        cases.append((a.cuda(), b, sp, gs.cuda()))
    want = [pk.mul_nvfp4_a16(a, b, sp, gs, m, n, k, -1) for a, b, sp, gs in cases]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream(priority=-1)]
    outs = [torch.empty_like(w) for w in want]
    bad = torch.zeros(3, dtype=torch.int32, device="cuda")
    for it in range(300):
        for i, st in enumerate(streams):
            with torch.cuda.stream(st):
                a, b, sp, gs = cases[i]
                pk.ops.mul_nvfp4_a16_out(outs[i], a, b, sp, gs, m, n, k, -1)
                bad[i] += (outs[i] != want[i]).any().to(torch.int32)
    torch.cuda.synchronize()
    assert bad.tolist() == [0, 0, 0]
    for st in streams:
        with torch.cuda.stream(st):
            assert pk.ops.workspace_status() == 0
            pk.ops.release_workspace()
    assert pk.ops.workspace_status() == 0


def test_gemm_directly_after_repack_on_the_same_stream(pk):
    """The weight producer warp does not wait for the grid dependency (weights are constants);
    a GEMM that directly follows repack_* on the stream must still see the repacked weights
    (the library launches it without programmatic dependent launch)."""
    m, n, k = 16, 4096, 4096
    a, q, s, gs = orc.make_nvfp4_case(m, n, k, 31)
    ac, gsc = a.cuda(), gs.cuda()
    qw = q.cuda().contiguous().view(torch.int32)
    sc = s.cuda()
    b0, sp0 = pack_nvfp4(pk, q, s, n, k)
    want = pk.mul_nvfp4_a16(ac, b0, sp0, gsc, m, n, k, -1)
    torch.cuda.synchronize()
    for _ in range(20):
        sp = pk.process_nvfp4_scales(sc, n, k)
        b = pk.repack_nvfp4(qw, n, k)
        c = pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1)
        assert torch.equal(c, want)
        del b, sp


# ------------------------------------------------------------------ full-size properties
@pytest.mark.parametrize("name,n,k", [("qkv", 10240, 8192), ("o", 8192, 8192), ("down", 8192, 28672)])
@pytest.mark.parametrize("fmt", ["nvfp4", "mxfp4"])
def test_llama70b_shapes_decode(pk, fmt, name, n, k):
    for m in (1, 16):
        run_gemm_case(pk, fmt, torch.bfloat16, m, n, k)


def test_gate_up_full_size_properties(pk):
    """BASELINE config 2 largest shape: sampled-row oracle check + linearity."""
    m, n, k = 16, 57344, 8192
    a, q, s, gs = orc.make_gtest_style_case(m, n, k, "nvfp4", torch.bfloat16)
    b, sp = pack_nvfp4(pk, q, s, n, k)
    ac, gsc = a.cuda(), gs.cuda()
    c = pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1)
    rows = np.random.RandomState(0).choice(n, 256, replace=False)
    w = torch.from_numpy(orc.dequant_nvfp4(q.numpy()[rows], s.view(torch.uint8).numpy()[rows]))
    ref = a.float() @ w.t()
    assert orc.max_rel_err(c[:, torch.from_numpy(rows).cuda()], ref) <= GEMM_TOL
    # the packed dequant hook -- what gpu_ref_f32 builds the large-shape references from -- against
    # the CPU oracle at full size: sampled rows (every tile position incl. the last tile) bit-exact
    dense = pk.ops.dequant_dense(b, sp, 1.0, torch.bfloat16, n, k, False, True)
    rows2 = np.concatenate([rows, np.arange(128), np.arange(n - 128, n)])
    w2 = torch.from_numpy(orc.dequant_nvfp4(q.numpy()[rows2], s.view(torch.uint8).numpy()[rows2]))
    assert orc.bits_equal_pm0(dense[torch.from_numpy(rows2).cuda()].cpu(), w2.to(torch.bfloat16))
    del dense
    # linearity: C(a) + C(a2) == C(a + a2) up to bf16 rounding of three outputs
    a2 = torch.roll(ac, 1, dims=1) * 0.5
    lhs = pk.mul_nvfp4_a16((ac + a2).to(torch.bfloat16), b, sp, gsc, m, n, k, -1).float()
    rhs = c.float() + pk.mul_nvfp4_a16(a2, b, sp, gsc, m, n, k, -1).float()
    assert (lhs - rhs).abs().max().item() <= 3e-2 * rhs.abs().max().item()


def test_prefill_shape(pk):
    run_gemm_case(pk, "nvfp4", torch.bfloat16, 2048, 8192, 8192)
    run_gemm_case(pk, "mxfp4", torch.bfloat16, 1024, 10240, 8192)


# ------------------------------------------------------------------ tensor parallel (1 GPU)
@pytest.mark.parametrize("tp", [2, 8])
def test_tp_shards_match_single_gpu(pk, tp):
    import petit_tp

    m = 16
    for name, (n, k, kind) in petit_tp.LLAMA70B_LAYER.items():
        if name == "gate_up":
            n = 57344 // 8  # keep the CPU generator quick; same code path
        a, q, s, gs = orc.make_gtest_style_case(m, n, k, "nvfp4", torch.bfloat16, seed=1)
        sb = s.view(torch.uint8)
        b, sp = pack_nvfp4(pk, q, s, n, k)
        ac, gsc = a.cuda(), gs.cuda()
        full = pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1).float()
        if kind == "column":
            parts = []
            for r in range(tp):
                qs, ss = petit_tp.column_shard(q, sb, tp, r)
                lin = petit_tp.PackedLinear.from_native(qs, ss.view(torch.float8_e4m3fn), gs, "nvfp4", kind)
                parts.append(lin.forward(ac).float())
            got = torch.cat(parts, dim=1)
        else:
            got = torch.zeros_like(full)
            for r in range(tp):
                qs, ss = petit_tp.row_shard(q, sb, tp, r)
                lin = petit_tp.PackedLinear.from_native(qs, ss.view(torch.float8_e4m3fn), gs, "nvfp4", kind)
                got += lin.forward(petit_tp.row_shard_activation(ac, tp, r), reduce=False).float()
        assert orc.max_rel_err(got, full) <= GEMM_TOL, name


def test_out_variant_writes_in_place(pk):
    m, n, k = 16, 512, 1024
    a, q, s, gs = orc.make_nvfp4_case(m, n, k, 9)
    b, sp = pack_nvfp4(pk, q, s, n, k)
    ac, gsc = a.cuda(), gs.cuda()
    ref = pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1)
    out = torch.empty((m, n), dtype=torch.bfloat16, device="cuda")
    ret = pk.ops.mul_nvfp4_a16_out(out, ac, b, sp, gsc, m, n, k, -1)
    assert ret.data_ptr() == out.data_ptr() and torch.equal(out, ref)
    with pytest.raises(RuntimeError, match="out must be"):
        pk.ops.mul_nvfp4_a16_out(out[:, :256], ac, b, sp, gsc, m, n, k, -1)


def test_unaligned_operands_are_rejected(pk):
    """TMA needs 16-byte aligned bases: a view starting at an odd element must fail
    loudly (PETIT_ERROR_PROBLEM_SHAPE), never compute on the wrong bytes."""
    m, n, k = 16, 512, 1024
    a, q, s, gs = orc.make_nvfp4_case(m, n, k, 10)
    b, sp = pack_nvfp4(pk, q, s, n, k)
    gsc = gs.cuda()
    flat = torch.zeros(m * k + 8, dtype=torch.bfloat16, device="cuda")
    a_off = flat[1 : 1 + m * k].view(m, k)
    a_off.copy_(a.cuda())
    assert a_off.data_ptr() % 16 != 0
    with pytest.raises(RuntimeError):
        pk.mul_nvfp4_a16(a_off, b, sp, gsc, m, n, k, -1)
    # the same values from an aligned buffer are fine
    ref = pk.mul_nvfp4_a16(a_off.clone(), b, sp, gsc, m, n, k, -1)
    assert torch.isfinite(ref.float()).all()


@pytest.mark.parametrize("m,n,k", [(1024, 2048, 2048), (700, 4096, 1024), (2048, 1024, 4096)])
def test_prefill_tiles_and_cluster_variant(pk, m, n, k):
    """128/256-token tiles (with and without the 2-CTA multicast cluster variant, chosen by
    the default rule or forced through explicit solution ids) against the oracle GEMM."""
    a, q, s, gs = orc.make_nvfp4_case(m, n, k, 11)
    b, sp = pack_nvfp4(pk, q, s, n, k)
    ac, gsc = a.cuda(), gs.cuda()
    want = orc.nvfp4_gemm_ref_torch(a, q, s, gs)
    sols = [sid for sid in pk.get_fp4_solutions(m, n, k, torch.bfloat16, torch.bfloat16)
            if "128" in pk.ops.solution_name(int(sid)) or "256" in pk.ops.solution_name(int(sid))]
    assert len(sols) >= 2
    outs = [pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1)]
    for sid in sols:
        outs.append(pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, int(sid)))
    w = orc.dequant_nvfp4(q.numpy(), s.view(torch.uint8).numpy())
    for o in outs:
        assert orc.max_rel_err(o.float().cpu(), want) <= GEMM_TOL
        assert orc.elementwise_ok(o, ac, w, gs.item(), torch.bfloat16)
    # every tile shape computes the same sums up to fp32 accumulation order
    for o in outs[1:]:
        assert orc.max_rel_err(o.float().cpu(), outs[0].float().cpu()) <= GEMM_TOL


def test_native_selftest_binary(pk):
    exe = os.path.join(ROOT, "tests", "native", "selftest")
    if not os.path.exists(exe):
        pytest.skip("native selftest not built")
    r = subprocess.run([exe, "quick"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:]


@pytest.mark.parametrize("fmt,dtype", [("nvfp4", torch.bfloat16), ("nvfp4", torch.float16),
                                       ("mxfp4", torch.bfloat16)])
@pytest.mark.parametrize("m,n,k", [(16, 2048, 4096), (5, 1040, 768), (300, 512, 1024)])
def test_fused_bias_and_residual_epilogue(pk, fmt, dtype, m, n, k):
    """petit_gemm_*_ex: C = round(acc * gs + bias[n] + residual[m, n]) with the additions in
    fp32 before the one rounding -- split (stream-K) tiles, a partial n-tile, every token-tile
    width; checked against the oracle's fp32 reference plus the same terms, and against the
    unfused op + torch adds (which round twice, hence only close)."""
    if fmt == "nvfp4":
        a, q, s, gs = orc.make_nvfp4_case(m, n, k, 7, dtype=dtype)
        b, sp = pack_nvfp4(pk, q, s, n, k)
        w = orc.dequant_nvfp4(q.numpy(), s.view(torch.uint8).numpy())
    else:
        n = (n + 31) // 32 * 32  # MXFP4 scales come in [N/32, K] (fp4.cc:146-148)
        a, q, s, gs = orc.make_mxfp4_case(m, n, k, 7)
        b, sp = pack_mxfp4(pk, q, s, n, k)
        w = orc.dequant_mxfp4(q.numpy(), s.numpy())
    g = torch.Generator().manual_seed(3)
    ref32 = (a.float() @ torch.from_numpy(w).t()) * gs.item()
    scale = ref32.abs().max().item()
    bias = (torch.randn(n, generator=g) * scale * 0.1).to(dtype)
    resid = (torch.randn(m, n, generator=g) * scale * 0.1).to(dtype)
    ac, gsc = a.cuda(), gs.cuda()
    mx = fmt == "mxfp4"
    for bb, rr in ((bias, None), (None, resid), (bias, resid)):
        want = ref32.clone()
        if bb is not None:
            want += bb.float()
        if rr is not None:
            want += rr.float()
        got = pk.ops.mul_fp4_a16_ex_out(None, ac, b, sp, gsc, m, n, k, -1, mx,
                                        None if bb is None else bb.cuda(),
                                        None if rr is None else rr.cuda())
        assert got.dtype == dtype and orc.max_rel_err(got, want) <= GEMM_TOL
        assert orc.elementwise_ok(got, ac, w, gs.item(), dtype, bb, rr)
    # residual may alias the output (in-place residual stream update)
    out = resid.cuda().clone()
    pk.ops.mul_fp4_a16_ex_out(out, ac, b, sp, gsc, m, n, k, -1, mx, bias.cuda(), out)
    assert orc.max_rel_err(out, ref32 + bias.float() + resid.float()) <= GEMM_TOL
    assert orc.elementwise_ok(out, ac, w, gs.item(), dtype, bias, resid)
    # the glue uses it instead of output.add_(bias)
    from petit_kernel import petit_utils as pu

    apply = pu.apply_petit_mxfp4_linear if mx else pu.apply_petit_nvfp4_linear
    y = apply(ac.view(1, m, k), b, sp, gsc, n, k, bias.cuda(), resid.cuda().view(1, m, n))
    assert tuple(y.shape) == (1, m, n)
    assert orc.max_rel_err(y.view(m, n), ref32 + bias.float() + resid.float()) <= GEMM_TOL
    with pytest.raises(RuntimeError):
        pk.ops.mul_fp4_a16_ex_out(None, ac, b, sp, gsc, m, n, k, -1, mx, bias.cuda()[:-1].contiguous(), None)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("m,inter,k", [(16, 1024, 2048), (3, 128, 512), (200, 512, 1024)])
def test_fused_silu_mul_epilogue(pk, dtype, m, inter, k):
    """PETIT_ACT_SILU_MUL: the gate_up projection returns silu(gate) * up.  Reference = what the
    frameworks run unfused on the same kernel's output: GEMM (rounded), silu in fp32 (rounded),
    product (rounded).  Same arithmetic, so equal up to the last bit of expf."""
    from petit_kernel import petit_utils as pu

    n = 2 * inter
    a, q, s, gs = orc.make_nvfp4_case(m, n, k, 17, dtype=dtype)
    ac, gsc = a.cuda(), (gs * 0.02).cuda()  # keep silu's argument in its interesting range
    b, sp = pack_nvfp4(pk, q, s, n, k)
    c = pk.mul_nvfp4_a16(ac, b, sp, gsc, m, n, k, -1)          # unfused: [m, 2 I] = gate | up
    want = (torch.nn.functional.silu(c[:, :inter].float()).to(dtype).float() * c[:, inter:].float()).to(dtype)
    lay = _FakeLinear(q, s, n, k)
    pu.prepare_nvfp4_layer_for_petit(lay, fuse_silu_mul=True)
    got = pu.apply_petit_nvfp4_linear(ac, lay.weight, lay.weight_scale, gsc, n, k, None, None, True)
    assert tuple(got.shape) == (m, inter) and got.dtype == dtype
    diff = (got.float() - want.float()).abs()
    tol = want.float().abs() * 2 ** -6 + 1e-6   # one 16-bit ulp: expf vs torch's exp
    assert bool((diff <= tol).all()), diff.max().item()
    assert (got == want).float().mean().item() > 0.98
    # with a bias (indexed in the interleaved row order)
    g = torch.Generator().manual_seed(5)
    bias = (torch.randn(n, generator=g) * 0.5).to(dtype)
    cb = (c.float() + bias.cuda().float()).to(dtype)  # unfused rounds the GEMM first: close, not equal
    want_b = (torch.nn.functional.silu(cb[:, :inter].float()) * cb[:, inter:].float())
    got_b = pu.apply_petit_nvfp4_linear(ac, lay.weight, lay.weight_scale, gsc, n, k,
                                        pu.interleave_gate_up(bias).cuda(), None, True)
    assert orc.max_rel_err(got_b.cpu(), want_b.cpu()) <= 2e-2
    with pytest.raises(RuntimeError):  # residual has the GEMM's shape, the output does not
        pk.ops.mul_fp4_a16_ex_out(None, ac, lay.weight, lay.weight_scale, gsc, m, n, k, -1, False,
                                  None, c, True)


@pytest.mark.parametrize("fmt", ["nvfp4", "mxfp4"])
def test_grouped_moe_gemm(pk, fmt):
    """petit_gemm_fp4_a16_grouped: token-grouped expert GEMMs (tokens sorted by expert, ragged
    and empty groups) against the oracle per expert.  The single-launch grouped kernel (one
    stream-K schedule over the token tiles of all experts) must agree with the same GEMMs issued
    one by one (PETIT_GROUPED_SINGLE=0; the two cut the k range at different places, so they
    agree to an output ulp, not bit for bit), on whole and on split tiles, for every decode tile
    width, and must not touch the rows of a neighbouring expert."""
    make = orc.make_nvfp4_case if fmt == "nvfp4" else orc.make_mxfp4_case
    pack = pack_nvfp4 if fmt == "nvfp4" else pack_mxfp4
    for (n, k, counts) in ((512, 1024, [5, 0, 33, 1, 16, 70]),        # 64-token tiles, 2 for the last
                           (2048, 4096, [3, 1, 0, 7, 2, 16, 4, 1]),   # 16-token tiles, split by stream-K
                           (1040 // 16 * 16, 768, [17, 32, 0, 0, 9]),  # 32-token tiles, partial n-tile
                           (256, 256, [1] * 100)):                    # > 96 tiles: issued one by one
        e = len(counts)
        offsets = [0]
        for c in counts:
            offsets.append(offsets[-1] + c)
        total = offsets[-1]
        if fmt == "mxfp4":
            n = (n + 31) // 32 * 32
        a_all, bs, ss, gss, refs, ws = [], [], [], [], [], []
        for g in range(e):
            a, q, s, gs = make(max(counts[g], 1), n, k, 100 + g)
            a = a[:counts[g]]
            if g < 8 or not bs:
                b, sp = pack(pk, q, s, n, k)
                w = (orc.dequant_nvfp4(q.numpy(), s.view(torch.uint8).numpy()) if fmt == "nvfp4"
                     else orc.dequant_mxfp4(q.numpy(), s.numpy()))
                wt = torch.from_numpy(w).t()
            else:  # many experts: reuse the 8th expert's weights, own activations and scale
                b, sp = bs[7], ss[7]
            refs.append((a.float() @ wt) * gs.item())
            ws.append(w)
            a_all.append(a); bs.append(b); ss.append(sp); gss.append(gs)
        a_cat = torch.cat(a_all).cuda().contiguous()
        outs = []
        for single in ("1", "0"):
            os.environ["PETIT_GROUPED_SINGLE"] = single
            try:
                out = torch.full((total, n), float("nan"), dtype=torch.bfloat16, device="cuda")
                pk.ops.mul_fp4_a16_grouped_out(out, a_cat, torch.stack(bs), torch.stack(ss),
                                               torch.cat(gss).cuda(), offsets, n, k, -1, fmt == "mxfp4")
                torch.cuda.synchronize()
            finally:
                os.environ.pop("PETIT_GROUPED_SINGLE", None)
            assert not torch.isnan(out.float()).any()
            outs.append(out)
        scale = outs[1].float().abs().max().item()
        assert (outs[0].float() - outs[1].float()).abs().max().item() <= scale * 2 ** -7, (n, k, counts)
        for g in range(e):
            if counts[g]:
                assert orc.max_rel_err(outs[0][offsets[g]:offsets[g + 1]].cpu(), refs[g]) <= GEMM_TOL
                for o in outs:
                    assert orc.elementwise_ok(o[offsets[g]:offsets[g + 1]], a_all[g].cuda(), ws[g],
                                              gss[g].item(), torch.bfloat16), (n, k, counts, g)
        assert pk.ops.workspace_status() == 0


def test_grouped_moe_silu_mul(pk):
    """Grouped GEMM with the fused SiLU * mul epilogue (an MoE MLP's w13 in one launch): against
    the unfused grouped output of the same packed weights, rows interleaved per 128-row tile
    (columns [128 t, 128 t + 64) gate, [128 t + 64, 128 t + 128) up).  Ragged groups: the stores
    behind a group's last token must not reach the next group's rows."""
    n, k, counts = 1024, 2048, [3, 0, 17, 1, 16, 5]
    offsets = [0]
    for c in counts:
        offsets.append(offsets[-1] + c)
    total, e = offsets[-1], len(counts)
    bs, ss, gss, a_all = [], [], [], []
    for g in range(e):
        a, q, s, gs = orc.make_nvfp4_case(max(counts[g], 1), n, k, 300 + g)
        b, sp = pack_nvfp4(pk, q, s, n, k)
        bs.append(b); ss.append(sp); gss.append(gs * 0.02); a_all.append(a[:counts[g]])
    a_cat = torch.cat(a_all).cuda().contiguous()
    b, sp, gsc = torch.stack(bs), torch.stack(ss), torch.cat(gss).cuda()
    plain = torch.empty((total, n), dtype=torch.bfloat16, device="cuda")
    pk.ops.mul_fp4_a16_grouped_out(plain, a_cat, b, sp, gsc, offsets, n, k, -1, False)
    t = plain.view(total, n // 128, 2, 64).float()
    want = (torch.nn.functional.silu(t[:, :, 0]).to(torch.bfloat16).float() * t[:, :, 1]).to(torch.bfloat16)
    want = want.reshape(total, n // 2)
    for single in ("1", "0"):
        os.environ["PETIT_GROUPED_SINGLE"] = single
        try:
            got = torch.full((total, n // 2), float("nan"), dtype=torch.bfloat16, device="cuda")
            pk.ops.mul_fp4_a16_grouped_out(got, a_cat, b, sp, gsc, offsets, n, k, -1, False, True)
            torch.cuda.synchronize()
        finally:
            os.environ.pop("PETIT_GROUPED_SINGLE", None)
        assert not torch.isnan(got.float()).any()
        # the unfused reference came from another k split: allow an output ulp on top of expf's
        diff = (got.float() - want.float()).abs()
        tol = want.float().abs() * 2 ** -5 + plain.float().abs().max().item() * 2 ** -7
        assert bool((diff <= tol).all()), (single, diff.max().item())
        if single == "1":
            assert (got == want).float().mean().item() > 0.95
    with pytest.raises(RuntimeError):
        pk.ops.mul_fp4_a16_grouped_out(torch.empty((total, n), dtype=torch.bfloat16, device="cuda"),
                                       a_cat, b, sp, gsc, offsets, n, k, -1, False, True)


def test_fp16_native_weight_layout(pk):
    """repack with a_dtype=float16 -> fp16-native packed layout (cvt.rn.f16x2.e2m1x2 path):
    round trip bit-exact, exhaustive dequant bit-exact (16 codes x all positive e4m3 scales),
    GEMM within tolerance on decode / split-tile / prefill shapes, bfloat16 activations rejected,
    and the glue picks it for float16 layers."""
    from petit_kernel import petit_utils as pu

    dtype = torch.float16
    # exhaustive table
    sb = golden("nvfp4_exhaustive.npz")["scale_bits"]
    n, k = 128, 2048
    q = torch.from_numpy(np.repeat(((np.arange(n) % 16).astype(np.uint8) * 0x11)[:, None], k // 2, axis=1).copy())
    sc = np.tile(np.resize(sb, k // 16), (n, 1))
    s = torch.from_numpy(sc.copy()).view(torch.float8_e4m3fn)
    qw = q.cuda().contiguous().view(torch.int32)
    b16 = pu.repack_nvfp4_for(qw, n, k, torch.float16)
    assert tuple(b16.shape) == (n // 32, 4 * k) and b16.dtype == torch.int32
    assert torch.equal(pk.ops.unpack_fp4(b16, n, k), qw)                      # round trip
    assert not torch.equal(b16.view(-1), pk.repack_nvfp4(qw, n, k).view(-1))  # really another layout
    sp = pk.process_nvfp4_scales(s.cuda(), n, k)
    expect = torch.from_numpy(orc.dequant_nvfp4(q.numpy(), sc)).to(dtype)
    got = pk.ops.dequant_dense(b16, sp, 1.0, dtype, n, k, False, True)
    assert orc.bits_equal_pm0(got, expect)
    table = torch.from_numpy(golden("nvfp4_exhaustive.npz")["table"].copy()).to(dtype)
    assert orc.bits_equal_pm0(got[:16, :126 * 16:16].cpu(), table)
    # GEMMs: every token-tile width, split tiles, a partial n-tile, prefill
    for (m, n, k) in ((16, 2048, 4096), (1, 512, 1024), (33, 1056, 768), (64, 1024, 2048),
                      (300, 1024, 1024), (1024, 2048, 2048)):
        a, q, s, gs = orc.make_nvfp4_case(m, n, k, 41, dtype=dtype)
        gs = gs * 0.05  # keep fp16 outputs finite
        qw = q.cuda().contiguous().view(torch.int32)
        b16 = pu.repack_nvfp4_for(qw, n, k, torch.float16)
        sp = pk.process_nvfp4_scales(s.cuda(), n, k)
        c = pk.mul_nvfp4_a16(a.cuda(), b16, sp, gs.cuda(), m, n, k, -1)
        w = orc.dequant_nvfp4(q.numpy(), s.view(torch.uint8).numpy())
        ref32 = (a.float() @ torch.from_numpy(w).t()) * gs.item()
        assert c.dtype == dtype and orc.max_rel_err(c, ref32) <= GEMM_TOL, (m, n, k)
        # same result class as the default layout on the same inputs
        c_def = pk.mul_nvfp4_a16(a.cuda(), pk.repack_nvfp4(qw, n, k), sp, gs.cuda(), m, n, k, -1)
        assert orc.max_rel_err(c, c_def.float().cpu()) <= GEMM_TOL
        with pytest.raises(RuntimeError, match="float16 activations"):
            pk.mul_nvfp4_a16(a.cuda().to(torch.bfloat16), b16, sp, gs.cuda(), m, n, k, -1)
    # the glue: a float16 layer is prepared in the fp16-native layout
    lay = _FakeLinear(q, s, n, k)
    lay.params_dtype = torch.float16
    pu.prepare_nvfp4_layer_for_petit(lay)
    assert tuple(lay.weight.shape) == (n // 32, 4 * k)
    y = pu.apply_petit_nvfp4_linear(a.cuda(), lay.weight, lay.weight_scale, gs.cuda(), n, k)
    assert orc.max_rel_err(y, ref32) <= GEMM_TOL


def test_cpp_source_compat_header_runs_a_gemm(pk, tmp_path):
    """The reference-style C++ unit (tests/native/compat_user.cc over gemm_compat.h) repacks and
    multiplies on the GPU through the namespace-compatible shim and the hal::Device object."""
    from test_capi_and_host import _build_compat_user

    exe = _build_compat_user(tmp_path)
    r = subprocess.run([exe, "gpu"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "compat gpu GEMM ok" in r.stdout, (r.returncode, r.stdout, r.stderr)


def test_bench_matmul_cli_tune(pk):
    """`bench_matmul -algo tune` lists every solution, prints the reference's result line
    for the fastest five, and a printed id can be fed back through -algo."""
    import re

    exe = os.path.join(ROOT, "tools", "bench_matmul")
    if not os.path.exists(exe):
        pytest.skip("bench_matmul not built")
    base = [exe, "-m", "16", "-n", "1024", "-k", "1024", "-atype", "bf16", "-ctype", "bf16",
            "-btype", "nvfp4", "-warmup", "2", "-repeat", "5"]
    r = subprocess.run(base + ["-algo", "tune"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert "Finished enumerating 5 algorithms" in r.stdout
    lines = re.findall(r"Matmul 16x1024x1024 bf16:bf16\. Backend: petit, batch: 1, algorithm: "
                       r"([0-9a-f]{16}), 5 times total [0-9.]+ ms\. [0-9.]+ TFLOPS", r.stdout)
    assert len(lines) == 5
    r2 = subprocess.run(base + ["-algo", lines[0]], capture_output=True, text=True, timeout=300)
    assert r2.returncode == 0 and f"algorithm: {lines[0]}" in r2.stdout


@pytest.mark.parametrize("end_barrier", [True, False])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape", [(16, 2048), (48, 5504)])
@pytest.mark.parametrize("world", range(2, 9))
def test_peer_allreduce_two_ranks_emulated_on_one_gpu(pk, end_barrier, dtype, shape, world):
    """csrc/allreduce.cu with `world` ranks emulated on one device: the ranks run as concurrent
    kernels on streams of their own and exchange flags through each other's pads.  The result
    must be oracle.rank_order_sum (fp32 sum in rank order, then one rounding), bit-identical on
    every rank, for several calls in a row with new data on every call (monotonic flag
    counters).  16 x 2048 needs 16 CTAs; 48 x 5504 more than 64 x 256 16-byte vectors, so the
    grid-stride loop of its 64 CTAs runs three times.  Order-sensitive columns: (+big, +small,
    -big) and (+big, -big, +small) on ranks 0..2 sum to 0 and to small in rank order only."""
    m, n = shape
    numel = m * n
    big, tiny = (2.0 ** 25, 1.0) if dtype == torch.bfloat16 else (32768.0, 2.0 ** -10)
    g = torch.Generator(device="cpu").manual_seed(5 + world)
    pad_words = pk.ops.allreduce_pad_bytes() // 4
    pads = [torch.zeros(pad_words, dtype=torch.int32, device="cuda") for _ in range(world)]
    epochs = [torch.zeros(pk.ops.allreduce_epoch_bytes() // 4, dtype=torch.int32, device="cuda")
              for _ in range(world)]
    bufs = [torch.empty((m, n), dtype=dtype, device="cuda") for _ in range(world)]
    outs = [torch.empty((m, n), dtype=dtype, device="cuda") for _ in range(world)]
    streams = [torch.cuda.Stream() for _ in range(world)]
    torch.cuda.synchronize()
    for it in range(4):
        vals = [(torch.randn((m, n), generator=g) * 100).to(dtype) for _ in range(world)]
        if world >= 3:
            for r in range(world):  # ranks 3.. add zeros there
                vals[r][:, 7 + it] = vals[r][:, n - 3 - it] = 0
            for r, (x, y) in enumerate(((big, big), (tiny, -big), (-big, tiny))):
                vals[r][:, 7 + it] = x
                vals[r][:, n - 3 - it] = y
        for r in range(world):
            bufs[r].copy_(vals[r])
        torch.cuda.synchronize()
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                pk.ops.allreduce_oneshot(outs[r], [b.data_ptr() for b in bufs],
                                         [p.data_ptr() for p in pads], epochs[r], r, numel,
                                         end_barrier)
        torch.cuda.synchronize()
        want = orc.rank_order_sum(vals, dtype)
        if world >= 3:
            assert bool((want[:, 7 + it].float() == 0).all()) and bool((want[:, n - 3 - it].float() == tiny).all())
        for r in range(world):
            assert torch.equal(outs[r].cpu().view(torch.int16), want.view(torch.int16)), (it, r)
    for r in range(world):
        assert int(pk.ops.allreduce_status(epochs[r])) == 0
        assert int(epochs[r][0]) == 4


TP_RUNS = [(world, two_shot) for world in (2, 4, 8) for two_shot in (None, "0", "1")]


@pytest.mark.parametrize("world,two_shot", TP_RUNS, ids=[f"{w}-{t or 'unset'}" for w, t in TP_RUNS])
def test_peer_allreduce_two_gpus(pk, world, two_shot):
    """torchrun over `world` GPUs with PETIT_AR_TWO_SHOT unset / 0 / 1: PeerAllReduce (own kernel
    over symmetric memory) equals ncclAllReduce on a row-parallel NVFP4 layer, and the fused
    GEMM + all-reduce is bit-exact on exact cases in all three formats."""
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    env = {k: v for k, v in os.environ.items() if k != "PETIT_AR_TWO_SHOT"}
    if two_shot is not None:
        env["PETIT_AR_TWO_SHOT"] = two_shot
    script = os.path.join(ROOT, "tests", "tp_peer_allreduce_check.py")
    port = 29541 + TP_RUNS.index((world, two_shot))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                        "--nproc-per-node", str(world), "--master-addr", "127.0.0.1", "--master-port",
                        str(port), script], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "PEER_ALLREDUCE_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


# ------------------------------------------------------------------ section 8f rows: glue + tuning
class _FakeLinear(torch.nn.Module):
    """What a framework's quantised linear layer looks like right after weight loading."""

    def __init__(self, q_u8, scales, n, k):
        super().__init__()
        self.output_size_per_partition, self.input_size_per_partition = n, k
        self.weight = torch.nn.Parameter(q_u8.cuda(), requires_grad=False)          # [N, K/2] u8
        self.weight_scale = torch.nn.Parameter(scales.cuda(), requires_grad=False)  # e4m3 / e8m0


@pytest.mark.parametrize("fmt", ["nvfp4", "mxfp4"])
def test_framework_glue_prepare_apply_and_versioned_state(pk, fmt):
    """petit_kernel.petit_utils: weight-load -> forward exactly as vLLM / SGLang drive the ops
    (3-D activations, in-place bias add), then export / reload of the packed tensors."""
    import petit_kernel.petit_utils as pu

    n, k, seed = 384, 1024, 7
    make = orc.make_nvfp4_case if fmt == "nvfp4" else orc.make_mxfp4_case
    a, q, s, gs = make(2 * 5, n, k, seed)
    layer = _FakeLinear(q, s, n, k)
    prepare = pu.prepare_nvfp4_layer_for_petit if fmt == "nvfp4" else pu.prepare_mxfp4_layer_for_petit
    apply = pu.apply_petit_nvfp4_linear if fmt == "nvfp4" else pu.apply_petit_mxfp4_linear
    prepare(layer)
    assert not layer.weight.requires_grad and layer.petit_layout_version == pk.ops.packed_layout_version()
    assert tuple(layer.weight.shape) == (n // 16, 2 * k) and layer.weight.dtype == torch.int32

    x = a.cuda().reshape(2, 5, k)
    bias = torch.linspace(-1, 1, n, dtype=torch.bfloat16, device="cuda")
    y = apply(x, layer.weight, layer.weight_scale, gs.cuda(), n, k, bias)
    assert y.shape == (2, 5, n) and y.dtype == torch.bfloat16
    w = orc.dequant_nvfp4(q.numpy(), s.view(torch.uint8).numpy()) if fmt == "nvfp4" \
        else orc.dequant_mxfp4(q.numpy(), s.numpy())
    ref = (a.float() @ torch.from_numpy(w).t()) * gs.item() + bias.float().cpu()
    assert orc.max_rel_err(y.reshape(-1, n), ref) <= GEMM_TOL
    y0 = apply(x, layer.weight, layer.weight_scale, gs.cuda(), n, k)  # no bias
    assert orc.max_rel_err(y0.reshape(-1, n), ref - bias.float().cpu()) <= GEMM_TOL

    state = pu.export_packed_state(layer)
    other = torch.nn.Module()
    pu.load_packed_state(other, {key: (v.clone() if torch.is_tensor(v) else v) for key, v in state.items()})
    y1 = apply(x, other.weight, other.weight_scale, gs.cuda(), n, k, bias)
    assert torch.equal(y1, y)
    with pytest.raises(ValueError, match="layout version"):
        pu.load_packed_state(torch.nn.Module(), dict(state, petit_layout_version=1))


def test_tune_gemm_feeds_the_default_chooser(pk, tmp_path):
    """petit_kernel.tuning.tune_gemm times every listed solution on the caller's tensors and
    makes the fastest the default; solution_id=-1 then runs exactly that kernel."""
    import petit_kernel.tuning as tuning

    tuning.clear_table()
    m, n, k = 48, 1024, 2048
    a, q, s, gs = orc.make_nvfp4_case(m, n, k, 11)
    b, sp = pack_nvfp4(pk, q, s, n, k)
    a, gs = a.cuda(), gs.cuda()
    res = tuning.tune_gemm(a, b, sp, gs, m, n, k, repeat=5)
    assert len(res) == 5 and all(us > 0 for us, _ in res) and res == sorted(res)
    best = res[0][1]
    assert tuning.default_solution(m, n, k, torch.bfloat16) == best
    c_auto = pk.mul_nvfp4_a16(a, b, sp, gs, m, n, k, -1)
    c_best = pk.mul_nvfp4_a16(a, b, sp, gs, m, n, k, best)
    assert torch.equal(c_auto, c_best)
    ref = gpu_ref_f32(pk, a, b, sp, gs, n, k, False)
    assert orc.max_rel_err(c_auto, ref.cpu()) <= GEMM_TOL
    # a forced large-tile entry is honoured too (any tile is valid for any m)
    tok256 = [sol for _, sol in res if (sol & 0xFF) * 16 == 256][0]
    tuning.set_solution(m, n, k, torch.bfloat16, False, tok256)
    assert pk.ops.solution_name(tuning.default_solution(m, n, k, torch.bfloat16)).endswith("tok256")
    c_256 = pk.mul_nvfp4_a16(a, b, sp, gs, m, n, k, -1)
    assert orc.max_rel_err(c_256, ref.cpu()) <= GEMM_TOL
    path = tmp_path / "table.txt"
    assert tuning.save_table(str(path)) == 1
    tuning.clear_table()
    assert tuning.default_solution(m, n, k, torch.bfloat16) != tok256


def test_bench_matmul_cli_writes_a_loadable_table(pk, tmp_path):
    import petit_kernel.tuning as tuning

    exe = os.path.join(ROOT, "tools", "bench_matmul")
    if not os.path.exists(exe):
        pytest.skip("bench_matmul not built")
    table = tmp_path / "tuned.txt"
    r = subprocess.run([exe, "-m", "16", "-n", "1024", "-k", "1024", "-atype", "bf16", "-ctype", "bf16",
                        "-btype", "mxfp4", "-warmup", "2", "-repeat", "5", "-algo", "tune",
                        "-table", str(table)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    fields = table.read_text().split()
    assert fields[:5] == ["mxfp4", "bf16", "16", "1024", "1024"] and len(fields[5]) == 16
    tuning.clear_table()
    assert tuning.load_table(str(table)) == 1
    sol = tuning.default_solution(16, 1024, 1024, torch.bfloat16, mx=True)
    assert tuning.solution_hex(sol) == fields[5]
    tuning.clear_table()
