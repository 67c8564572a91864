"""Bit-exact GEMM tests on exactly representable data (oracle.make_exact_case): every fp32 sum
the kernel forms is exact in any order, so the output must equal RN16(RN32(S * gs)) bit for bit
(oracle.exact_ref) whatever the token tile, the stream-K cuts, the reducer path, the cluster
variant, programmatic dependent launch or graph replay.  A dropped or duplicated k-tile, a
partial from the wrong CTA, a scale from the neighbouring group, a swapped row or column or a
wrong rounding mode fails by at least one bit.  Shapes are chosen with oracle.stream_k_plan and
the test asserts which reducer paths they reach, so a shape edit cannot drop one silently.

Run as a script (``python tests/test_gemm_exact.py OUT_DIR``) it computes INVARIANCE_CASES and
writes their output bits to OUT_DIR; the invariance test does that in fresh processes with the
launcher's once-per-process environment switches set."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import LIB_PATH, ROOT, orc, pack_mxfp4, pack_nvfp4, stream_k_cuts_fn

# mode -> (weight format, activation / output dtype, fp16-native weight layout)
MODES = {
    "nv_bf16": ("nvfp4", torch.bfloat16, False),
    "nv_f16": ("nvfp4", torch.float16, False),
    "nv_f16n": ("nvfp4", torch.float16, True),
    "mx_bf16": ("mxfp4", torch.bfloat16, False),
}
# (m, n, k): what each shape is for, per stream_k_plan at 148 SMs (asserted in
# test_dense_exact_all_solutions for the device's SM count)
DENSE_SHAPES = [
    (16, 8192, 1024),   # TP-8 o_proj: whole-tile grid for 16/32/64-token tiles
    (48, 4096, 4096),   # >= 8 units per CTA: tilted cuts (16-token tiles)
    (16, 2048, 8192),   # 4 .. kRingFit contributors (ring), > kRingFit with m_valid <= 16
    (64, 128, 28672),   # > kRingFit contributors with m_valid > 16: the L2 tail
    (17, 1040, 4096),   # partial n-tile (n % 128 = 16) and partial token tile in split tiles
    (100, 240, 2048),   # partial n-tile (n % 128 = 112)
    (256, 1024, 2048),  # 2-CTA cluster variant (even n-tiles)
    (256, 1152, 2048),  # odd n-tiles: cluster fallback; unsplit tiles
    (5, 512, 4096),     # few tokens, many contributors
]
# every row must be reached by at least one launch of every mode
REQUIRED_PATHS = ("whole_tiles", "tilt", "unsplit", "reg_1_3", "ring", "many_m_le16", "many_m_gt16",
                  "l2_tail", "split_partial_n", "split_partial_m", "cluster", "cluster_fallback")
SEED = 11


def mode_shape(mode, m, n, k):
    """MXFP4 scales come in [N / 32, K]: partial n-tiles of 32 / 96 rows stand in for 16 / 112."""
    if MODES[mode][0] == "mxfp4" and n % 32:
        n = n + 16 if n % 128 == 16 else n - 16
    return m, n, k


@pytest.fixture(scope="module")
def pk():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import petit_kernel  # fails loudly if the extension is missing

    assert torch.cuda.get_device_capability()[0] == 10, "sm_100 required"
    return petit_kernel


@pytest.fixture(scope="module")
def cuts_fn():
    return stream_k_cuts_fn(ctypes.CDLL(LIB_PATH))


def num_sms():
    return min(torch.cuda.get_device_properties(0).multi_processor_count, orc.MAX_GRID)


def pack(pk, mode, q, s, n, k):
    fmt, _, native = MODES[mode]
    if fmt == "mxfp4":
        return pack_mxfp4(pk, q, s, n, k)
    if native:
        from petit_kernel import petit_utils as pu

        qw = q.cuda().contiguous().view(torch.int32)
        return pu.repack_nvfp4_for(qw, n, k, torch.float16), pk.process_nvfp4_scales(s.cuda(), n, k)
    return pack_nvfp4(pk, q, s, n, k)


def solutions(pk, mode, m, n, k):
    """Every listed solution id, then -1 (the default chooser)."""
    fmt, dt, _ = MODES[mode]
    b_type = pk.ops.kDataTypeMxFp4e2m1 if fmt == "mxfp4" else pk.ops.kDataTypeFp4e2m1
    sols = [int(x) for x in pk.ops.get_fp4_solutions(m, n, k, dt, dt, b_type=int(b_type))]
    assert len(sols) == 5
    return sols + [-1]


def solution_ntok(pk, mode, m, n, k, sid):
    if sid == -1:
        import petit_kernel.tuning as tuning

        sid = tuning.default_solution(m, n, k, MODES[mode][1], mx=MODES[mode][0] == "mxfp4")
    return (sid & 0xFF) * 16


def gemm(pk, mode, a, b, sp, gs, m, n, k, sid, out=None, bias=None, residual=None, silu=False):
    mx = MODES[mode][0] == "mxfp4"
    return pk.ops.mul_fp4_a16_ex_out(out, a, b, sp, gs, m, n, k, sid, mx, bias, residual, silu)


def assert_bits(got, want, what):
    """Bit-exact, +0 == -0; NaN only where expected (same positions)."""
    got, want = got.cpu(), want.cpu()
    assert got.dtype == want.dtype and got.shape == want.shape, what
    nan_g, nan_w = torch.isnan(got.float()), torch.isnan(want.float())
    assert torch.equal(nan_g, nan_w), (what, "NaN positions differ", int((nan_g ^ nan_w).sum()))
    gi, wi = got.view(torch.int16), want.view(torch.int16)
    bad = (gi != wi) & ~(((gi & 0x7FFF) == 0) & ((wi & 0x7FFF) == 0)) & ~nan_w
    if bool(bad.any()):
        idx = bad.nonzero()[:5].tolist()
        vals = [(got[i, j].item(), want[i, j].item()) for i, j in idx]
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} outputs differ, first {idx}: {vals}")


def plan_labels(cuts_fn, mode, m, n, k, ntok, sms, all_reduce=False):
    """Coverage labels that hold with and without programmatic dependent launch (the first GEMM
    after a repack on a stream runs without it)."""
    got = None
    for pdl in (True, False):
        p = orc.stream_k_plan(m, n, k, ntok, sms, pdl, True, cuts_fn, mode=mode, all_reduce=all_reduce)
        lab = orc.plan_paths(p)
        got = lab if got is None else got & lab
    return got


def coverage_table(pk, cuts_fn, mode, sms):
    """{label: sorted list of (shape, token tile) that reach it} over DENSE_SHAPES x solutions."""
    table = {}
    for shape in DENSE_SHAPES:
        m, n, k = mode_shape(mode, *shape)
        for sid in solutions(pk, mode, m, n, k):
            ntok = solution_ntok(pk, mode, m, n, k, sid)
            for lab in plan_labels(cuts_fn, mode, m, n, k, ntok, sms):
                table.setdefault(lab, set()).add(((m, n, k), ntok))
    return {lab: sorted(v) for lab, v in table.items()}


# ------------------------------------------------------------------ dense exact GEMMs
@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_dense_exact_all_solutions(pk, cuts_fn, mode):
    """Every solution id and -1 on every DENSE_SHAPES entry: bit-exact against oracle.exact_ref.
    The stream-K plan of the launches must reach every REQUIRED_PATHS row."""
    fmt, dt, _ = MODES[mode]
    table = coverage_table(pk, cuts_fn, mode, num_sms())
    print(f"\ncoverage {mode}: " + "; ".join(
        f"{lab}: {sorted({t for _, t in table.get(lab, [])})}" for lab in REQUIRED_PATHS))
    missing = [lab for lab in REQUIRED_PATHS if lab not in table]
    assert not missing, f"{mode}: no launch reaches {missing}"
    for shape in DENSE_SHAPES:
        m, n, k = mode_shape(mode, *shape)
        a, q, s, gs, w, _ = orc.make_exact_case(fmt, dt, m, n, k, SEED)
        b, sp = pack(pk, mode, q, s, n, k)
        ac, gsc = a.cuda(), gs.cuda()
        want = orc.exact_ref(ac, w, gs.item(), dt)
        assert torch.isfinite(want.float()).all()
        for sid in solutions(pk, mode, m, n, k):
            got = gemm(pk, mode, ac, b, sp, gsc, m, n, k, sid)
            assert_bits(got, want, f"{mode} m={m} n={n} k={k} sol={sid:#x}")


# ------------------------------------------------------------------ one-hot probes
PROBE_M, PROBE_N, PROBE_K = 256, 256, 4096


def probe_columns(r):
    """k column probed by each of the 256 tokens in launch r: token m = 16 t + l reads k-tile l,
    chunk (t + r) % 8 of it and position (5 t + 3 l + 11 r) % 32 inside that 32-weight chunk, so
    every token tile has a non-zero input in every k-tile (every CTA of every plan adds a
    non-zero partial) and the launches together cover every 16-group and chunk position."""
    m = np.arange(PROBE_M)
    t, l = m // 16, m % 16
    return 256 * l + 32 * ((t + r) % 8) + (5 * t + 3 * l + 11 * r) % 32


def probe_weights(fmt):
    n, k = PROBE_N, PROBE_K
    nn, jj = np.meshgrid(np.arange(n), np.arange(k), indexing="ij")
    codes = ((3 * nn + jj) % 16).astype(np.uint8)
    q = (codes[:, 0::2] | (codes[:, 1::2] << 4)).astype(np.uint8)
    if fmt == "nvfp4":   # every e4m3 code 0x00 .. 0x7E in every probed group
        g = np.arange(k // 16)[None, :]
        s = ((np.arange(n)[:, None] + 7 * g) % 127).astype(np.uint8)
    else:                # every e8m0 1 .. 237; small and large inside every 32-row warp group
        g = np.arange(k // 32)[None, :]
        s = (1 + (29 * np.arange(n)[:, None] + 13 * g) % 237).astype(np.uint8)
    return q, s


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_one_hot_probes(pk, cuts_fn, mode):
    """Token m's activations are +-2^e at one k: C[m, :] = RN16(RN32(+-2^e w[:, j_m] gs)), one
    exact product.  Covers every scale code (NVFP4 e4m3 0x00..0x7E, MXFP4 e8m0 1..237 with the
    forced two-step multiply on small scales next to large ones in one warp), every 16-group,
    every position in a 32-weight chunk, the first and last k-tile and every stream-K range."""
    fmt, dt, _ = MODES[mode]
    m, n, k = PROBE_M, PROBE_N, PROBE_K
    q, s = probe_weights(fmt)
    w = orc.dequant_nvfp4(q, s) if fmt == "nvfp4" else orc.dequant_mxfp4(q, s)
    st = torch.from_numpy(s)
    b, sp = pack(pk, mode, torch.from_numpy(q), st.view(torch.float8_e4m3fn) if fmt == "nvfp4" else st, n, k)
    gs = 0.7
    gsc = torch.tensor([gs], device="cuda")
    group = 16 if fmt == "nvfp4" else 32
    seen_groups, seen_pos, seen_scales = set(), set(), set()
    for r in range(4):
        cols = probe_columns(r)
        rs = np.random.RandomState(r)
        sign = np.where(rs.rand(m) < 0.5, -1.0, 1.0)
        mag = 4.0 if fmt == "mxfp4" else 2.0 ** rs.randint(0, 2, size=m)  # outputs stay normal
        a = np.zeros((m, k), dtype=np.float32)
        a[np.arange(m), cols] = sign * mag
        ac = torch.from_numpy(a).to(dt).cuda()
        want = orc.exact_ref(ac, w, gs, dt)
        nz = want.float().abs()
        assert torch.isfinite(nz).all() and bool((nz[nz > 0] >= torch.finfo(dt).tiny).all())
        for sid in solutions(pk, mode, m, n, k):
            got = gemm(pk, mode, ac, b, sp, gsc, m, n, k, sid)
            assert_bits(got, want, f"{mode} probe r={r} sol={sid:#x}")
        seen_groups |= set((cols // group).tolist())
        seen_pos |= set((cols % 32).tolist())
        for j in set(cols.tolist()):
            seen_scales |= set(s[:, j // group].tolist())
        if fmt == "mxfp4":  # the per-warp two-step decision really is mixed
            for j in set(cols.tolist()):
                blocks = s[:, j // group].reshape(-1, 32)
                assert bool(((blocks > 125).any(1) & (blocks <= 125).any(1)).all())
    assert seen_groups == set(range(k // group)) and seen_pos == set(range(32))
    assert seen_scales == (set(range(127)) if fmt == "nvfp4" else set(range(1, 238)))
    # every token tile has a non-zero input in every k-tile, so every CTA's range matters
    ktiles = {(mm // 16, c // 256) for mm, c in enumerate(probe_columns(0))}
    assert ktiles == {(t, kt) for t in range(m // 16) for kt in range(k // 256)}


# ------------------------------------------------------------------ range edges
def run_exact(pk, mode, a, q, s, gs, m, n, k, sols=None):
    """Pack, run every solution, compare bit for bit with exact_ref; return the expectation."""
    fmt, dt, _ = MODES[mode]
    w = orc.dequant_nvfp4(q, s) if fmt == "nvfp4" else orc.dequant_mxfp4(q, s)
    st = torch.from_numpy(np.ascontiguousarray(s))
    b, sp = pack(pk, mode, torch.from_numpy(np.ascontiguousarray(q)),
                 st.view(torch.float8_e4m3fn) if fmt == "nvfp4" else st, n, k)
    ac = a.to(dt).cuda()
    want = orc.exact_ref(ac, w, gs, dt)
    gsc = torch.tensor([gs], dtype=torch.float32, device="cuda")
    for sid in sols or solutions(pk, mode, m, n, k):
        assert_bits(gemm(pk, mode, ac, b, sp, gsc, m, n, k, sid), want, f"{mode} sol={sid:#x} gs={gs}")
    return want


def uniform_weights(fmt, n, k, code, scale):
    q = np.full((n, k // 2), code * 0x11, dtype=np.uint8)
    s = np.full((n, k // (16 if fmt == "nvfp4" else 32)), scale, dtype=np.uint8)
    return q, s


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_overflow_to_signed_inf(pk, mode):
    """Outputs beyond the 16-bit range are +-inf with the product's sign; the other tokens and
    columns of the same tiles are unaffected."""
    fmt, dt, _ = MODES[mode]
    m, n, k = 32, 256, 1024
    q, s = uniform_weights(fmt, n, k, 0x7, 0x7E if fmt == "nvfp4" else 200)  # +6 x 448 / x 2^73
    q[n // 2:] = 0x11  # +0.5 x a small scale: stays finite
    s[n // 2:] = 0x08 if fmt == "nvfp4" else 100       # 2^-6 / 2^-27
    w_big = 6 * (448.0 if fmt == "nvfp4" else 2.0 ** 73)
    if dt == torch.float16:
        e_big, gs = 4, 2.0                      # 2688 x 16 x 2 = 86016 > 65504
    else:
        e_big, gs = (100 if fmt == "nvfp4" else 50), 2.0 ** 20
    a = torch.zeros((m, k))
    a[0, 5], a[1, 700], a[2, 3] = 2.0 ** e_big, -(2.0 ** e_big), 1.0
    want = run_exact(pk, mode, a, q, s, gs, m, n, k)
    assert w_big * 2.0 ** e_big * gs > torch.finfo(dt).max
    assert bool(torch.isposinf(want[0, : n // 2].float()).all()) and bool(torch.isneginf(want[1, : n // 2].float()).all())
    assert bool(torch.isfinite(want[:, n // 2:].float()).all()) and bool(torch.isfinite(want[2:].float()).all())


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_subnormal_outputs_round_exactly(pk, mode):
    """A tiny global scale puts dense exact outputs into the 16-bit subnormal range (bf16: also
    the fp32 one).  The epilogue runs on CUDA cores without flush-to-zero, so RN32 and RN16 of
    the subnormal values must match the host's IEEE rounding bit for bit."""
    fmt, dt, _ = MODES[mode]
    m, n, k = 48, 256, 2048
    a, q, s, _, w, _ = orc.make_exact_case(fmt, dt, m, n, k, 5)
    if dt == torch.float16:
        gs = 0.7 * 2.0 ** -30                    # |S| ~ 2^6..2^11 -> 2^-24 .. 2^-19
    elif fmt == "nvfp4":
        gs = 0.7 * 2.0 ** -138                   # fp32 subnormal gs; gs * 256 is exact
    else:
        gs = 2.0 ** -134                         # gs * 0.25 stays exact
    s_np = s.view(torch.uint8).numpy() if fmt == "nvfp4" else s.numpy()
    want = run_exact(pk, mode, a, q.numpy(), s_np, gs, m, n, k)
    v = want.float().abs()
    tiny = torch.finfo(dt).tiny
    assert bool(((v > 0) & (v < tiny)).float().mean() > 0.5), "most outputs must be subnormal"


@pytest.mark.gpu
def test_products_below_fp32_normal_inside_the_mma(pk):
    """Products below 2^-126 inside tcgen05.mma (bf16 x bf16 -> fp32): one-hot activations of
    2^-120 (NVFP4, A operand 2^-18) / 2^-10 (MXFP4 e8m0 1, A operand 2^-125) make products of
    2^-138 / 2^-135, and a large global scale lifts the result into the bf16 normal range.  Measured on B200: the MMA
    keeps fp32 subnormal products and accumulates them exactly (IEEE), it does not flush them to
    zero -- the outputs are 2^-90 / 2^-86 / 2^-89 (NVFP4) and 2^-37 / 2^-33 / 2^-36 (MXFP4), not
    0 (DESIGN.md, 'Numerics')."""
    m, n, k = 16, 128, 1024
    results = {}
    for mode, scale, e, gs in (("nv_bf16", 0x01, -120, 2.0 ** 40), ("mx_bf16", 1, -10, 2.0 ** 100)):
        fmt = MODES[mode][0]
        q, s = uniform_weights(fmt, n, k, 0x1, scale)  # +0.5 x smallest scale
        a = torch.zeros((m, k))
        a[0, 7] = 2.0 ** e                  # one subnormal product
        a[1, :16] = 2.0 ** e                # sixteen in one MMA k-step
        a[2, 7], a[2, 300] = 2.0 ** e, 2.0 ** e  # two, in different k-tiles
        fmt_w = orc.dequant_nvfp4(q, s) if fmt == "nvfp4" else orc.dequant_mxfp4(q, s)
        ieee = orc.exact_ref(a.to(torch.bfloat16), fmt_w, gs, torch.bfloat16)
        b, sp = pack(pk, mode, torch.from_numpy(q), torch.from_numpy(s).view(torch.float8_e4m3fn)
                     if fmt == "nvfp4" else torch.from_numpy(s), n, k)
        got = gemm(pk, mode, a.to(torch.bfloat16).cuda(), b, sp, torch.tensor([gs], device="cuda"),
                   m, n, k, -1).cpu()
        results[mode] = (got[:3, 0].float().tolist(), ieee[:3, 0].float().tolist())
    print("\nsubnormal products (got, ieee):", results)
    for mode, (got, ieee) in results.items():
        assert got == ieee and all(v > 0 for v in got), (mode, got, ieee)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_nan_zero_and_negative_global_scale(pk, mode):
    """A NaN activation in one token stays in that token's row through split tiles (every
    reducer path); gs = 0 gives zeros; a negative gs flips every sign exactly."""
    fmt, dt, _ = MODES[mode]
    for shape in ((16, 2048, 8192), (64, 128, 28672), (17, 1040, 4096)):
        m, n, k = mode_shape(mode, *shape)
        a, q, s, gs, w, _ = orc.make_exact_case(fmt, dt, m, n, k, 7)
        s_np = s.view(torch.uint8).numpy() if fmt == "nvfp4" else s.numpy()
        a[3, k - 100] = float("nan")
        want = run_exact(pk, mode, a, q.numpy(), s_np, gs.item(), m, n, k)
        assert bool(torch.isnan(want[3].float()).all()) and not bool(torch.isnan(want[torch.arange(m) != 3].float()).any())
    m, n, k = 33, 256, 2048
    a, q, s, _, w, _ = orc.make_exact_case(fmt, dt, m, n, k, 8)
    s_np = s.view(torch.uint8).numpy() if fmt == "nvfp4" else s.numpy()
    zero = run_exact(pk, mode, a, q.numpy(), s_np, 0.0, m, n, k)
    assert not bool(zero.float().abs().max())
    neg = run_exact(pk, mode, a, q.numpy(), s_np, -0.7, m, n, k)
    pos = orc.exact_ref(a.to(dt), w, 0.7, dt)
    assert torch.equal(neg.float(), -pos.float())


# ------------------------------------------------------------------ fused epilogues
@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_fused_bias_residual_bit_exact(pk, mode):
    """bias[n] and residual[m, n] (arbitrary 16-bit values) added in fp32 after RN32(S * gs),
    in that order, then one RN16: bit-exact on split tiles, partial n- and token tiles, every
    solution, and with the residual aliasing the output."""
    fmt, dt, _ = MODES[mode]
    for shape in ((17, 1040, 4096), (100, 240, 2048), (5, 512, 4096), (256, 1024, 2048)):
        m, n, k = mode_shape(mode, *shape)
        a, q, s, gs, w, _ = orc.make_exact_case(fmt, dt, m, n, k, 9)
        b, sp = pack(pk, mode, q, s, n, k)
        ac, gsc = a.cuda(), gs.cuda()
        g = torch.Generator().manual_seed(m + n)
        bias = (torch.randn(n, generator=g) * 500).to(dt)
        resid = (torch.randn(m, n, generator=g) * 500).to(dt)
        for bb, rr in ((bias, None), (None, resid), (bias, resid)):
            want = orc.exact_ref(ac, w, gs.item(), dt, bb, rr)
            for sid in solutions(pk, mode, m, n, k):
                got = gemm(pk, mode, ac, b, sp, gsc, m, n, k, sid, None,
                           None if bb is None else bb.cuda(), None if rr is None else rr.cuda())
                assert_bits(got, want, f"{mode} {shape} bias={bb is not None} res={rr is not None} sol={sid:#x}")
        out = resid.cuda().clone()
        gemm(pk, mode, ac, b, sp, gsc, m, n, k, -1, out, bias.cuda(), out)
        assert_bits(out, orc.exact_ref(ac, w, gs.item(), dt, bias, resid), f"{mode} {shape} in place")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["nv_bf16", "nv_f16", "mx_bf16"])
def test_fused_silu_mul_on_exact_gemm(pk, mode):
    """SiLU(gate) * up on an exact GEMM: the GEMM outputs are known bit for bit, so the fused
    epilogue must equal RN16(RN16(silu(g)) * u) from them up to the last bit of expf."""
    fmt, dt, _ = MODES[mode]
    for m, n, k in ((16, 1024, 4096), (37, 512, 1024)):
        a, q, s, _, w, _ = orc.make_exact_case(fmt, dt, m, n, k, 13)
        gs = 0.7 * 2.0 ** -9   # keeps silu's argument in its interesting range
        b, sp = pack(pk, mode, q, s, n, k)
        ac = a.cuda()
        c = orc.exact_ref(ac, w, gs, dt).float().view(m, n // 128, 2, 64)
        want = (torch.nn.functional.silu(c[:, :, 0]).to(dt).float() * c[:, :, 1]).to(dt).reshape(m, n // 2)
        for sid in solutions(pk, mode, m, n, k):
            got = gemm(pk, mode, ac, b, sp, torch.tensor([gs], device="cuda"), m, n, k, sid, silu=True).cpu()
            diff = (got.float() - want.float()).abs()
            assert bool((diff <= orc.ulp16(want.float(), dt)).all()), (mode, m, sid, diff.max().item())
            assert (got == want).float().mean().item() > 0.98


GROUPED_CASES = ((512, 1024, [5, 0, 33, 1, 16, 70]),      # 64-token tiles
                 (2048, 4096, [3, 1, 0, 7, 2, 16, 4, 1]),  # 16-token tiles split by stream-K
                 (1040, 768, [17, 32, 0, 0, 9]))           # 32-token tiles, partial n-tile


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["nv_bf16", "nv_f16", "mx_bf16"])
def test_grouped_exact_single_launch_equals_one_by_one(pk, mode):
    """Grouped GEMM with a distinct non-power-of-two gs per expert, ragged and empty groups,
    NaN-filled outputs: the single-launch kernel and the one-by-one launches both equal the
    per-expert exact reference, hence each other, bit for bit."""
    fmt, dt, _ = MODES[mode]
    for n, k, counts in GROUPED_CASES:
        n = mode_shape(mode, 16, n, k)[1]
        offsets = np.concatenate([[0], np.cumsum(counts)]).tolist()
        a_all, bs, ss, gss, wants = [], [], [], [], []
        for g, cnt in enumerate(counts):
            a, q, s, _, w, _ = orc.make_exact_case(fmt, dt, max(cnt, 1), n, k, 200 + g)
            gs = 0.7 + 0.05 * g
            b, sp = pack(pk, mode, q, s, n, k)
            a_all.append(a[:cnt]); bs.append(b); ss.append(sp); gss.append(gs)
            wants.append(orc.exact_ref(a[:cnt], w, gs, dt))
        a_cat = torch.cat(a_all).cuda().contiguous()
        gsc = torch.tensor(gss, dtype=torch.float32, device="cuda")
        outs = []
        for single in ("1", "0"):
            os.environ["PETIT_GROUPED_SINGLE"] = single
            try:
                out = torch.full((offsets[-1], n), float("nan"), dtype=dt, device="cuda")
                pk.ops.mul_fp4_a16_grouped_out(out, a_cat, torch.stack(bs), torch.stack(ss), gsc, offsets,
                                               n, k, -1, fmt == "mxfp4")
                torch.cuda.synchronize()
            finally:
                os.environ.pop("PETIT_GROUPED_SINGLE", None)
            outs.append(out.cpu())
            assert_bits(out, torch.cat(wants), f"{mode} grouped n={n} k={k} single={single}")
        assert torch.equal(outs[0].view(torch.int16), outs[1].view(torch.int16))


# ------------------------------------------------------------------ launch configuration
# (mode, m, n, k): computed in this process and again in subprocesses with PETIT_PDL=0,
# PETIT_CLUSTER=0, PETIT_WHOLE_TILES=0 and other tilt parameters
INVARIANCE_CASES = [(mode, *mode_shape(mode, *shape)) for mode in ("nv_bf16", "nv_f16", "mx_bf16")
                    for shape in ((16, 8192, 1024), (48, 4096, 4096), (64, 128, 28672), (256, 1024, 2048))]
SUBPROCESS_ENV = {"PETIT_PDL": "0", "PETIT_CLUSTER": "0", "PETIT_WHOLE_TILES": "0",
                  "PETIT_TILT_UNITS": "2", "PETIT_TILT_LATE": "7"}


def invariance_outputs(pk):
    """{name: output bits} of INVARIANCE_CASES for every solution id."""
    res = {}
    for mode, m, n, k in INVARIANCE_CASES:
        fmt, dt, _ = MODES[mode]
        a, q, s, gs, _, _ = orc.make_exact_case(fmt, dt, m, n, k, 21)
        b, sp = pack(pk, mode, q, s, n, k)
        for sid in solutions(pk, mode, m, n, k):
            c = gemm(pk, mode, a.cuda(), b, sp, gs.cuda(), m, n, k, sid)
            res[f"{mode}_{m}_{n}_{k}_{sid & 0xFFFFFFFFFFFFFFFF:x}"] = c.cpu().view(torch.int16).numpy()
    return res


@pytest.mark.gpu
def test_results_do_not_depend_on_launch_switches(pk, cuts_fn, tmp_path):
    """The same exact GEMMs in fresh processes with programmatic dependent launch, clusters and
    whole-tile grids off and different cut parameters (read once per process): identical bits,
    and those switches do change the launch plans."""
    here = invariance_outputs(pk)
    sms = num_sms()
    changed = 0
    for mode, m, n, k in INVARIANCE_CASES:
        for ntok in (16, 32, 64, 128, 256):
            dflt = orc.stream_k_plan(m, n, k, ntok, sms, True, True, cuts_fn, mode=mode)
            env = orc.stream_k_plan(m, n, k, ntok, sms, False, False, cuts_fn, mode=mode,
                                    whole_tiles_rule=False, tilt_units=2, tilt_late=7)
            changed += (dflt["grid"], dflt["cuts"], dflt["cluster"]) != (env["grid"], env["cuts"], env["cluster"])
    assert changed >= 8, changed
    env = dict(os.environ, **SUBPROCESS_ENV)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "test_gemm_exact.py"), str(tmp_path)],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    for name, bits in here.items():
        other = np.load(tmp_path / f"{name}.npy")
        assert np.array_equal(bits, other), name


def chain_layers(fmt, dt, m):
    """Three GEMMs whose inputs are the previous outputs: G1's one-hot activations pick weight
    columns of {+-1/2, +-1, +-2} (gs = 1), so its output is an exact activation matrix for G2;
    G3 takes G2's output as residual."""
    k1, k2, n2, k3 = 1024, 4096, 2048, 2048
    rs = np.random.RandomState(3)
    codes = np.array([1, 2, 4, 9, 10, 12], dtype=np.uint8)  # +-0.5, +-1, +-2
    nib = codes[rs.randint(0, 6, size=(k2, k1))]
    q1 = (nib[:, 0::2] | (nib[:, 1::2] << 4)).astype(np.uint8)
    s1 = np.full((k2, k1 // (16 if fmt == "nvfp4" else 32)), 0x38 if fmt == "nvfp4" else 127, dtype=np.uint8)
    a1 = np.zeros((m, k1), dtype=np.float32)
    a1[np.arange(m), rs.randint(0, k1, size=m)] = 1.0
    _, q2, s2, _, w2, _ = orc.make_exact_case(fmt, dt, m, n2, k2, 31)
    a3, q3, s3, _, w3, _ = orc.make_exact_case(fmt, dt, m, n2, k3, 32)
    s2 = s2.view(torch.uint8).numpy() if fmt == "nvfp4" else s2.numpy()
    s3 = s3.view(torch.uint8).numpy() if fmt == "nvfp4" else s3.numpy()
    return [(torch.from_numpy(a1), q1, s1, 1.0, k2, k1), (None, q2.numpy(), s2, 0.7, n2, k2),
            (a3, q3.numpy(), s3, 0.9, n2, k3)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["nv_bf16", "mx_bf16"])
def test_pdl_chain_and_graph_replay(pk, mode):
    """G1 -> G2 (activations = G1's output) -> G3 (residual = G2's output), repeated on one
    stream with programmatic dependent launch (a stale read ahead of griddepcontrol.wait would
    show), then captured in a CUDA graph and replayed: every output bit-exact."""
    fmt, dt, _ = MODES[mode]
    m = 32
    layers = chain_layers(fmt, dt, m)
    packed, ws = [], []
    for a, q, s, gs, n, k in layers:
        st = torch.from_numpy(s)
        packed.append(pack(pk, mode, torch.from_numpy(q), st.view(torch.float8_e4m3fn) if fmt == "nvfp4" else st, n, k))
        ws.append(orc.dequant_nvfp4(q, s) if fmt == "nvfp4" else orc.dequant_mxfp4(q, s))
    gscs = [torch.tensor([l[3]], device="cuda") for l in layers]
    a1, a3 = layers[0][0].to(dt).cuda(), layers[2][0].to(dt).cuda()
    c1_want = orc.exact_ref(a1, ws[0], 1.0, dt)
    assert set(c1_want.float().unique().tolist()) <= {0.0, 0.5, 1.0, 2.0, -0.5, -1.0, -2.0}
    c2_want = orc.exact_ref(c1_want.cuda(), ws[1], 0.7, dt)
    c3_want = orc.exact_ref(a3, ws[2], 0.9, dt, None, c2_want)
    (b1, s1), (b2, s2), (b3, s3) = packed

    def step():
        c1 = gemm(pk, mode, a1, b1, s1, gscs[0], m, layers[0][4], layers[0][5], -1)
        c2 = gemm(pk, mode, c1, b2, s2, gscs[1], m, layers[1][4], layers[1][5], -1)
        c3 = gemm(pk, mode, a3, b3, s3, gscs[2], m, layers[2][4], layers[2][5], -1, None, None, c2)
        return c1, c2, c3

    for it in range(4):
        outs = step()
    for got, want, name in zip(outs, (c1_want, c2_want, c3_want), ("c1", "c2", "c3")):
        assert_bits(got, want, f"{mode} chain {name}")
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        gouts = step()
    for it in range(3):
        for o in gouts:
            o.fill_(float("nan"))
        g.replay()
        torch.cuda.synchronize()
        for got, want, name in zip(gouts, (c1_want, c2_want, c3_want), ("c1", "c2", "c3")):
            assert_bits(got, want, f"{mode} graph replay {it} {name}")


if __name__ == "__main__":
    import petit_kernel

    for name, bits in invariance_outputs(petit_kernel).items():
        np.save(os.path.join(sys.argv[1], f"{name}.npy"), bits)
