"""Bit-exact tests of the grouped (MoE) GEMM (petit_gemm_fp4_a16_grouped, ops.mul_fp4_a16_grouped_out)
against per-expert exact references, in both launch forms.

Every expert is an oracle.make_exact_case of its own (own seed, own non-power-of-two gs), so expert
g's rows of the output must equal oracle.exact_ref of that expert bit for bit, whichever form the
call takes:
  single      one launch of fp4_gemm_kernel<..., GR = true> whose stream-K schedule runs over the
              token tiles of all experts (oracle.group_table): weights, scales and gs change from
              one table entry to the next inside one CTA's k-range, a token tile loads NTOK rows
              (the rows behind an expert's last token are the next expert's), and a tile whose
              rows are not a multiple of 16 writes its last 16-token group with direct stores;
  one_by_one  one plain stream-K launch per live expert, chained by programmatic dependent launch.
Which form a call takes (oracle.grouped_launch) is asserted from the kernel names torch.profiler
records (their template arguments carry NTOK and GR), not assumed.  The outputs are views into a
larger buffer with sentinel guard rows on both sides, which must stay untouched.  Which stream-K
paths the single launches reach is asserted per mode (GROUPED_REQUIRED)."""
import ctypes
import functools
import os
import re

import numpy as np
import pytest
import torch

from helpers import LIB_PATH, orc, stream_k_cuts_fn
import test_gemm_exact as tge
from test_gemm_exact import MODES, assert_bits, pack

GUARD_ROWS = 2
SENTINEL = -3.0          # exact in bf16 and fp16; the guard rows must keep these bits
SEED = 500


def topk_counts(experts, tokens, topk, seed):
    """Tokens per expert when each of `tokens` tokens is routed to `topk` distinct experts."""
    rs = np.random.RandomState(seed)
    counts = np.zeros(experts, dtype=np.int64)
    for _ in range(tokens):
        counts[rs.choice(experts, topk, replace=False)] += 1
    return counts.tolist()


BENCH_DECODE = [4, 5, 3, 4, 6, 2, 4, 4]           # bench.py moe_grouped: a decode step, 8 experts
BENCH_BATCH = [16, 20, 12, 16, 24, 8, 16, 16]
QWEN3 = topk_counts(128, 16, 8, 7)                 # 128 experts, top-8 routing of 16 tokens
# name: (n, k, tokens per expert)
ROUTINGS = {
    "ragged_64": (512, 1024, [5, 0, 33, 1, 16, 70]),                 # 64-token tiles, two for the last
    "ragged_16_split": (2048, 4096, [3, 1, 0, 7, 2, 16, 4, 1]),      # 16-token tiles split by stream-K
    "ragged_32_partial_n": (1040, 768, [17, 32, 0, 0, 9]),           # partial n-tile
    "empties_at_both_ends": (1040, 4096, [0, 0, 5, 0, 33, 1, 16, 70, 0]),
    "tile_edges": (2048, 768, [16, 15, 17, 32, 31, 33, 64, 63, 65]),  # exactly 16/32/64 and +-1
    "one_expert": (512, 1024, [0, 0, 40, 0]),                        # one live group: one by one
    "all_empty": (512, 1024, [0, 0, 0]),                             # no launch at all
    "tiles_96": (256, 512, [(7 * i) % 16 + 1 for i in range(96)]),   # a full table at 16-token tiles
    "tiles_97": (256, 512, [(7 * i) % 16 + 1 for i in range(97)]),   # one entry too many
    "ring": (1152, 8192, [7, 0, 12]),                                # 4 .. kRingFit contributors
    "l2_tail": (128, 28672, [40, 5, 0, 20]),                         # > kRingFit contributors
    "whole_tiles": (2048, 768, [9, 30, 0, 21, 2]),                   # one whole tile per CTA
    "qwen3_w13": (1536, 2048, QWEN3),
    "qwen3_w2": (2048, 768, QWEN3),
    "mixtral_tp8_w13_decode": (3584, 4096, BENCH_DECODE),
    "mixtral_tp8_w2_decode": (4096, 1792, BENCH_DECODE),
    "mixtral_tp8_w13_batch": (3584, 4096, BENCH_BATCH),
    "bench_64_experts": (2048, 2048, [2] * 64),
}
# every label must be reached by a single launch of every mode
GROUPED_REQUIRED = ("whole_tiles", "tilt", "unsplit", "reg_1_3", "ring", "many_m_le16", "many_m_gt16", "l2_tail",
                    "split_partial_n", "group_switch", "split_group_tail", "direct_store", "multi_tile_group",
                    "table_full")
KERNEL_NAME = re.compile(r"fp4_gemm_kernel<(\d+), (\d+), (\d+), (true|false), (true|false), (true|false)>")


def mode_n(mode, n):
    """MXFP4 scales and the fp16-native layout's shape tag need n % 32 == 0: partial n-tiles of
    32 / 96 rows stand in for 16 / 112 there."""
    fmt, _, native = MODES[mode]
    if (fmt == "mxfp4" or native) and n % 32:
        n = n + 16 if n % 128 == 16 else n - 16
    return n


def expert_gs(g):
    """A distinct global scale per expert, none a power of two, all in (0.43, 0.7] so that the
    fp16 outputs of the exact cases stay finite."""
    return 0.7 - 0.0021 * g


def offsets_of(counts):
    return np.concatenate([[0], np.cumsum(counts)]).astype(np.int64).tolist()


@functools.lru_cache(maxsize=2)
def expert_cases(fmt, n, k, counts, seed):
    """Per expert g: (activations [counts[g], k] bf16 (exact in fp16 too), e2m1 bytes, scale bytes,
    S = a @ w^T in float64).  The dequantised weights are not kept (128 experts of Qwen3's w13
    would be 1.6 GB of them)."""
    out = []
    for g, c in enumerate(counts):
        a, q, s, _, w, _ = orc.make_exact_case(fmt, torch.bfloat16, max(c, 1), n, k, seed + g)
        a = a[:c]
        s_np = s.view(torch.uint8).numpy() if fmt == "nvfp4" else s.numpy()
        out.append((a, q.numpy(), s_np, (a.double() @ torch.from_numpy(w).double().t()).numpy()))
    return tuple(out)


def pack_experts(pk, mode, cases, n, k):
    """[E, ...] stacks of the packed weights and scales."""
    fmt, _, native = MODES[mode]
    bs, ss = [], []
    for _, q, s, _ in cases:
        st = torch.from_numpy(s)
        b, sp = pack(pk, mode, torch.from_numpy(q), st.view(torch.float8_e4m3fn) if fmt == "nvfp4" else st, n, k)
        if native:
            assert tuple(b.shape) == (n // 32, 4 * k), "not the fp16-native layout"
        bs.append(b)
        ss.append(sp)
    return torch.stack(bs), torch.stack(ss)


def guarded_out(rows, cols, dt):
    """(buffer, out): out = rows NaN-filled rows of a buffer with SENTINEL guard rows around it."""
    buf = torch.full((rows + 2 * GUARD_ROWS, cols), SENTINEL, dtype=dt, device="cuda")
    out = buf[GUARD_ROWS:GUARD_ROWS + rows]
    out.fill_(float("nan"))
    return buf, out


def assert_guards(buf, what):
    g = torch.cat([buf[:GUARD_ROWS], buf[buf.shape[0] - GUARD_ROWS:]]).cpu()
    assert bool((g.float() == SENTINEL).all()), f"{what}: a guard row was written"


def gemm_kernels(fn):
    """Run fn() under torch.profiler: (fn's result, [(ntok, grouped)] of the fp4_gemm_kernel launches
    in launch order)."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    found = []
    for e in prof.events():
        mm = KERNEL_NAME.search(e.name)
        if mm and e.device_type == torch.autograd.DeviceType.CUDA:
            found.append((e.time_range.start, int(mm.group(2)), mm.group(6) == "true"))
    return res, [(t, gr) for _, t, gr in sorted(found)]


def expected_kernels(pk, mode, counts, n, k, sid, single_env=True, contiguous=True, bias=False):
    """[(ntok, grouped)] that oracle.grouped_launch predicts for one call."""
    form, ntok, launches = orc.grouped_launch(counts, n, k, sid, MODES[mode][1], contiguous, bias, single_env)
    if form == "single":
        return [(ntok, True)]
    return [(tge.solution_ntok(pk, mode, m, n, k, sid), False) for _, m in launches]


def sid_by_ntok(pk, mode, n, k):
    """{ntok: explicit solution id} for 16 .. 256-token tiles."""
    return {tge.solution_ntok(pk, mode, 16, n, k, s): s for s in tge.solutions(pk, mode, 16, n, k) if s != -1}


def call_grid(pk, mode, n, k):
    """(sid, PETIT_GROUPED_SINGLE) of every call: -1 and every decode id in both settings, and the
    128-token id (which must go one by one)."""
    ids = sid_by_ntok(pk, mode, n, k)
    return [(sid, env) for sid in (-1, ids[16], ids[32], ids[64]) for env in ("1", "0")] + [(ids[128], "1")]


def grouped(pk, mode, out, a, b, sp, gsc, counts, n, k, sid, env="1", silu=False):
    os.environ["PETIT_GROUPED_SINGLE"] = env
    try:
        pk.ops.mul_fp4_a16_grouped_out(out, a, b, sp, gsc, offsets_of(counts), n, k, sid,
                                       MODES[mode][0] == "mxfp4", silu)
    finally:
        os.environ.pop("PETIT_GROUPED_SINGLE", None)
    return out


def run_calls(pk, mode, counts, n, k, a_cat, b, sp, gs_list, want, what, calls=None):
    """Every call of call_grid (or `calls`) into a fresh guarded NaN-filled output: bit-exact
    against `want`, guard rows untouched, and the launch form and token tile oracle.grouped_launch
    predicts.  Returns the output bits of every call."""
    dt = MODES[mode][1]
    gsc = torch.tensor(gs_list, dtype=torch.float32, device="cuda")
    calls = calls or call_grid(pk, mode, n, k)
    outs = []

    def run():
        for sid, env in calls:
            buf, out = guarded_out(a_cat.shape[0], n, dt)
            grouped(pk, mode, out, a_cat, b, sp, gsc, counts, n, k, sid, env)
            outs.append((buf, out, sid, env))

    _, kernels = gemm_kernels(run)
    expect = []
    for sid, env in calls:
        expect += expected_kernels(pk, mode, counts, n, k, sid, env == "1")
    assert kernels == expect, (what, "launches (ntok, grouped)", kernels, expect)
    bits = []
    for buf, out, sid, env in outs:
        tag = f"{what} sol={sid & 0xFFFFFFFFFFFFFFFF:#x} single={env}"
        assert_bits(out, want, tag)
        assert_guards(buf, tag)
        bits.append(out.cpu().view(torch.int16))
    return bits


def routing_case(pk, mode, routing, seed=SEED):
    """(n, k, counts, a_cat on the device, b stack, scale stack, gs per expert, exact want)."""
    fmt, dt, _ = MODES[mode]
    n0, k, counts = ROUTINGS[routing]
    n = mode_n(mode, n0)
    cases = expert_cases(fmt, n, k, tuple(counts), seed)
    b, sp = pack_experts(pk, mode, cases, n, k)
    gs = [expert_gs(g) for g in range(len(counts))]
    want = torch.cat([orc.exact_epilogue(S, gs[g], dt) for g, (_, _, _, S) in enumerate(cases)])
    a_cat = torch.cat([a for a, _, _, _ in cases]).to(dt).cuda().contiguous()
    return n, k, list(counts), a_cat, b, sp, gs, want


def grouped_labels(cuts_fn, mode, n, k, ntok, table, sms):
    """Coverage labels of one single launch that hold with and without programmatic dependent
    launch (the first GEMM after a repack on a stream runs without it)."""
    got = None
    for pdl in (True, False):
        p = orc.stream_k_plan(sum(r for _, _, r in table), n, k, ntok, sms, pdl, True, cuts_fn, mode=mode,
                              tile_rows=[r for _, _, r in table], tile_groups=[g for g, _, _ in table])
        lab = orc.plan_paths(p)
        got = lab if got is None else got & lab
    return got


def grouped_coverage(pk, cuts_fn, mode, sms):
    """{label: sorted (routing, ntok)} over the single launches of every routing's calls."""
    table = {}
    for routing, (n0, k, counts) in ROUTINGS.items():
        n = mode_n(mode, n0)
        for sid, env in call_grid(pk, mode, n, k):
            form, ntok, tab = orc.grouped_launch(counts, n, k, sid, MODES[mode][1], single_env=env == "1")
            if form == "single":
                for lab in grouped_labels(cuts_fn, mode, n, k, ntok, tab, sms):
                    table.setdefault(lab, set()).add((routing, ntok))
    return {lab: sorted(v) for lab, v in table.items()}


# ------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def pk():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import petit_kernel

    assert torch.cuda.get_device_capability()[0] == 10, "sm_100 required"
    return petit_kernel


@pytest.fixture(scope="module")
def cuts_fn():
    return stream_k_cuts_fn(ctypes.CDLL(LIB_PATH))


@pytest.fixture(autouse=True)
def workspace_ok(pk):
    yield
    assert pk.ops.workspace_status() == 0, "a stream-K reducer timed out"


# ------------------------------------------------------------------ routings x solutions x modes
@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_grouped_single_launches_cover_every_path(pk, cuts_fn, mode):
    """At the device's SM count, the single launches of the routings reach every
    GROUPED_REQUIRED stream-K path and grouped-table edge."""
    table = grouped_coverage(pk, cuts_fn, mode, tge.num_sms())
    print(f"\ngrouped coverage {mode}: " + "; ".join(f"{lab}: {table.get(lab, [])[:3]}" for lab in GROUPED_REQUIRED))
    assert [lab for lab in GROUPED_REQUIRED if lab not in table] == []


@pytest.mark.gpu
@pytest.mark.parametrize("routing", list(ROUTINGS))
def test_grouped_exact_all_solutions(pk, routing):
    """Every mode, solution -1 and every 16/32/64-token id with PETIT_GROUPED_SINGLE unset and 0,
    and the 128-token id: each expert's rows bit-exact against its own exact_ref, guard rows
    untouched, the launch form and token tile as oracle.grouped_launch predicts; the single
    launch and the one-by-one launches give identical bits."""
    for mode in MODES:
        n, k, counts, a_cat, b, sp, gs, want = routing_case(pk, mode, routing)
        assert torch.isfinite(want.float()).all()
        bits = run_calls(pk, mode, counts, n, k, a_cat, b, sp, gs, want, f"{mode} {routing}")
        for x in bits[1:]:
            assert torch.equal(x, bits[0]), (mode, routing)
        if routing == "all_empty":
            assert a_cat.shape[0] == 0 and want.shape[0] == 0


EDGE_COUNTS = [5, 7, 3, 9, 12, 0, 6, 4]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_grouped_range_edges(pk, mode):
    """The first token of experts 1 / 2 / 3 is a NaN / +inf / -inf row, which the partial token
    tile of the expert before loads as padding: each stays in its own row.  Expert 4 has gs = 0,
    expert 6 a negative gs, and (fp16) expert 7 a gs that overflows its outputs to +-inf; the
    other experts are unaffected."""
    fmt, dt, _ = MODES[mode]
    n, k, counts = mode_n(mode, 1040), 2048, EDGE_COUNTS
    cases = expert_cases(fmt, n, k, tuple(counts), SEED + 100)
    b, sp = pack_experts(pk, mode, cases, n, k)
    off = offsets_of(counts)
    a = torch.cat([c[0] for c in cases]).double()
    S = [c[3].copy() for c in cases]
    for g, v in ((1, float("nan")), (2, float("inf")), (3, float("-inf"))):
        a[off[g], 17 * g] = v
        S[g][0] = (a[off[g]:off[g] + 1] @ torch.from_numpy(orc.dequant_nvfp4(cases[g][1], cases[g][2]) if fmt == "nvfp4"
                   else orc.dequant_mxfp4(cases[g][1], cases[g][2])).double().t()).numpy()[0]
    gs = [expert_gs(g) for g in range(len(counts))]
    gs[4], gs[6] = 0.0, -0.83
    if dt == torch.float16:
        gs[7] = 4 * 65504.0 / float(np.abs(S[7]).max())
    want = torch.cat([orc.exact_epilogue(S[g], gs[g], dt) for g in range(len(counts))])
    wf = want.float()
    assert bool(torch.isnan(wf[off[1]]).all()) and bool(torch.isinf(wf[off[2]]).any())
    assert bool(torch.isinf(wf[off[3]]).any()) and not bool(wf[off[4]:off[5]].abs().max())
    planted = {off[1], off[2], off[3]} | (set(range(off[7], off[8])) if dt == torch.float16 else set())
    rest = [r for r in range(off[-1]) if r not in planted]
    assert bool(torch.isfinite(wf[rest]).all())
    if dt == torch.float16:
        assert bool(torch.isinf(wf[off[7]:]).any()) and bool(torch.isfinite(wf[off[7]:]).any())
    a_cat = a.to(dt).cuda().contiguous()
    run_calls(pk, mode, counts, n, k, a_cat, b, sp, gs, want, f"{mode} edges")


# ------------------------------------------------------------------ fused SiLU * mul
SILU_ROUTINGS = ((1024, 2048, [3, 0, 17, 1, 16, 5, 40]), (1536, 2048, QWEN3))


def silu_case(pk, mode, n, k, counts, seed):
    """Gate / up rows interleaved per 128-row tile (petit_utils.interleave_gate_up) before packing;
    returns the packed stacks, gs per expert and the exact GEMM outputs [tokens, n] in the
    interleaved row order."""
    from petit_kernel import petit_utils as pu

    fmt, dt, _ = MODES[mode]
    cases = expert_cases(fmt, n, k, tuple(counts), seed)
    # interleaving permutes the weight rows: the exact sums follow the same permutation
    perm = pu.interleave_gate_up(torch.arange(n)).numpy()
    il = tuple((a, q[perm], s[perm], S[:, perm]) for a, q, s, S in cases)
    b, sp = pack_experts(pk, mode, il, n, k)
    gs = [0.7 * 2.0 ** -9 * (1 + 0.013 * g) for g in range(len(counts))]  # silu's argument in its interesting range
    c = torch.cat([orc.exact_epilogue(S, gs[g], dt) for g, (_, _, _, S) in enumerate(il)])
    a_cat = torch.cat([x[0] for x in il]).to(dt).cuda().contiguous()
    return a_cat, b, sp, gs, c


def silu_of(c, dt):
    """RN16(RN16(silu(gate)) * up) of exact GEMM outputs in the interleaved row order."""
    t = c.float().view(c.shape[0], c.shape[1] // 128, 2, 64)
    return (torch.nn.functional.silu(t[:, :, 0]).to(dt).float() * t[:, :, 1]).to(dt).reshape(c.shape[0], -1)


def assert_silu_close(got, want, dt, what):
    """Within one ulp of torch's silu on the exact GEMM outputs, at least 98 % bit-equal."""
    diff = (got.cpu().float() - want.float()).abs()
    assert bool((diff <= orc.ulp16(want.float(), dt)).all()), (what, diff.max().item())
    assert (got.cpu() == want).float().mean().item() > 0.98, what


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_grouped_silu_mul(pk, cuts_fn, mode):
    """Fused SiLU(gate) * up on ragged routings whose single launches write direct stores: the
    single launch and the one-by-one launches give identical bits, within one ulp of torch's silu
    on the exact GEMM outputs."""
    fmt, dt, _ = MODES[mode]
    for n, k, counts in SILU_ROUTINGS:
        a_cat, b, sp, gs, c = silu_case(pk, mode, n, k, counts, SEED + 200)
        want = silu_of(c, dt)
        gsc = torch.tensor(gs, dtype=torch.float32, device="cuda")
        ids = sid_by_ntok(pk, mode, n, k)
        for sid in (-1, ids[16], ids[32], ids[64]):
            form, ntok, table = orc.grouped_launch(counts, n, k, sid, dt)
            assert form == "single"
            outs = []
            for env in ("1", "0"):
                buf, out = guarded_out(a_cat.shape[0], n // 2, dt)
                _, kernels = gemm_kernels(lambda: grouped(pk, mode, out, a_cat, b, sp, gsc, counts, n, k, sid, env, True))
                assert kernels == expected_kernels(pk, mode, counts, n, k, sid, env == "1"), (mode, sid, env, kernels)
                what = f"{mode} silu n={n} sol={sid & 0xFFFFFFFFFFFFFFFF:#x} single={env}"
                assert_guards(buf, what)
                assert_silu_close(out, want, dt, what)
                outs.append(out.cpu().view(torch.int16))
            assert torch.equal(outs[0], outs[1]), (mode, n, sid)
            assert "direct_store" in grouped_labels(cuts_fn, mode, n, k, ntok, table, tge.num_sms())


# ------------------------------------------------------------------ C ABI
class _Hints(ctypes.Structure):
    _fields_ = [(f, ctypes.c_int32) for f in ("a_type", "b_type", "c_type", "require_high_precision")]


class _Epilogue(ctypes.Structure):
    _fields_ = [("bias", ctypes.c_void_p), ("residual", ctypes.c_void_p), ("activation", ctypes.c_int32),
                ("weight_layout", ctypes.c_int32)]


class _Problem(ctypes.Structure):
    _fields_ = [("c", ctypes.c_void_p), ("a", ctypes.c_void_p), ("b", ctypes.c_void_p), ("scales", ctypes.c_void_p),
                ("global_scale_dev", ctypes.c_void_p), ("m", ctypes.c_uint)]


def abi_fn():
    fn = ctypes.CDLL(LIB_PATH).petit_gemm_fp4_a16_grouped
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.POINTER(_Problem), ctypes.c_uint, ctypes.c_uint, ctypes.c_uint, ctypes.POINTER(_Hints),
                   ctypes.c_uint64, ctypes.POINTER(_Epilogue), ctypes.c_void_p]
    return fn


def abi_call(problems, n, k, hints, sid, epi):
    arr = (_Problem * len(problems))(*problems)
    return abi_fn()(arr, len(problems), n, k, ctypes.byref(hints), ctypes.c_uint64(sid & 0xFFFFFFFFFFFFFFFF),
                    ctypes.byref(epi) if epi is not None else None, torch.cuda.current_stream().cuda_stream)


ABI_N, ABI_K = 1040, 2048


@pytest.mark.gpu
def test_grouped_c_abi_forms(pk):
    """Through the C ABI (NVFP4 x bf16): groups in separate tensors, listed in reverse order, go
    one by one and stay exact; empty groups with NULL pointers between contiguous live groups
    still make one launch; a bias goes one by one and is exact against exact_ref(..., bias)."""
    mode = "nv_bf16"
    fmt, dt, _ = MODES[mode]
    n, k = ABI_N, ABI_K
    hints = _Hints(5, 3, 5, 0)
    counts = [4, 0, 9, 0, 0, 6, 20]
    cases = expert_cases(fmt, n, k, tuple(counts), SEED + 300)
    b, sp = pack_experts(pk, mode, cases, n, k)
    gs = [expert_gs(g) for g in range(len(counts))]
    gsc = torch.tensor(gs, dtype=torch.float32, device="cuda")
    wants = [orc.exact_epilogue(S, gs[g], dt) for g, (_, _, _, S) in enumerate(cases)]
    live = [g for g, c in enumerate(counts) if c]

    # separate tensors, reverse order
    a_sep = {g: cases[g][0].to(dt).cuda() for g in live}
    bufs = {g: guarded_out(counts[g], n, dt) for g in live}
    probs = [_Problem(bufs[g][1].data_ptr(), a_sep[g].data_ptr(), b[g].data_ptr(), sp[g].data_ptr(),
                      gsc[g:].data_ptr(), counts[g]) for g in reversed(live)]
    rc, kernels = gemm_kernels(lambda: abi_call(probs, n, k, hints, -1, None))
    assert rc == 0
    assert kernels == [(tge.solution_ntok(pk, mode, counts[g], n, k, -1), False) for g in reversed(live)], kernels
    for g in live:
        assert_bits(bufs[g][1], wants[g], f"C ABI separate tensors expert {g}")
        assert_guards(bufs[g][0], f"C ABI separate tensors expert {g}")

    # one tensor; the empty groups carry NULL pointers
    off = offsets_of(counts)
    a_cat = torch.cat([c[0] for c in cases]).to(dt).cuda().contiguous()
    buf, out = guarded_out(off[-1], n, dt)
    esz = 2

    def contiguous_problems():
        return [_Problem(out.data_ptr() + off[g] * n * esz, a_cat.data_ptr() + off[g] * k * esz, b[g].data_ptr(),
                         sp[g].data_ptr(), gsc[g:].data_ptr(), counts[g]) if counts[g] else _Problem(None, None, None,
                                                                                                     None, None, 0)
                for g in range(len(counts))]

    rc, kernels = gemm_kernels(lambda: abi_call(contiguous_problems(), n, k, hints, -1, None))
    assert rc == 0
    assert kernels == expected_kernels(pk, mode, counts, n, k, -1) == [(32, True)], kernels
    assert_bits(out, torch.cat(wants), "C ABI NULL empty groups")
    assert_guards(buf, "C ABI NULL empty groups")

    # a bias: one by one, the bias added in fp32 before the rounding
    bias = (torch.randn(n, generator=torch.Generator().manual_seed(5)) * 300).to(dt)
    bias_d = bias.cuda()
    out.fill_(float("nan"))
    epi = _Epilogue(bias_d.data_ptr(), None, 0, 0)
    rc, kernels = gemm_kernels(lambda: abi_call(contiguous_problems(), n, k, hints, -1, epi))
    assert rc == 0
    assert kernels == expected_kernels(pk, mode, counts, n, k, -1, bias=True), kernels
    assert all(not gr for _, gr in kernels) and len(kernels) == len(live)
    want_b = torch.cat([orc.exact_epilogue(S, gs[g], dt, bias) for g, (_, _, _, S) in enumerate(cases)])
    assert_bits(out, want_b, "C ABI bias")
    assert_guards(buf, "C ABI bias")


@pytest.mark.gpu
def test_grouped_c_abi_rejects_mismatched_types(pk):
    """A bf16 solution id with fp16 activations, and an fp16-native stack with bf16 activations:
    PETIT_ERROR_KERNEL_SHAPE, nothing launched, out untouched."""
    n, k = 1024, 2048
    counts = [5, 0, 11, 3]
    off = offsets_of(counts)
    for mode, a_dt, hints, layout in (("nv_f16", torch.float16, _Hints(4, 3, 4, 0), 0),
                                      ("nv_f16n", torch.bfloat16, _Hints(5, 3, 5, 0), 1)):
        fmt = MODES[mode][0]
        cases = expert_cases(fmt, n, k, tuple(counts), SEED + 400)
        b, sp = pack_experts(pk, mode, cases, n, k)
        gsc = torch.ones(len(counts), dtype=torch.float32, device="cuda")
        a_cat = torch.cat([c[0] for c in cases]).to(a_dt).cuda().contiguous()
        buf, out = guarded_out(off[-1], n, a_dt)
        before = buf.cpu().view(torch.int16).clone()
        bf16_ids = sid_by_ntok(pk, "nv_bf16", n, k)
        sids = [bf16_ids[16], bf16_ids[64]] if mode == "nv_f16" else [-1, bf16_ids[16]]
        for sid in sids:
            for env in ("1", "0"):
                probs = [_Problem(out.data_ptr() + off[g] * n * 2, a_cat.data_ptr() + off[g] * k * 2, b[g].data_ptr(),
                                  sp[g].data_ptr(), gsc[g:].data_ptr(), counts[g]) for g in range(len(counts))]
                os.environ["PETIT_GROUPED_SINGLE"] = env
                try:
                    rc, kernels = gemm_kernels(lambda: abi_call(probs, n, k, hints, sid, _Epilogue(None, None, 0, layout)))
                finally:
                    os.environ.pop("PETIT_GROUPED_SINGLE", None)
                assert rc == 2 and kernels == [], (mode, sid, env, rc, kernels)
                assert torch.equal(buf.cpu().view(torch.int16), before), (mode, sid, env)


# ------------------------------------------------------------------ CUDA graph
GRAPH_COUNTS = [5, 0, 17, 3, 9]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_grouped_graph_replay(pk, mode):
    """One single-launch call and one one-by-one call captured in a CUDA graph, replayed after the
    activations (rows permuted and signs flipped inside each expert: still exact) and the
    per-expert gs are updated in place: both outputs equal fresh exact references."""
    fmt, dt, _ = MODES[mode]
    n, k, counts = mode_n(mode, 1040), 2048, GRAPH_COUNTS
    cases = expert_cases(fmt, n, k, tuple(counts), SEED + 500)
    b, sp = pack_experts(pk, mode, cases, n, k)
    a0 = torch.cat([c[0] for c in cases])
    S0 = np.concatenate([c[3] for c in cases])
    off = offsets_of(counts)
    a_static = a0.to(dt).cuda().contiguous()
    gs_static = torch.tensor([expert_gs(g) for g in range(len(counts))], dtype=torch.float32, device="cuda")
    assert orc.grouped_launch(counts, n, k, -1, dt)[0] == "single"
    outs = [guarded_out(off[-1], n, dt) for _ in range(2)]
    for (_, out), env in zip(outs, ("1", "0")):
        grouped(pk, mode, out, a_static, b, sp, gs_static, counts, n, k, -1, env)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for (_, out), env in zip(outs, ("1", "0")):
            grouped(pk, mode, out, a_static, b, sp, gs_static, counts, n, k, -1, env)
    for it in range(3):
        rs = np.random.RandomState(it)
        perm = np.concatenate([off[e] + rs.permutation(counts[e]) for e in range(len(counts))]).astype(np.int64)
        sign = np.where(rs.rand(off[-1]) < 0.5, -1.0, 1.0)
        gs = [expert_gs(e) * (1.0 + 0.11 * (it + 1)) * (-1 if (e + it) % 3 == 0 else 1) for e in range(len(counts))]
        a_static.copy_((a0[perm].double() * torch.from_numpy(sign)[:, None]).to(dt))
        gs_static.copy_(torch.tensor(gs, dtype=torch.float32))
        for _, out in outs:
            out.fill_(float("nan"))
        g.replay()
        torch.cuda.synchronize()
        s_new = S0[perm] * sign[:, None]
        want = torch.cat([orc.exact_epilogue(s_new[off[e]:off[e + 1]], gs[e], dt) for e in range(len(counts))])
        for (buf, out), env in zip(outs, ("1", "0")):
            assert_bits(out, want, f"{mode} graph replay {it} single={env}")
            assert_guards(buf, f"{mode} graph replay {it} single={env}")


# ------------------------------------------------------------------ MoE MLP chain
CHAIN_COUNTS = [3, 0, 5, 1, 4, 2, 6, 3]
CHAIN_HIDDEN, CHAIN_INTER, CHAIN_K1 = 4096, 512, 1024   # hidden, K1: test_gemm_exact.chain_layers' layer 1


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["nv_bf16", "mx_bf16"])
def test_grouped_moe_mlp_chain(pk, mode):
    """Dense GEMM (one-hot activations picking weights of {+-1/2, +-1, +-2}: an exact activation
    matrix, as in test_gemm_exact.chain_layers) -> grouped w13 with SiLU * mul -> grouped w2 on
    its output, on one stream under programmatic dependent launch, four times eagerly and then as
    a graph replay.  w13 is within an ulp of torch's silu on its exact outputs; w2 equals the same
    call rerun alone (after a sync, on a clone of its input) bit for bit, and elementwise_ok."""
    fmt, dt, _ = MODES[mode]
    counts = CHAIN_COUNTS
    off = offsets_of(counts)
    tokens, hidden, inter, e = off[-1], CHAIN_HIDDEN, CHAIN_INTER, len(counts)
    # dense layer: [tokens, K1] one-hot x [hidden, K1] weights of {+-1/2, +-1, +-2}
    layers = tge.chain_layers(fmt, dt, tokens)
    a1, q1, s1, gs1, n1, k1 = layers[0]
    assert (n1, k1) == (hidden, CHAIN_K1)
    st1 = torch.from_numpy(s1)
    b1, sp1 = pack(pk, mode, torch.from_numpy(q1), st1.view(torch.float8_e4m3fn) if fmt == "nvfp4" else st1, n1, k1)
    w1 = orc.dequant_nvfp4(q1, s1) if fmt == "nvfp4" else orc.dequant_mxfp4(q1, s1)
    a1 = a1.to(dt).cuda()
    c1_want = orc.exact_ref(a1, w1, 1.0, dt)
    # w13: [2 inter, hidden] per expert, gate / up interleaved; w2: [hidden, inter] per expert
    from petit_kernel import petit_utils as pu

    perm = pu.interleave_gate_up(torch.arange(2 * inter)).numpy()
    w13s, w2s, b13, s13, b2, s2 = [], [], [], [], [], []
    for g in range(e):
        _, q, s, _, w, quantum = orc.make_exact_case(fmt, dt, 16, 2 * inter, hidden, SEED + 600 + g)
        q, s_np, w = q.numpy()[perm], (s.view(torch.uint8) if fmt == "nvfp4" else s).numpy()[perm], w[perm]
        rows = slice(off[g], off[g + 1])
        if counts[g]:  # the exactness precondition, with the dense layer's output as activations
            assert float(orc.exact_magnitude_bound(c1_want[rows], torch.from_numpy(w)).max()) <= 2.0 ** 22 * quantum
        st = torch.from_numpy(s_np)
        bb, ss = pack(pk, mode, torch.from_numpy(q), st.view(torch.float8_e4m3fn) if fmt == "nvfp4" else st,
                      2 * inter, hidden)
        b13.append(bb); s13.append(ss); w13s.append(w)
        _, q, s, _, w, _ = orc.make_exact_case(fmt, dt, 16, hidden, inter, SEED + 700 + g)
        bb, ss = pack(pk, mode, q, s, hidden, inter)
        b2.append(bb); s2.append(ss); w2s.append(w)
    b13, s13, b2, s2 = torch.stack(b13), torch.stack(s13), torch.stack(b2), torch.stack(s2)
    gs13 = [0.7 * 2.0 ** -9 * (1 + 0.013 * g) for g in range(e)]
    gs2 = [0.9 + 0.021 * g for g in range(e)]
    gsc1 = torch.tensor([1.0], device="cuda")
    gsc13 = torch.tensor(gs13, dtype=torch.float32, device="cuda")
    gsc2 = torch.tensor(gs2, dtype=torch.float32, device="cuda")
    c13 = torch.cat([orc.exact_ref(c1_want[off[g]:off[g + 1]], w13s[g], gs13[g], dt) for g in range(e)])
    h_want = silu_of(c13, dt)
    for gs_list, n_, k_ in ((gs13, 2 * inter, hidden), (gs2, hidden, inter)):
        assert orc.grouped_launch(counts, n_, k_, -1, dt)[0] == "single"

    def step():
        c1 = tge.gemm(pk, mode, a1, b1, sp1, gsc1, tokens, n1, k1, -1)
        h = torch.empty((tokens, inter), dtype=dt, device="cuda")
        grouped(pk, mode, h, c1, b13, s13, gsc13, counts, 2 * inter, hidden, -1, silu=True)
        o = torch.empty((tokens, hidden), dtype=dt, device="cuda")
        grouped(pk, mode, o, h, b2, s2, gsc2, counts, hidden, inter, -1)
        return c1, h, o

    def check(c1, h, o, what):
        assert_bits(c1, c1_want, f"{what} dense")
        assert_silu_close(h, h_want, dt, f"{what} w13")
        torch.cuda.synchronize()
        h_alone = h.clone()
        torch.cuda.synchronize()
        o_alone = torch.empty_like(o)
        grouped(pk, mode, o_alone, h_alone, b2, s2, gsc2, counts, hidden, inter, -1)
        torch.cuda.synchronize()
        assert torch.equal(o.cpu().view(torch.int16), o_alone.cpu().view(torch.int16)), f"{what} w2: stale read"
        for g in range(e):
            rows = slice(off[g], off[g + 1])
            if counts[g]:
                assert orc.elementwise_ok(o[rows], h[rows], w2s[g], gs2[g], dt), (what, g)

    for it in range(4):
        outs = step()
    check(*outs, f"{mode} eager")
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gouts = step()
    for it in range(2):
        for t in gouts:
            t.fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        check(*gouts, f"{mode} graph replay {it}")
