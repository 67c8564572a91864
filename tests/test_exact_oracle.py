"""CPU tests of the exact-arithmetic oracle (oracle.make_exact_case / exact_ref /
elementwise_ok / stream_k_plan) that tests/test_gemm_exact.py relies on: the checks reject
planted kernel defects, the stream-K plan agrees with what the launcher documents, and every
case the GPU file builds meets the exactness precondition and reaches the reducer paths it is
meant to reach."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import ensure_built, orc, stream_k_cuts_fn
import test_gemm_exact as tge


@pytest.fixture(scope="module")
def cuts_fn():
    return stream_k_cuts_fn(ctypes.CDLL(ensure_built()))


def _exact_equal(c, want):
    return orc.bits_equal_pm0(c, want)


# ------------------------------------------------------------------ sensitivity
def test_exact_and_elementwise_checks_reject_planted_defects():
    """Each planted defect (the output a subtly wrong kernel would produce) must fail bit
    equality with exact_ref AND elementwise_ok.  The normwise bar max_rel_err <= 1e-2 of the
    older tests accepts the truncating rounding (0.6 %) and the wrong two-step multiply (0.7 %);
    it rejects the other three here (neighbour scale 1.9 % -- with the row's largest scale jump;
    dropped k-tile 18 %; swapped columns 64 %)."""
    dt = torch.bfloat16
    # NVFP4, K = 8192: one 16-group of one row, one k-tile of one tile, two columns, rounding
    m, n, k = 32, 144, 8192          # n-tile 1 is partial (16 rows)
    a, q, s, gs, w, quantum = orc.make_exact_case("nvfp4", dt, m, n, k, 1)
    g = float(gs)
    ad = a.double()
    want = orc.exact_ref(a, w, g, dt)
    s_exact = (ad @ torch.from_numpy(w).double().t()).numpy()
    defects = {}
    # 1. one scale taken from the neighbouring group (row 5: the group whose neighbour differs most)
    sb = s.view(torch.uint8).numpy().copy()
    sv = orc.e4m3_to_f32(sb)
    row = 5
    grp = int(np.argmax(np.abs(sv[row, :-1] - sv[row, 1:])))
    assert sb[row, grp] != sb[row, grp + 1]
    sb[row, grp] = sb[row, grp + 1]
    defects["neighbour_scale"] = orc.exact_ref(a, orc.dequant_nvfp4(q.numpy(), sb), g, dt)
    # 2. one k-tile of one (16-token x 128-row) tile dropped
    drop = ad[:16, 256 * 7:256 * 8] @ torch.from_numpy(w[:128, 256 * 7:256 * 8]).double().t()
    s2 = s_exact.copy()
    s2[:16, :128] -= drop.numpy()
    defects["dropped_k_tile"] = orc.exact_epilogue(s2, g, dt)
    # 3. two output columns of the partial n-tile swapped
    sw = want.clone()
    sw[:, [130, 131]] = sw[:, [131, 130]]
    assert not torch.equal(sw, want)
    defects["swapped_columns"] = sw
    # 4. RN16 replaced by truncation
    v32 = (s_exact.astype(np.float32) * np.float32(g)).astype(np.float32)
    defects["truncating_rn16"] = torch.from_numpy(
        (v32.view(np.uint32) >> 16).astype(np.uint16).view(np.int16)).view(torch.bfloat16)
    old_bar = {}
    for name, c in defects.items():
        assert not _exact_equal(c, want), name
        assert not orc.elementwise_ok(c, a, w, g, dt), name
        old_bar[name] = orc.max_rel_err(c, torch.from_numpy(s_exact * g)) <= 1e-2
    assert orc.elementwise_ok(want, a, w, g, dt)

    # 5. MXFP4: the per-warp two-step multiply forced on a group with e8m0 <= 125, computed
    # wrongly (second multiplier 2^(s-126) instead of 2^(s-125): those weights halved) in one
    # 32-row warp group and one 32-k chunk in which another row has e8m0 > 125
    m, n, k = 32, 128, 4096
    a, q, s, gs, w, _ = orc.make_exact_case("mxfp4", dt, m, n, k, 2)
    g = float(gs)
    want = orc.exact_ref(a, w, g, dt)
    sc = s.numpy()
    chunk = 17
    blk = sc[32:64, chunk]
    assert (blk > 125).any() and (blk <= 125).any()
    w5 = w.copy()
    rows = 32 + np.nonzero(blk <= 125)[0]
    w5[rows, 32 * chunk:32 * (chunk + 1)] *= 0.5
    c5 = orc.exact_ref(a, w5, g, dt)
    ref = (a.double() @ torch.from_numpy(w).double().t()) * g
    assert not _exact_equal(c5, want)
    assert not orc.elementwise_ok(c5, a, w, g, dt)
    old_bar["two_step"] = orc.max_rel_err(c5, ref) <= 1e-2
    assert old_bar == {"neighbour_scale": False, "dropped_k_tile": False, "swapped_columns": False,
                       "truncating_rn16": True, "two_step": True}
    assert orc.elementwise_ok(want, a, w, g, dt)


def test_elementwise_ok_accepts_fp32_accumulation_in_any_order():
    """The bound holds for a plain fp32 GEMM on general data (several summation orders), and
    is still far below the normwise bar."""
    dt = torch.bfloat16
    a, q, s, gs = orc.make_gtest_style_case(24, 256, 2048, "nvfp4", dt, seed=4)
    w = orc.dequant_nvfp4(q.numpy(), s.view(torch.uint8).numpy())
    wt = torch.from_numpy(w)
    g = 0.8
    for c in ((a.float() @ wt.t()) * g,
              sum((a.float()[:, i:i + 256] @ wt[:, i:i + 256].t()) for i in range(0, 2048, 256)) * g):
        assert orc.elementwise_ok(c.to(dt), a, w, g, dt)
    assert orc.elementwise_ok((a.float() @ wt.t() * g).to(dt), a, w, g, dt, return_excess=True) <= 1.0


# ------------------------------------------------------------------ stream-K plan facts
def test_stream_k_plan_agrees_with_the_launcher(cuts_fn):
    """Facts the launcher states in csrc/fp4_gemm.cu (launch_variant / launch_mode)."""
    # TP-8 o_proj (64 tiles x 4 k-tiles on 148 SMs): one whole tile per CTA on 64 CTAs
    p = orc.stream_k_plan(16, 8192, 1024, 16, 148, True, True, cuts_fn)
    assert p["whole_tiles"] and p["grid"] == 64 and not p["tilt"]
    assert all(t["contributors"] == 0 for t in p["tiles"])
    assert not orc.stream_k_plan(16, 8192, 1024, 16, 148, True, True, cuts_fn, whole_tiles_rule=False)["whole_tiles"]
    # cuts are tilted only from 8 units per CTA on: 37 n-tiles x 32 k-tiles = 1184 = 8 x 148
    for n, tilt in ((37 * 128, True), (36 * 128, False)):
        for pdl in (True, False):
            p = orc.stream_k_plan(16, n, 8192, 16, 148, pdl, True, cuts_fn)
            assert p["tilt"] == tilt and (p["units"] >= 8 * p["grid"]) == tilt
            equal = [p["units"] * b // p["grid"] for b in range(p["grid"] + 1)]
            assert (p["cuts"] != equal) == tilt
            # the arrival term only exists under programmatic dependent launch
            assert p["late"] == (4 if (tilt and pdl) else 0) and p["lat"] == (5 if tilt else 0)
    on = orc.stream_k_plan(16, 37 * 128, 8192, 16, 148, True, True, cuts_fn)
    off = orc.stream_k_plan(16, 37 * 128, 8192, 16, 148, False, True, cuts_fn)
    assert on["cuts"] != off["cuts"] and off["cuts"] == cuts_fn(off["units"], 32, 148, 5, 0)
    # 64-token tiles: lat 3 / late 3
    p = orc.stream_k_plan(64, 37 * 128 * 4, 8192, 64, 148, True, True, cuts_fn)
    assert p["tilt"] and (p["lat"], p["late"]) == (3, 3)
    # 2-CTA clusters: prefill tiles, an even number of full n-tiles; grid = 2 x clusters
    p = orc.stream_k_plan(256, 1024, 2048, 128, 148, True, True, cuts_fn)
    assert p["cluster"] and p["grid"] == 2 * p["sched_grid"] and p["sched_grid"] <= 74 and not p["tilt"]
    for n in (1152, 1040):
        assert not orc.stream_k_plan(256, n, 2048, 128, 148, True, True, cuts_fn)["cluster"]
    assert not orc.stream_k_plan(256, 1024, 2048, 128, 148, True, False, cuts_fn)["cluster"]
    assert not orc.stream_k_plan(256, 1024, 2048, 64, 148, True, True, cuts_fn)["cluster"]
    # kRingFit from Cfg: the stage ring holds this many partial tiles of the token tile
    assert [orc.ring_fit("nv_bf16", t) for t in (16, 32, 64, 128, 256)] == [19, 12, 6, 3, 1]
    assert orc.ring_fit("mx_bf16", 16) == 18
    # n = 128, k = 28672, m = 64 on 64-token tiles: one tile, 112 CTAs, L2 tail
    p = orc.stream_k_plan(64, 128, 28672, 64, 148, True, True, cuts_fn)
    (t,) = p["tiles"]
    assert p["grid"] == 112 and t["contributors"] == 111 and t["m_valid"] == 64 and t["l2_tail"]


# ------------------------------------------------------------------ preconditions / coverage
def _all_exact_cases():
    for mode in tge.MODES:
        fmt, dt, _ = tge.MODES[mode]
        for shape in tge.DENSE_SHAPES:
            yield fmt, dt, tge.mode_shape(mode, *shape), tge.SEED
    for mode, m, n, k in tge.INVARIANCE_CASES:
        yield tge.MODES[mode][0], tge.MODES[mode][1], (m, n, k), 21


@pytest.mark.parametrize("fmt,dt,shape,seed", list(dict.fromkeys(_all_exact_cases())))
def test_exact_cases_meet_the_precondition(fmt, dt, shape, seed):
    """Every dense exact case of the GPU file: T = |a| @ |w|^T <= 2^22 q, S exact in fp32,
    MXFP4 scales straddle the two-step threshold in every 32-row warp group."""
    m, n, k = shape
    a, q, s, gs, w, quantum = orc.make_exact_case(fmt, dt, m, n, k, seed)
    t = orc.exact_magnitude_bound(a, torch.from_numpy(w))
    assert float(t.max()) <= 2.0 ** orc.EXACT_BOUND_LOG2 * quantum
    w_q = torch.from_numpy(w).double() / quantum
    assert bool((w_q * 4 == torch.round(w_q * 4)).all())  # |a| >= 1/2: products are multiples of q
    orc.exact_ref(a, w, gs.item(), dt)  # asserts S is exact in fp32
    if fmt == "mxfp4" and n >= 32:
        blocks = s.numpy()[: n // 32 * 32].reshape(n // 32, 32, -1)
        assert bool(((blocks > 125).any(1) & (blocks <= 125).any(1)).mean() > 0.95)


def test_chain_case_meets_the_precondition():
    for fmt, dt in (("nvfp4", torch.bfloat16), ("mxfp4", torch.bfloat16)):
        layers = tge.chain_layers(fmt, dt, 32)
        a1, q1, s1, _, _, _ = layers[0]
        w1 = orc.dequant_nvfp4(q1, s1) if fmt == "nvfp4" else orc.dequant_mxfp4(q1, s1)
        c1 = orc.exact_ref(a1.to(dt), w1, 1.0, dt)
        assert set(c1.float().unique().tolist()) <= {0.5, 1.0, 2.0, -0.5, -1.0, -2.0}
        _, q2, s2, _, _, k2 = layers[1]
        w2 = orc.dequant_nvfp4(q2, s2) if fmt == "nvfp4" else orc.dequant_mxfp4(q2, s2)
        quantum = orc.exact_quantum(fmt, np.unique(s2).tolist())
        assert float(orc.exact_magnitude_bound(c1, torch.from_numpy(w2)).max()) <= 2.0 ** 22 * quantum


def test_one_hot_probe_columns_cover_every_group_and_position():
    for fmt, group in (("nvfp4", 16), ("mxfp4", 32)):
        cols = np.concatenate([tge.probe_columns(r) for r in range(4)])
        assert set((cols // group).tolist()) == set(range(tge.PROBE_K // group))
        assert set((cols % 32).tolist()) == set(range(32))
        _, s = tge.probe_weights(fmt)
        if fmt == "mxfp4":
            for j in set(cols.tolist()):
                blocks = s[:, j // 32].reshape(-1, 32)
                assert bool(((blocks > 125).any(1) & (blocks <= 125).any(1)).all())


@pytest.mark.parametrize("mode", list(tge.MODES))
def test_dense_shapes_cover_every_reducer_path(cuts_fn, mode):
    """The GPU file's coverage assertion, at the B200's 148 SMs: a shape edit that drops a
    reducer path fails here already."""
    import petit_kernel

    table = tge.coverage_table(petit_kernel, cuts_fn, mode, 148)
    assert [lab for lab in tge.REQUIRED_PATHS if lab not in table] == []
    ntoks = {lab: {t for _, t in v} for lab, v in table.items()}
    for lab in ("reg_1_3", "ring", "l2_tail"):
        assert len(ntoks[lab]) >= 2, (lab, ntoks[lab])


# ------------------------------------------------------------------ fused all-reduce
def test_all_reduce_plan_agrees_with_the_launcher(cuts_fn):
    """launch_mode with ar_world > 1: launch_variant<..., CL = false, AR = true> for 16/32/64-token
    tiles only (m <= 64), never a cluster, no arrival term in the tilt (late = 0); the grid,
    whole-tile rule and lat are those of the plain decode launch."""
    for ntok in (128, 256):
        with pytest.raises(AssertionError):
            orc.stream_k_plan(16, 1024, 2048, ntok, 148, True, True, cuts_fn, all_reduce=True)
    with pytest.raises(AssertionError):
        orc.stream_k_plan(65, 1024, 2048, 64, 148, True, True, cuts_fn, all_reduce=True)
    # tilted shape (37 n-tiles x 32 k-tiles): same lat, late 0 even under PDL, so the cuts equal
    # those of a plain launch without PDL
    ar = orc.stream_k_plan(16, 37 * 128, 8192, 16, 148, True, True, cuts_fn, all_reduce=True)
    plain_nopdl = orc.stream_k_plan(16, 37 * 128, 8192, 16, 148, False, True, cuts_fn)
    plain_pdl = orc.stream_k_plan(16, 37 * 128, 8192, 16, 148, True, True, cuts_fn)
    assert ar["tilt"] and (ar["lat"], ar["late"]) == (5, 0) and plain_pdl["late"] == 4
    assert ar["cuts"] == plain_nopdl["cuts"] != plain_pdl["cuts"]
    # TP-8 o_proj: whole tiles under the all-reduce too; no cluster even where the plain launch has one
    p = orc.stream_k_plan(16, 8192, 1024, 16, 148, True, True, cuts_fn, all_reduce=True)
    assert p["whole_tiles"] and p["grid"] == 64 and not p["cluster"]
    # small shards: one k-tile per CTA, grid = units, contributors = k_tiles - 1
    p = orc.stream_k_plan(64, 144, 2048, 64, 148, True, True, cuts_fn, all_reduce=True)
    assert p["grid"] == p["units"] == 16 and [t["contributors"] for t in p["tiles"]] == [7, 7]


def test_rank_order_sum_rejects_planted_defects():
    """rank_order_sum is the fp32 sum from +0.0f in rank order of the 16-bit partials, then RN16.
    Three planted defects change bits: ranks added in reverse order, the sum formed in fp64, and
    partials summed before their rounding to 16 bits.  The 1e-2 normwise bar accepts all three;
    elementwise_ok, with the partials as the inputs of the sum, accepts the first two.  Order-
    sensitive columns: bf16 (+2^25, +1, -2^25) sums to 0 in rank order and to 1 in fp64;
    (+2^25, -2^25, +1) to 1 in rank order and to 0 reversed (fp16: 32768 and 2^-10)."""
    for dt, big, tiny in ((torch.bfloat16, 2.0 ** 25, 1.0), (torch.float16, 32768.0, 2.0 ** -10)):
        rs = np.random.RandomState(3)
        raw = (rs.randn(3, 8, 64) * 100).astype(np.float32)   # per-rank fp32 partials, 3 ranks
        raw[:, :, 0] = np.array([big, tiny, -big], dtype=np.float32)[:, None]
        raw[:, :, 1] = np.array([big, -big, tiny], dtype=np.float32)[:, None]
        parts = [torch.from_numpy(x).to(dt) for x in raw]
        want = orc.rank_order_sum(parts, dt)
        assert want[:, 0].float().eq(0).all() and want[:, 1].float().eq(tiny).all()
        f64 = sum(p.double() for p in parts)
        defects = {
            "reversed": orc.rank_order_sum(parts[::-1], dt),
            "fp64_sum": f64.to(dt),
            "unrounded_partials": orc.rn16(raw.sum(0, dtype=np.float32), dt),
        }
        assert defects["reversed"][:, 1].float().eq(0).all() and defects["fp64_sum"][:, 0].float().eq(tiny).all()
        # the sum as a GEMM: a = the partials side by side, w = three identities
        a_full = torch.cat([p.double() for p in parts], 1)
        w = np.hstack([np.eye(64, dtype=np.float32)] * 3)
        assert orc.elementwise_ok(want, a_full, w, 1.0, dt)
        for name, c in defects.items():
            assert not orc.bits_equal_pm0(c, want), (dt, name)
            assert orc.max_rel_err(c.float(), f64.float()) <= 1e-2, (dt, name)
            assert orc.elementwise_ok(c, a_full, w, 1.0, dt) == (name != "unrounded_partials"), (dt, name)
    # the sum starts from +0.0f: -0 + -0 gives +0
    z = orc.rank_order_sum([torch.tensor([-0.0], dtype=torch.bfloat16)] * 2, torch.bfloat16)
    assert z.view(torch.int16).item() == 0


@pytest.mark.parametrize("mode", list(tge.MODES))
def test_fused_allreduce_cases_fit_and_cover_every_path(cuts_fn, mode):
    """Every emulated all-reduce case of tests/test_fused_allreduce_exact.py, at the B200's 148
    SMs: all ranks' grids fit at once (world x grid, 2 x world x grid for chained calls), every
    grid is its unit or whole-tile count without tilted cuts, and the calls of the mode reach
    every reducer path the file requires."""
    import petit_kernel
    import test_fused_allreduce_exact as tfa

    for case in tfa.all_cases(petit_kernel, mode):
        tfa.check_budget(petit_kernel, cuts_fn, mode, case, tfa.AR_SMS)
    table = tfa.coverage(petit_kernel, cuts_fn, mode)
    assert [lab for lab in tfa.AR_REQUIRED if lab not in table] == []
    worlds = {w for w, *_ in tfa.sequence_cases(petit_kernel, mode)}
    assert worlds == set(range(2, 9))
    ntoks = {tge.solution_ntok(petit_kernel, mode, 64, n, k, sid) for _, sid, n, k, _ in tfa.sequence_cases(petit_kernel, mode)}
    assert ntoks == {16, 32, 64}
    # partial n-tiles of both kinds, and m values that change on every call
    rems = {n % 128 for _, _, n, _, _ in tfa.sequence_cases(petit_kernel, mode)}
    assert rems == ({32, 96} if mode in ("mx_bf16", "nv_f16n") else {16, 112})
    assert all(x != y for x, y in zip(tfa.SEQ_M, tfa.SEQ_M[1:])) and set(tfa.SEQ_M) == {1, 5, 16, 17, 33, 48, 64}
