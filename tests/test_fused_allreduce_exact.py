"""Bit-exact tests of the row-parallel GEMM fused with its all-reduce (csrc/fp4_gemm.cu, "fused
all-reduce"; petit_tp.FusedAllReduce), with every world size 2..8 emulated on one GPU.

Emulation: rank r is a stream of its own (hence its own stream-K workspace) with its own zeroed
receive buffer and `state` words; every rank gets the same list of receive-buffer pointers, so
the packets travel through device memory instead of NVLink and the protocol -- {data, epoch}
packets, two buffer parities, slots per (n-tile, 16-token group), one-shot and two-shot paths,
the rank-ordered fp32 sum -- runs as it does across GPUs.  All ranks' grids must be resident at
once (a rank spins until its peers' packets arrive), so every case asserts its co-residency
budget from oracle.stream_k_plan(all_reduce=True) before it launches.

Data: oracle.make_exact_case sharded along K (petit_tp.row_shard / row_shard_activation), so
each rank's partial P_r is oracle.exact_ref of its shard bit for bit; the output must equal
oracle.rank_order_sum(P_0 .. P_world-1) bit for bit, on every rank.  Inputs change on every
call and m changes between calls, so a packet left over from an earlier call, a slot of the
wrong 16-token group or a skipped peer changes bits.

Run as a script (``python tests/test_fused_allreduce_exact.py OUT_DIR``) it runs every call
sequence, checks it and writes the output bits to OUT_DIR; the one-shot / two-shot test does
that in fresh processes, because PETIT_AR_TWO_SHOT is read once per process."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import LIB_PATH, ROOT, orc, stream_k_cuts_fn
import petit_tp  # noqa: E402  (helpers put the package directory on sys.path)
import test_gemm_exact as tge

# The cases are sized for the B200's 148 SMs; a device with fewer skips them.
AR_SMS = 148
MAX_WORLD = 8
# m of the successive calls of a sequence: every m the tests use, changing on every call
SEQ_M = (64, 16, 33, 1, 48, 5, 17, 64)
GRAPH_M = (33, 16)      # the two calls captured in a CUDA graph
GRAPH_REPLAYS = 3
# every row must be reached by at least one call of every mode
AR_REQUIRED = ("whole_tiles", "unsplit", "reg_1_3", "ring", "many_m_le16", "many_m_gt16", "l2_tail",
               "split_partial_n", "split_partial_m")
SLEEP_CYCLES = 2_000_000  # ~1 ms at the B200's clocks
SEED = 41


def ar_n(mode, n):
    """MXFP4 scales and the fp16-native layout's shape tag need n % 32 == 0: partial n-tiles
    of 32 / 96 rows stand in for 16 / 112 there."""
    if (mode == "mx_bf16" or tge.MODES[mode][2]) and n % 32:
        n = n + 16 if n % 128 == 16 else n - 16
    return n


def ar_budget(world, chained, sms=AR_SMS):
    """Largest grid per rank with every rank's grid resident.  Calls chained without a host sync
    need room for two grids per rank: the kernel triggers programmatic dependent launch at entry,
    so a rank's next grid is resident while the current one runs."""
    return sms // ((2 if chained else 1) * world)


def ar_shape(mode, world, ntok):
    """(n, k per rank) of the call sequences at `world` with `ntok`-token tiles.  The grid of a
    decode GEMM this small is its unit count (one k-tile per CTA), so a tile of k_tiles k-tiles
    has k_tiles - 1 contributors: k_tiles picks the reducer path (2-4: registers, 5 ..
    ring_fit + 1: the stage ring, beyond: many contributors), capped by the budget at m = 64.
    Even worlds use two n-tiles, odd ones one; the last n-tile is partial."""
    n_tiles = 2 if world % 2 == 0 else 1
    rem = 16 if world in (2, 3, 6, 7) else 112
    k_tiles = min(ar_budget(world, True) // ((64 // ntok) * n_tiles), {16: 6, 32: 9, 64: 8}[ntok])
    return ar_n(mode, (n_tiles - 1) * 128 + rem), 256 * k_tiles


def sequence_cases(pk, mode):
    """[(world, sid, n, k per rank, ms)]: every world, every solution with a 16-, 32- or 64-token
    tile and -1 (sized like the 16-token case: it fits whatever tile the chooser takes)."""
    out = []
    for world in range(2, MAX_WORLD + 1):
        probe_n, probe_k = ar_shape(mode, world, 16)
        for sid in tge.solutions(pk, mode, 64, probe_n, probe_k):
            ntok = 16 if sid == -1 else tge.solution_ntok(pk, mode, 64, probe_n, probe_k, sid)
            if ntok > 64:
                continue
            n, k = ar_shape(mode, world, ntok)
            out.append((world, sid, n, k, SEQ_M))
    # one whole tile per CTA (tiles in [sms / 3, sms], <= 6 k-tiles): a single call at world 2
    n = ar_n(mode, 12 * 128 + 112)
    out.append((2, sid_with_ntok(pk, mode, n, 512, 16), n, 512, (64,)))
    return out


def sid_with_ntok(pk, mode, n, k, ntok):
    return next(s for s in tge.solutions(pk, mode, 64, n, k) if s != -1 and tge.solution_ntok(pk, mode, 64, n, k, s) == ntok)


EDGE_WORLDS, GRAPH_WORLDS, EPOCH_WORLDS, ABI_WORLDS = (3, 4, 8), (2, 5, 8), (2, 8), (2, 3)


def edge_case(mode, world):
    return (world, -1, ar_n(mode, 144), 512, (16,) * 6)


def graph_case(pk, mode, world):
    n, ks = ar_shape(mode, world, 16)
    return (world, sid_with_ntok(pk, mode, n, ks, 32), n, ks, GRAPH_M)


def epoch_case(pk, world):
    return (world, sid_with_ntok(pk, "nv_bf16", 128, 256, 16), 128, 256, (16, 16, 64))


def abi_case(world):
    return (world, -1, ar_shape("nv_bf16", world, 16)[0], 512, (33,))


def all_cases(pk, mode):
    """Every (world, sid, n, k per rank, ms) the GPU tests of `mode` launch."""
    out = sequence_cases(pk, mode) + [edge_case(mode, w) for w in EDGE_WORLDS]
    out += [graph_case(pk, mode, w) for w in GRAPH_WORLDS]
    if mode == "nv_bf16":
        out += [epoch_case(pk, w) for w in EPOCH_WORLDS] + [abi_case(w) for w in ABI_WORLDS]
    return out


def call_plans(pk, cuts_fn, mode, case, sms=AR_SMS):
    """stream_k_plan of every call of a case (the launcher's rules for a fused all-reduce)."""
    world, sid, n, k, ms = case
    return [orc.stream_k_plan(m, n, k, tge.solution_ntok(pk, mode, m, n, k, sid), sms, True, True,
                              cuts_fn, mode=mode, all_reduce=True) for m in ms]


def check_budget(pk, cuts_fn, mode, case, sms):
    """Co-residency: world x grid <= SMs for a single call, 2 x world x grid for a chain.  Also
    every grid is its unit count or its whole-tile count, without tilted cuts -- so a rank's
    partial is the plain GEMM of its shard under the same stream-K plan."""
    world, _, _, _, ms = case
    for p in call_plans(pk, cuts_fn, mode, case, sms):
        assert not p["tilt"] and p["grid"] == (len(p["tiles"]) if p["whole_tiles"] else p["units"]), case
        assert p["grid"] <= ar_budget(world, len(ms) > 1, sms), (case, p["grid"])


def coverage(pk, cuts_fn, mode, sms=AR_SMS):
    """{label: sorted (world, ntok)} over every call of sequence_cases."""
    table = {}
    for case in sequence_cases(pk, mode):
        world, sid, n, k, ms = case
        for m in ms:
            ntok = tge.solution_ntok(pk, mode, m, n, k, sid)
            for lab in tge.plan_labels(cuts_fn, mode, m, n, k, ntok, sms, all_reduce=True):
                table.setdefault(lab, set()).add((world, ntok))
    return {lab: sorted(v) for lab, v in table.items()}


# ------------------------------------------------------------------ emulation harness
class Ranks:
    """`world` emulated ranks on the current device: a stream, a zeroed receive buffer and zeroed
    state words each; `ptrs` is the receive-buffer list every rank gets."""

    def __init__(self, pk, streams, world, n):
        self.pk, self.world = pk, world
        self.streams = streams[:world]
        nbytes = pk.ops.fused_allreduce_recv_bytes(n)
        self.recv = [torch.zeros(nbytes, dtype=torch.uint8, device="cuda") for _ in range(world)]
        self.state = [torch.zeros(pk.ops.fused_allreduce_state_bytes() // 4, dtype=torch.int32, device="cuda")
                      for _ in range(world)]
        self.ptrs = [t.data_ptr() for t in self.recv]
        torch.cuda.synchronize()

    def launch(self, r, out, a, b, sp, gsc, n, k, sid, mx, sleep=False):
        with torch.cuda.stream(self.streams[r]):
            if sleep:
                torch.cuda._sleep(SLEEP_CYCLES)
            self.pk.ops.mul_fp4_a16_allreduce_out(out, a, b, sp, gsc, a.shape[0], n, k, sid, mx,
                                                  self.ptrs, self.state[r], r)

    def assert_status_ok(self, what):
        torch.cuda.synchronize()
        st = [int(self.pk.ops.fused_allreduce_status(s)) for s in self.state]
        assert st == [0] * self.world, (what, "watchdog fired", st)


def shard_case(pk, mode, world, a, q, s, w, n, k_total):
    """Per-rank (activations on the device, packed b, processed scales, dequantised w)."""
    ks = k_total // world
    out = []
    for r in range(world):
        qr, sr = petit_tp.row_shard(q, s, world, r)
        b, sp = tge.pack(pk, mode, qr, sr, n, ks)
        if tge.MODES[mode][2]:
            assert tuple(b.shape) == (n // 32, 4 * ks), "not the fp16-native layout"
        out.append((petit_tp.row_shard_activation(a, world, r).cuda(), b, sp,
                    np.ascontiguousarray(w[:, r * ks:(r + 1) * ks])))
    return out


def expected(shards, rows, gs, dt):
    """(P_r of every rank, rank_order_sum of them) for activation rows `rows`."""
    parts = [orc.exact_ref(a[rows].cpu(), w, gs, dt) for a, _, _, w in shards]
    return parts, orc.rank_order_sum(parts, dt)


def run_sequence(pk, streams, mode, world, sid, n, ks, shards, gs, ms, what, check_partials=True):
    """Every rank makes len(ms) calls back to back on its stream (no host sync in between), call
    i on activation rows [sum(ms[:i]), sum(ms[:i + 1])): each output must be rank_order_sum of
    the exact partials, on every rank.  Returns the output bits of rank 0."""
    fmt, dt, _ = tge.MODES[mode]
    mx = fmt == "mxfp4"
    gsc = torch.tensor([gs], dtype=torch.float32, device="cuda")
    bounds = np.concatenate([[0], np.cumsum(ms)]).tolist()
    wants = []
    for i, m in enumerate(ms):
        parts, want = expected(shards, slice(bounds[i], bounds[i + 1]), gs, dt)
        wants.append(want)
        if check_partials and i < 2:  # P_r is the plain GEMM of the shard (same stream-K plan)
            for r, (a, b, sp, _) in enumerate(shards):
                got = tge.gemm(pk, mode, a[bounds[i]:bounds[i + 1]], b, sp, gsc, m, n, ks, sid)
                tge.assert_bits(got, parts[r], f"{what} plain GEMM of shard {r}, call {i}")
    ranks = Ranks(pk, streams, world, n)
    outs = [[torch.full((m, n), float("nan"), dtype=dt, device="cuda") for m in ms] for _ in range(world)]
    for i, m in enumerate(ms):
        for r, (a, b, sp, _) in enumerate(shards):
            ranks.launch(r, outs[r][i], a[bounds[i]:bounds[i + 1]], b, sp, gsc, n, ks, sid, mx)
    ranks.assert_status_ok(what)
    for i in range(len(ms)):
        for r in range(world):
            tge.assert_bits(outs[r][i], wants[i], f"{what} call {i} (m={ms[i]}) rank {r}")
    return [o.cpu().view(torch.int16).numpy() for o in outs[0]]


def sequence_data(pk, mode, world, n, ks, ms, seed):
    fmt, dt, _ = tge.MODES[mode]
    a, q, s, gs, w, _ = orc.make_exact_case(fmt, dt, sum(ms), n, ks * world, seed)
    return shard_case(pk, mode, world, a, q, s, w, n, ks * world), gs.item()


EDGE_GS = 4.0


def tiny_of(dt):
    return 0.25 if dt == torch.bfloat16 else 2.0 ** -12


def edge_data(pk, mode, world, shift):
    """Range edges with uniform weights 1 and gs = 4, so that P_r[row, :] is RN16 of 4 x the row
    sum of rank r's activations (rows 0-4 below, the rest random exact values; the values quoted
    are the partials).  gs = 4 keeps every fp32 sum inside the MMA below the fp32 maximum: the
    MXFP4 A operand holds 4 w, so partials near 2^127 would overflow there.
      0: order probe on ranks 0, 1, 2: bf16 +2^25, +1, -2^25 / fp16 32768, 2^-10, -32768 -- the
         rank-order fp32 sum is 0, every other order gives the small value;
      1: +inf on rank 0 and -inf on rank 1 (each partial overflows the 16-bit range): NaN;
      2: finite partials whose fp32 sum overflows only when it is rounded to 16 bits: +inf;
      3: +inf on rank 0 only, finite elsewhere;
      4: the order probe as +big, -big, +small: the small value in rank order, 0 reversed.
    `shift` rolls the rows so that the data changes from call to call."""
    fmt, dt, _ = tge.MODES[mode]
    _, _, n, ks, _ = edge_case(mode, world)
    m = 16
    q, s = tge.uniform_weights(fmt, n, ks * world, 0x2, 0x38 if fmt == "nvfp4" else 127)  # 1.0
    rs = np.random.RandomState(shift)
    a = orc.EXACT_ACTS[rs.randint(0, 6, size=(m, ks * world))].astype(np.float64)
    a[:5] = 0
    col = lambda r, j=0: r * ks + 37 * r + j  # noqa: E731  (a column of rank r's shard)
    if dt == torch.bfloat16:
        big, tiny, f = 2.0 ** 23, tiny_of(dt), 2.0 ** 125
        inf_pair = (1.9921875 * f, 1.0078125 * 2.0 ** 117)        # x 4: above bf16's rounding edge
        late = (1.5 * f, 0.498046875 * f)                         # x 4: 1.998046875 * 2^127 in fp32
    else:
        big, tiny = 8192.0, tiny_of(dt)
        inf_pair = (8192.0, 8192.0)                               # x 4: 65536
        late = (15000.0, 1500.0)                                  # x 4: 60000 + 6000 = 66000
    for r, v in enumerate((big, tiny, -big)):
        a[0, col(r)] = v
    a[1, col(0)], a[1, col(0, 1)] = inf_pair
    a[1, col(1)], a[1, col(1, 1)] = -inf_pair[0], -inf_pair[1]
    a[2, col(0)], a[2, col(1)] = late
    a[3, col(0)], a[3, col(0, 1)] = inf_pair
    a[3, col(2)] = -250.0
    for r, v in enumerate((big, -big, tiny)):
        a[4, col(r)] = v
    a = torch.from_numpy(np.roll(a, shift, axis=0)).to(dt)
    w = orc.dequant_nvfp4(q, s) if fmt == "nvfp4" else orc.dequant_mxfp4(q, s)
    st = torch.from_numpy(s)
    shards = shard_case(pk, mode, world, a, torch.from_numpy(q),
                        st.view(torch.float8_e4m3fn) if fmt == "nvfp4" else st, w, n, ks * world)
    return shards, n, ks


def run_edges(pk, streams, mode, world, ncalls=6):
    """ncalls calls of the range-edge rows (rolled differently on every call), one sequence."""
    fmt, dt, _ = tge.MODES[mode]
    parts = [edge_data(pk, mode, world, shift) for shift in range(ncalls)]
    n, ks = parts[0][1], parts[0][2]
    # the calls of one sequence take consecutive row blocks of one activation tensor per rank
    shards = [(torch.cat([p[0][r][0] for p in parts]), *parts[0][0][r][1:]) for r in range(world)]
    for p in parts:
        for r in range(world):
            assert np.array_equal(p[0][r][3], shards[r][3])
    ms = (16,) * ncalls
    bits = run_sequence(pk, streams, mode, world, -1, n, ks, shards, EDGE_GS, ms, f"{mode} edges world={world}")
    want = [expected(shards, slice(16 * i, 16 * (i + 1)), EDGE_GS, dt)[1] for i in range(ncalls)]
    # the planted edges really are there: NaN, +inf from a late overflow, order-sensitive zero
    w0 = want[0].float()
    assert bool(torch.isnan(w0[1]).all()) and bool(torch.isposinf(w0[2]).all()) and bool(torch.isposinf(w0[3]).all())
    assert bool((w0[0] == 0).all()) and bool((w0[4] == 4 * tiny_of(dt)).all())
    return bits


def all_sequences(pk, streams, modes):
    """{name: output bits} of every call sequence and range-edge sequence of `modes`."""
    res = {}
    for mode in modes:
        for case in sequence_cases(pk, mode):
            world, sid, n, ks, ms = case
            shards, gs = sequence_data(pk, mode, world, n, ks, ms, SEED + world)
            name = f"{mode}_w{world}_{sid & 0xFFFFFFFFFFFFFFFF:x}_{len(ms)}"
            for i, b in enumerate(run_sequence(pk, streams, mode, world, sid, n, ks, shards, gs, ms, name)):
                res[f"{name}_{i}"] = b
        for world in EDGE_WORLDS:
            for i, b in enumerate(run_edges(pk, streams, mode, world)):
                res[f"{mode}_edges_w{world}_{i}"] = b
    return res


def rank_streams(pk):
    """One stream per emulated rank.  A plain GEMM on each creates the stream's stream-K
    workspace now, and a first torch.cuda._sleep loads its module now: neither the allocation
    nor a lazy module load may happen while other ranks' grids wait for packets (a module load
    can wait for the device to go idle)."""
    streams = [torch.cuda.Stream() for _ in range(MAX_WORLD)]
    a, q, s, gs, _, _ = orc.make_exact_case("nvfp4", torch.bfloat16, 16, 128, 256, 0)
    b, sp = tge.pack(pk, "nv_bf16", q, s, 128, 256)
    a, gs = a.cuda(), gs.cuda()
    torch.cuda.synchronize()
    for st in streams:
        with torch.cuda.stream(st):
            tge.gemm(pk, "nv_bf16", a, b, sp, gs, 16, 128, 256, -1)
            torch.cuda._sleep(1000)
    torch.cuda.synchronize()
    return streams


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


@pytest.fixture(scope="module")
def streams(pk):
    """Shared by every test: the library keeps one stream-K workspace per stream."""
    return rank_streams(pk)


@pytest.fixture(scope="module")
def sms():
    got = torch.cuda.get_device_properties(0).multi_processor_count
    if got < AR_SMS:
        pytest.skip(f"the emulated ranks' grids are sized for {AR_SMS} co-resident CTAs; this device has {got} SMs")
    return got


# ------------------------------------------------------------------ tests
@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(tge.MODES))
def test_fused_allreduce_sequences_bit_exact(pk, cuts_fn, streams, sms, mode):
    """Worlds 2..8, every 16/32/64-token solution and -1, m changing on every call (64, 16, 33,
    1, 48, 5, 17, 64) with new inputs every call and no host sync: bit-exact rank_order_sum on
    every rank, status 0.  The calls reach every AR_REQUIRED reducer path."""
    table = coverage(pk, cuts_fn, mode, AR_SMS)
    print(f"\nfused all-reduce coverage {mode}: " + "; ".join(
        f"{lab}: {table.get(lab, [])}" for lab in AR_REQUIRED))
    missing = [lab for lab in AR_REQUIRED if lab not in table]
    assert not missing, f"{mode}: no call reaches {missing}"
    for case in all_cases(pk, mode):
        check_budget(pk, cuts_fn, mode, case, AR_SMS)
    all_sequences(pk, streams, [mode])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["nv_bf16", "nv_f16n", "mx_bf16"])
def test_fused_allreduce_graph_replay(pk, cuts_fn, streams, sms, mode):
    """Two calls per rank captured in a CUDA graph, replayed three times with the inputs updated
    in place in between: every replay bit-exact (the epoch in `state` advances inside the
    graph, so replays alternate the buffer parities like eager calls)."""
    fmt, dt, _ = tge.MODES[mode]
    mx = fmt == "mxfp4"
    for world in GRAPH_WORLDS:
        case = graph_case(pk, mode, world)
        check_budget(pk, cuts_fn, mode, case, AR_SMS)
        _, sid, n, ks, _ = case
        rows = sum(GRAPH_M)
        shards, gs = sequence_data(pk, mode, world, n, ks, GRAPH_M * (GRAPH_REPLAYS + 1), 300 + world)
        block = lambda it, lo, hi: slice(it * rows + lo, it * rows + hi)  # noqa: E731
        static = [sh[0][block(0, 0, rows)].clone() for sh in shards]  # per-rank graph inputs
        gsc = torch.tensor([gs], dtype=torch.float32, device="cuda")
        ranks = Ranks(pk, streams, world, n)
        bounds = np.concatenate([[0], np.cumsum(GRAPH_M)]).tolist()
        outs = [[torch.empty((m, n), dtype=dt, device="cuda") for m in GRAPH_M] for _ in range(world)]

        def calls(r):
            _, b, sp, _ = shards[r]
            for i, m in enumerate(GRAPH_M):
                ranks.launch(r, outs[r][i], static[r][bounds[i]:bounds[i + 1]], b, sp, gsc, n, ks, sid, mx)

        # one eager round first (every rank at once), then capture rank by rank
        for r in range(world):
            calls(r)
        ranks.assert_status_ok(f"{mode} world={world} eager")
        graphs = []
        for r in range(world):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=ranks.streams[r]):
                calls(r)
            graphs.append(g)
        torch.cuda.synchronize()
        for it in range(1, GRAPH_REPLAYS + 1):
            for r in range(world):
                static[r].copy_(shards[r][0][block(it, 0, rows)])
                for o in outs[r]:
                    o.fill_(float("nan"))
            torch.cuda.synchronize()
            for r in range(world):
                with torch.cuda.stream(ranks.streams[r]):
                    graphs[r].replay()
            ranks.assert_status_ok(f"{mode} world={world} replay {it}")
            for i in range(len(GRAPH_M)):
                want = expected(shards, block(it, bounds[i], bounds[i + 1]), gs, dt)[1]
                for r in range(world):
                    tge.assert_bits(outs[r][i], want, f"{mode} world={world} replay {it} call {i} rank {r}")


@pytest.mark.gpu
def test_one_shot_and_two_shot_give_the_same_bits(pk, sms, tmp_path):
    """Every sequence in fresh processes with PETIT_AR_TWO_SHOT unset, 0 and 1 (read once per
    process; worlds 2, 4 and 8 accept two-shot): each run checks its own bits against the
    reference, and the three runs agree bit for bit."""
    runs = {}
    for label, val in (("unset", None), ("one_shot", "0"), ("two_shot", "1")):
        env = {k: v for k, v in os.environ.items() if k != "PETIT_AR_TWO_SHOT"}
        if val is not None:
            env["PETIT_AR_TWO_SHOT"] = val
        out = tmp_path / label
        out.mkdir()
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "test_fused_allreduce_exact.py"), str(out)],
                           env=env, capture_output=True, text=True, timeout=1500)
        assert r.returncode == 0, (label, r.stdout[-3000:] + r.stderr[-3000:])
        runs[label] = dict(np.load(out / "bits.npz"))
    names = set(runs["unset"])
    assert names and all(set(v) == names for v in runs.values())
    for name in sorted(names):
        assert np.array_equal(runs["unset"][name], runs["one_shot"][name]), name
        assert np.array_equal(runs["unset"][name], runs["two_shot"][name]), name


@pytest.mark.gpu
@pytest.mark.parametrize("world", EPOCH_WORLDS)
def test_epoch_wrap_never_matches_zeroed_slots(pk, cuts_fn, streams, sms, world):
    """The call counter in state[0] wraps without ever giving epoch 0: a slot no call has written
    is all zero bytes, which would be a valid epoch-0 packet holding 0.  state[0] starts at
    2^32 - 3; two m = 16 calls, then an m = 64 call whose 16-token groups 1-3 are tiles (and
    CTAs) of their own and whose slots were never written.  Ranks > 0 start ~1 ms late, so a
    reader that accepted a zeroed slot would add 0 for their partials."""
    mode = "nv_bf16"
    fmt, dt, _ = tge.MODES[mode]
    case = epoch_case(pk, world)
    check_budget(pk, cuts_fn, mode, case, AR_SMS)
    _, sid, n, ks, ms = case
    p = orc.stream_k_plan(64, n, ks, 16, AR_SMS, True, True, cuts_fn, mode=mode, all_reduce=True)
    assert p["grid"] == 4 and all(t["contributors"] == 0 for t in p["tiles"])
    shards, gs = sequence_data(pk, mode, world, n, ks, ms, 77)
    gsc = torch.tensor([gs], dtype=torch.float32, device="cuda")
    ranks = Ranks(pk, streams, world, n)
    for st in ranks.state:
        st[0] = -3  # 2^32 - 3
    torch.cuda.synchronize()
    bounds = np.concatenate([[0], np.cumsum(ms)]).tolist()
    outs = [[torch.full((m, n), float("nan"), dtype=dt, device="cuda") for m in ms] for _ in range(world)]
    for i, m in enumerate(ms):
        for r, (a, b, sp, _) in enumerate(shards):
            ranks.launch(r, outs[r][i], a[bounds[i]:bounds[i + 1]], b, sp, gsc, n, ks, sid, False, sleep=r > 0)
    ranks.assert_status_ok(f"epoch wrap world={world}")
    for i in range(len(ms)):
        want = expected(shards, slice(bounds[i], bounds[i + 1]), gs, dt)[1]
        for r in range(world):
            tge.assert_bits(outs[r][i], want, f"epoch wrap world={world} call {i} (m={ms[i]}) rank {r}")
    # the counter went 2^32 - 3 -> 2^32 - 2 = the period -> 0 -> 1 -> 2
    assert [int(st[0]) for st in ranks.state] == [2] * world


class _Hints(ctypes.Structure):
    _fields_ = [(f, ctypes.c_int32) for f in ("a_type", "b_type", "c_type", "require_high_precision")]


class _Epilogue(ctypes.Structure):
    _fields_ = [("bias", ctypes.c_void_p), ("residual", ctypes.c_void_p), ("activation", ctypes.c_int32),
                ("weight_layout", ctypes.c_int32)]


class _FusedAllReduce(ctypes.Structure):
    _fields_ = [("world", ctypes.c_int32), ("rank", ctypes.c_int32), ("recv", ctypes.c_void_p * 8),
                ("state", ctypes.c_void_p)]


@pytest.mark.gpu
@pytest.mark.parametrize("world", ABI_WORLDS)
def test_c_abi_bias_and_residual_with_all_reduce(pk, cuts_fn, streams, sms, world):
    """petit_gemm_nvfp4_a16_ex with an all-reduce context and, on rank 0 only (petit.h), bias and
    a residual that aliases c: the result is rank_order_sum of rank 0's epilogue output and the
    other ranks' plain partials, bit for bit on every rank."""
    mode = "nv_bf16"
    fmt, dt, _ = tge.MODES[mode]
    case = abi_case(world)
    check_budget(pk, cuts_fn, mode, case, AR_SMS)
    _, _, n, ks, ms = case
    shards, gs = sequence_data(pk, mode, world, n, ks, ms, 91)
    m = ms[0]
    g = torch.Generator().manual_seed(world)
    bias = (torch.randn(n, generator=g) * 300).to(dt)
    resid = (torch.randn(m, n, generator=g) * 300).to(dt)
    parts = [orc.exact_ref(a.cpu(), w, gs, dt, *((bias, resid) if r == 0 else (None, None)))
             for r, (a, _, _, w) in enumerate(shards)]
    want = orc.rank_order_sum(parts, dt)
    lib = ctypes.CDLL(LIB_PATH)
    fn = lib.petit_gemm_nvfp4_a16_ex
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_uint] * 3 + [
        ctypes.POINTER(_Hints), ctypes.c_uint64, ctypes.POINTER(_Epilogue), ctypes.POINTER(_FusedAllReduce),
        ctypes.c_void_p]
    hints = _Hints(5, 3, 5, 0)  # bf16, NVFP4, bf16
    gsc = torch.tensor([gs], dtype=torch.float32, device="cuda")
    bias_d = bias.cuda()
    ranks = Ranks(pk, streams, world, n)
    outs = [resid.cuda() if r == 0 else torch.full((m, n), float("nan"), dtype=dt, device="cuda")
            for r in range(world)]
    torch.cuda.synchronize()
    keep = []
    for r, (a, b, sp, _) in enumerate(shards):
        epi = _Epilogue(bias_d.data_ptr() if r == 0 else None, outs[0].data_ptr() if r == 0 else None, 0, 0)
        ar = _FusedAllReduce(world, r, (ctypes.c_void_p * 8)(*ranks.ptrs), ranks.state[r].data_ptr())
        keep.append((epi, ar))
        rc = fn(outs[r].data_ptr(), a.data_ptr(), b.data_ptr(), sp.data_ptr(), gsc.data_ptr(), m, n, ks,
                ctypes.byref(hints), ctypes.c_uint64(-1 & 0xFFFFFFFFFFFFFFFF), ctypes.byref(epi),
                ctypes.byref(ar), ranks.streams[r].cuda_stream)
        assert rc == 0, rc
    ranks.assert_status_ok(f"C ABI world={world}")
    for r in range(world):
        tge.assert_bits(outs[r], want, f"C ABI bias + residual world={world} rank {r}")


if __name__ == "__main__":
    import petit_kernel

    bits = all_sequences(petit_kernel, rank_streams(petit_kernel), list(tge.MODES))
    np.savez(os.path.join(sys.argv[1], "bits.npz"), **bits)
