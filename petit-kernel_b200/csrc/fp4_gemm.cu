// FP4-weight x 16-bit-activation GEMM for sm_100a.
//
//   C[M,N] = A[M,K] * dequant(W[N,K])^T * global_scale
//
// Replaces the reference's GemmFp4Fp16KernelGrid + MultiStagePipeline +
// WarpPartitionMatmul + BlockReduce + WriteResult
// (lib/gemm/rocm/quantization/fp4/gemm_fp4_fp16_grid.cuh:199-498,
//  fp4/warp_schedule_fp16.cuh:10-193, gpu/quantization/reduce.cuh:7-58,
//  quantization/qgemm.cuh:95-192) with a design built for Blackwell:
//
//  * swap-AB: the 128 weight rows of an n-tile are the tcgen05.mma M dimension,
//    the tokens are the MMA N dimension (16..256), so decode-sized M wastes no
//    tensor-core rows and each weight is dequantised exactly once per tile.
//  * TS-form MMA: dequantised weights never touch shared memory.  One dequant
//    thread owns one weight row = one TMEM lane: it reads 16 bytes (32 fp4) per
//    ld.shared, converts (bit placement for the bf16-native layout, cvt.rn.f16x2.e2m1x2
//    for the fp16-native one, + HMUL2 by the block scale: dequant.cuh),
//    and writes the 16-bit pairs straight into the A-operand columns of TMEM
//    with tcgen05.st.  The MMA reads A from TMEM and the token tile (B operand)
//    from 128B-swizzled shared memory filled by TMA.
//  * weights + scales arrive through a multi-stage ring of 1-D bulk TMA copies
//    (cp.async.bulk) of contiguous packed tiles (layout.cuh).
//  * stream-K: the (n-tile x token-tile x k-tile) unit space is cut into one
//    contiguous range per SM, so all 148 SMs stream the same number of bytes
//    whatever the shape.  Tiles cut by a range boundary are reduced through an
//    fp32 workspace by the CTA that owns the tile's first k-part (a static choice: it
//    reaches the tile last, at the end of its range), in CTA order (bit-reproducible).
//    For decode tiles the ranges are not exactly equal: CTAs a reducer would wait for get
//    slightly shorter ones (tilt_cuts).
//  * warp roles: 2 TMA producers (weights / token tiles), 1 MMA issuer (2 for decode
//    tiles, each owning half of the accumulator chains), 16 dequant warps, 4 epilogue
//    warps; accumulators are double-buffered in TMEM so the epilogue overlaps the next tile.
//  * instantiations of the same kernel: CL (2-CTA cluster, token tile multicast, prefill),
//    AR (epilogue all-reduces the tile over NVLink peer memory, row-parallel TP layers),
//    GR (grouped / MoE: the token tiles of all experts in one schedule).
#include "fp4_gemm.h"
#include "dequant.cuh"
#include "layout.cuh"
#include "sm100_ptx.cuh"

#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstring>
#include <map>
#include <mutex>
#include <tuple>
#include <vector>
#include <cstddef>
#include <cstdlib>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <type_traits>

namespace petit::gemm {

using namespace petit::ptx;
using namespace petit::layout;
using namespace petit::dq;

#ifndef PETIT_DECODE_GROUPS
#define PETIT_DECODE_GROUPS 2
#endif
#ifndef PETIT_DECODE_GROUPS_NVBF16
#define PETIT_DECODE_GROUPS_NVBF16 2
#endif
// Knock-out experiments (tools/build_variant.sh <name> . -DPETIT_KO=<bits>; results are wrong on
// purpose, timing only): 1 = two MMAs per issuer and stage, 2 = no dequant arithmetic, 16 = no
// TMEM stores (arithmetic kept alive), 32 = no tcgen05.wait::st.  0 in production.
#ifndef PETIT_KO
#define PETIT_KO 0
#endif
#ifndef PETIT_PERIODIC
#define PETIT_PERIODIC 1 // decode dequant loop unrolled over its 3-iteration ring period (0: A/B)
#endif

namespace {

// Warp roles, aligned to warpgroups so setmaxnreg can rebalance registers:
//   WG0:   warp 0 = TMA producer (weights), warp 1 = MMA issuer, warp 2 = TMA producer
//          (token tiles), warp 3 = second MMA issuer for decode tiles (idle otherwise)
//   WG1:   warps 4-7  = epilogue (one per TMEM lane quarter)
//   WG2-5: warps 8-23 = dequant (4 per lane quarter -> 4 per SM sub-partition)
// (Measured: putting the two single-thread roles on the highest warp ids instead
// makes decode ~20 % slower -- their mbarrier polling then wins arbitration
// against the dequant warps.)
constexpr int kNumDequantWarps = 16;
constexpr int kNumEpilogueWarps = 4;
constexpr int kProducerWarp = 0;    // weights + scales
constexpr int kMmaWarp = 1;
constexpr int kActProducerWarp = 2; // token tiles
constexpr int kMmaWarp2 = 3;        // decode tiles: second MMA issuer (half of the accumulator chains)
constexpr int kFirstEpilogueWarp = 4;
constexpr int kFirstDequantWarp = 8;
constexpr int kNumWarps = kFirstDequantWarp + kNumDequantWarps;
constexpr int kNumThreads = kNumWarps * 32;
constexpr int kKSlices = kNumDequantWarps / 4; // dequant warps per lane quarter
// 768 threads x 80 registers = 61440 is the CTA pool setmaxnreg redistributes:
// 128 x 40 (WG0) + 128 x 88 (epilogue) + 512 x 88 (dequant / extra epilogue teams) = 61440.
constexpr int kRegsLight = 40, kRegsDequant = 88;
constexpr int kEpilogueBarId = 1;
constexpr int kSetupBarId = 2;
constexpr int kTeamBarId0 = 3; // 3, 4, 5: one named barrier per epilogue team
constexpr int kSmemBudget = 227 * 1024;

// Accumulator organisation of the 32- and 64-token tiles (experiment switches, see Cfg).
// Measured (profiles/r02_mid_m_ab.md): more chains do not help either tile (the MMAs are not
// latency-bound there); a second accumulator buffer for the 64-token tile (2 x 2 chains x 64
// columns, leaving two TMEM A stages) lets the epilogue overlap the next tile: gate_up M=64
// 71.2 -> 68.8 us, M=128 (two 64-token tiles) 141 -> 135 us, qkv M=128 30.5 -> 29.0 us;
// 128-k stages for the 64-token tile are 15 % slower.
#ifndef PETIT_NUMACC_32
#define PETIT_NUMACC_32 2
#endif
#ifndef PETIT_NUMACC_64
#define PETIT_NUMACC_64 2
#endif
#ifndef PETIT_ACC_COLS_32
#define PETIT_ACC_COLS_32 128
#endif
#ifndef PETIT_ACC_COLS_64
#define PETIT_ACC_COLS_64 256
#endif
#ifndef PETIT_KS_64
#define PETIT_KS_64 256   // k extent of a stage of the 64-token tile
#endif

template <int MODE, int NTOK, int KS> struct Cfg {
    static constexpr bool kIsMx = MODE == kModeMxBf16;
    static constexpr bool kIsBf16 = MODE == kModeNvBf16 || MODE == kModeMxBf16;
    static constexpr int kSubs = KS / 64;          // 64-k slabs per stage
    static constexpr int kStagesPerUnit = 256 / KS;
    static constexpr int kChunks = KS / 32;        // 16-byte chunks per row
    static constexpr int kScPerSub = kIsMx ? 2 : 4; // scale bytes per row per slab
    static constexpr int kActBytes = kSubs * NTOK * 128;
    static constexpr int kWBytes = kChunks * 128 * 16;
    static constexpr int kScBytes = kSubs * 128 * kScPerSub;
    static constexpr int kStageBytes =
        (kActBytes + kWBytes + kScBytes + 1023) / 1024 * 1024;
    static constexpr int kBarrierBytes = 1024;
    // epilogue staging: three [16 tokens][128 rows] 16-bit tiles feeding TMA stores
    static constexpr int kOutStageBytes = 16 * 128 * 2;
    // 256-token tiles have one accumulator, so their epilogue (16 groups) is exposed between
    // tiles (measured 8.8 of 57 us per tile): there the 8 dequant warps that prefill leaves
    // idle (kUsedSlices below) form two more epilogue teams and the groups are dealt round
    // robin to the three teams, each with its own staging buffers.
    static constexpr int kEpiTeams = NTOK >= 256 ? 3 : 1;
    // decode tiles store at most four 16-token groups per tile: two buffers are enough
    static constexpr int kOutBufs = (kEpiTeams > 1 || NTOK <= 64) ? 2 : 3; // per team
    static constexpr int kOutBytes = kEpiTeams * kOutBufs * kOutStageBytes;
    // reducer: running sum of the other CTAs' partials for the first 16 tokens,
    // [16 tokens][128 rows] fp32, each element private to one epilogue thread.  (Held in
    // registers it was spilled to local memory, and those spills miss the small L1 that is
    // left next to 227 KB of shared memory: +0.7 us on every reducer's exit path.)
    static constexpr int kPreBytes = 16 * 128 * 4;
    static constexpr int kRingBudget = kSmemBudget - kBarrierBytes - kOutBytes - kPreBytes - 1024;
    static constexpr int kStagesRaw = kRingBudget / kStageBytes > 16 ? 16 : kRingBudget / kStageBytes;
    // Decode tiles: a ring of exactly 6 stages (2 x the 3 TMEM A stages) makes the ring state of
    // a dequant group periodic with period 3 iterations, so its loop is unrolled by 3 with every
    // barrier / shared-memory / TMEM address a constant offset (kPeriodic below).  Six 18 KB
    // weight stages per SM are 16 MB in flight chip-wide, above the ~10 MB bandwidth-delay product.
    static constexpr int kStages = (NTOK <= 64 && kStagesRaw >= 6 && kStagesRaw < 12) ? 6 : kStagesRaw;
    // Small-N MMAs that accumulate into the same TMEM columns serialise on the
    // full MMA latency (~130 clk measured), so consecutive k-steps rotate over
    // kChains independent accumulators that the epilogue sums.
    // (Measured: 8 chains with a single accumulator buffer is slower than 4 chains
    // double-buffered -- the segment-boundary stall costs more than the extra chains
    // gain.)
    static constexpr int kNumAcc = NTOK == 32   ? PETIT_NUMACC_32
                                   : NTOK == 64 ? PETIT_NUMACC_64
                                                : ((NTOK <= 32 || NTOK == 128) ? 2 : 1);
    // TMEM columns of all accumulators of a decode tile (the rest holds the A stages)
    static constexpr int kDecodeAccCols = NTOK == 32 ? PETIT_ACC_COLS_32 : (NTOK == 64 ? PETIT_ACC_COLS_64 : 128);
    static constexpr int kChains = NTOK >= 128 ? 1 : kDecodeAccCols / (kNumAcc * NTOK);
    // When a stage has fewer chunks than k-slice warps (KS = 64), the warps form
    // kGroups groups that take alternate stages.
    // Prefill tiles (NTOK >= 128) are tensor-bound: only half of the dequant warps
    // work there, the rest would just compete with the MMA issuer for issue slots.
    static constexpr int kUsedSlices = NTOK >= 128 ? kKSlices / 2 : kKSlices;
    // Decode tiles (NTOK <= 64): two groups of 8 warps take alternate 256-k stages, 4 chunks
    // per thread, which halves the per-stage bookkeeping per weight (measured gate_up M=16:
    // fp16 76 -> 71 us, MXFP4 77 -> 65 us; NVFP4-bf16 was neutral while the single MMA issuer
    // was the critical path -- profiles/r01_variants_ab.log -- and gains 3 % with two issuers:
    // 53.2 -> 51.5 us, profiles/r02_decode_ab.md).
    static constexpr int kGroups =
        kUsedSlices > kChunks ? kUsedSlices / kChunks
                              : (NTOK <= 64 ? (MODE != kModeNvBf16 ? PETIT_DECODE_GROUPS
                                                                   : PETIT_DECODE_GROUPS_NVBF16)
                                            : 1);
    static constexpr int kActiveSlices = kUsedSlices / kGroups;  // k-slice warps per stage
    static constexpr int kStageWarps = 4 * kActiveSlices;        // dequant warps per stage
    static_assert(kChunks % kActiveSlices == 0, "chunks must split evenly over the k-slices");
    // Decode tiles: two MMA issuers on two SM sub-partitions, each owning half of the
    // accumulator chains.  One issuer's ~105 instructions per stage behind four dequant warps
    // of its sub-partition were the critical path of the TMEM hand-off (measured: 15 fewer
    // instructions per stage in that warp = -9 % on gate_up, profiles/r02_decode_ab.md).
    static constexpr int kMmaWarps = kChains >= 2 ? 2 : 1;
    static constexpr int kAccBufCols = kChains * NTOK;
    static constexpr int kAccCols = kNumAcc * kAccBufCols;
    static_assert(KS / 16 >= kChains, "stage must cover every accumulator chain");
    static constexpr int kACols = KS / 2;          // TMEM columns of one A stage
    static constexpr int kAStagesRaw = (512 - kAccCols) / kACols;
    static constexpr int kAStages = kAStagesRaw > 8 ? 8 : kAStagesRaw;
    static constexpr int kSmemBytes =
        kBarrierBytes + kOutBytes + kPreBytes + kStages * kStageBytes + 1024;
    static_assert(kSmemBytes <= kSmemBudget, "shared memory budget");
    static_assert(kStages >= 2, "need at least two smem stages");
    static_assert(kAStages >= 2, "need at least two TMEM A stages");
};

struct Barriers {
    uint64_t full[16];      // weights + scales of the stage landed (dequant warps wait)
    uint64_t full_act[16];  // token tile of the stage landed (MMA issuer waits)
    uint64_t empty[16];     // weights/scales of the stage consumed (dequant warps)
    uint64_t empty_act[16]; // token tile of the stage consumed (MMA commit; both CTAs if CL)
    uint64_t a_full[8];
    uint64_t a_empty[8];
    uint64_t acc_full[2];
    uint64_t acc_empty[2];
    uint64_t part_full;     // reducer: partial tiles landed in the (drained) stage ring
    uint32_t tmem_base;
    uint32_t flag;
};
static_assert(sizeof(Barriers) <= 1024, "barrier block too large");

// Work decomposition shared by every warp role.
struct Sched {
    uint32_t k_tiles, m_tiles, n_tiles;
    uint32_t total_units; // < 2^31, checked by the launcher
    uint32_t grid;
    uint32_t n_mul, n_add; // this CTA's n-tile = n_mul * (tile / m_tiles) + n_add
    const int8_t *adj;     // GemmArgs::cut_adj (kernel parameter space)

    __device__ __forceinline__ uint32_t begin(uint32_t b) const {
        return (uint32_t)((int32_t)((uint64_t)total_units * b / grid) + (int32_t)adj[b]);
    }
    // CTA that owns unit u (inverse of begin()): the equal-range owner, corrected for the cuts.
    __device__ __forceinline__ uint32_t owner(uint32_t u) const {
        uint32_t o = (uint32_t)((((uint64_t)u + 1) * grid - 1) / total_units);
        while (o > 0 && begin(o) > u) --o;
        while (o + 1 < grid && begin(o + 1) <= u) ++o;
        return o;
    }
};

struct Segment {
    uint32_t tile, n_tile, m_tile, kt0, kt1;
};

__device__ __forceinline__ Segment make_segment(const Sched &s, uint32_t u,
                                                uint32_t u_end) {
    Segment g;
    g.tile = u / s.k_tiles;
    g.kt0 = u - g.tile * s.k_tiles;
    uint32_t left = u_end - u;
    uint32_t room = s.k_tiles - g.kt0;
    g.kt1 = g.kt0 + (left < room ? left : room);
    g.n_tile = s.n_mul * (g.tile / s.m_tiles) + s.n_add;
    g.m_tile = g.tile % s.m_tiles;
    return g;
}

__device__ __forceinline__ void trace_stamp(const GemmArgs &args, int slot) {
    if (args.trace) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        args.trace[blockIdx.x * 16 + slot] = t;
    }
}
// Experiment hooks (per-stage timeline, PETIT_DEBUG_FLAGS knock-outs) cost ~20 % in the
// hot loops, so they only exist when compiled with -DPETIT_DEBUG_HOOKS.
#ifdef PETIT_DEBUG_HOOKS
#define PETIT_DBG(flags, bit) ((flags) & (bit))
#else
#define PETIT_DBG(flags, bit) false
#endif
// Per-stage timeline of CTA 0 (debug): slots [160*16 + stage*8 + ev], stage < 64.
__device__ __forceinline__ void trace_stage(const GemmArgs &args, uint32_t stage, int ev) {
#ifndef PETIT_DEBUG_HOOKS
    (void)args; (void)stage; (void)ev;
    return;
#endif
    if (args.trace && blockIdx.x == 0 && stage < 64) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        args.trace[160 * 16 + stage * 8 + ev] = t;
    }
}
template <int N> __device__ __forceinline__ void setmaxnreg_inc() {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N> __device__ __forceinline__ void setmaxnreg_dec() {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::
                     : "memory");
}
// 3-D tensor-map load delivered to every CTA in `mask` at the same smem / mbarrier offsets
__device__ __forceinline__ void tma_load_3d_mc(void *smem_dst, const CUtensorMap *map, uint64_t *bar,
                                               int c0, int c1, int c2, uint16_t mask) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
                 ".multicast::cluster [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(smem_u32(smem_dst)),
                 "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "h"(mask)
                 : "memory");
}
// tcgen05.commit arriving on the same mbarrier offset in every CTA of `mask`
__device__ __forceinline__ void tc_commit_mc(uint64_t *bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster"
                 ".b64 [%0], %1;" ::"r"(smem_u32(bar)),
                 "h"(mask)
                 : "memory");
}
__device__ __forceinline__ void griddep_wait() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
}
__device__ __forceinline__ void griddep_launch_dependents() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
    uint16_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr));
    return v;
}
template <bool kBf16> __device__ __forceinline__ uint16_t to_bits16(float r) {
    if (kBf16) return __bfloat16_as_ushort(__float2bfloat16_rn(r));
    return __half_as_ushort(__float2half_rn(r));
}

__device__ __forceinline__ void mbar_wait_addr(uint32_t bar_addr, uint32_t parity) {
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "W: mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                 "@p bra D;\n\tbra W;\n\tD:\n\t}" ::"r"(bar_addr),
                 "r"(parity)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive_addr(uint32_t bar_addr) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_addr) : "memory");
}

// ---------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------
// CL = true: thread-block clusters of two CTAs that work on the SAME token tile and k
// range but on adjacent n-tiles (2p, 2p+1).  Each CTA loads half of the token tile and
// TMA-multicasts it into both CTAs' shared memory, halving the L2->SM activation
// traffic that bounds the prefill kernel (measured 42.7 B/clk/SM, the L2 fabric cap).
// AR = true: the instantiation whose epilogue also all-reduces the output over NVLink (separate
// so that the plain GEMM's register allocation is untouched by the exchange code).
// GR = true: the grouped (MoE) instantiation -- token tile t of the schedule is row block
// table.e[t] of the concatenated activations and multiplies that entry's weights.
struct NoGroups {};
template <bool GR> struct GroupParam { using type = NoGroups; };
template <> struct GroupParam<true> { using type = GroupTable; };
__device__ __forceinline__ const GroupEntry &group_entry(const GroupTable &t, uint32_t i) { return t.e[i]; }
__device__ __forceinline__ GroupEntry group_entry(const NoGroups &, uint32_t) { return GroupEntry{}; }
__device__ __forceinline__ uint32_t group_tiles(const GroupTable &t) { return t.tiles; }
__device__ __forceinline__ uint32_t group_tiles(const NoGroups &) { return 0; }

// the grouped instantiation's parameters must fit the classic 4 KB kernel-parameter space
static_assert(2 * sizeof(CUtensorMap) + sizeof(GemmArgs) + sizeof(GroupTable) <= 4096,
              "kernel parameters of the grouped GEMM exceed 4 KB: shrink kMaxGroupTiles");

template <int MODE, int NTOK, int KS, bool CL, bool AR = false, bool GR = false>
__global__ void __launch_bounds__(kNumThreads, 1)
fp4_gemm_kernel(const __grid_constant__ CUtensorMap tmap_act,
                const __grid_constant__ CUtensorMap tmap_out,
                const __grid_constant__ GemmArgs args,
                const __grid_constant__ typename GroupParam<GR>::type table) {
    using C = Cfg<MODE, NTOK, KS>;
    uint32_t cta_rank = 0;
    if (CL) asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(cta_rank));
    const uint32_t sched_id = CL ? blockIdx.x / 2 : blockIdx.x; // cluster (or CTA) index
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // 1024-byte alignment for the 128B-swizzled activation slabs
    uint8_t *smem = reinterpret_cast<uint8_t *>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    Barriers *bars = reinterpret_cast<Barriers *>(smem);
    uint8_t *out_stage = smem + C::kBarrierBytes;
    const uint32_t pre_smem = smem_u32(out_stage + C::kOutBytes); // reducer pre-sums
    uint8_t *stage_base = out_stage + C::kOutBytes + C::kPreBytes;

    const uint32_t warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    if (threadIdx.x == 0) {
        trace_stamp(args, 0);
        if (args.trace) { // which SM this CTA landed on (trace buffer: [160][16] + [64][8] + [160])
            uint32_t smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            args.trace[160 * 16 + 64 * 8 + blockIdx.x] = smid;
        }
    }
    // Let the next kernel on the stream (if it was launched with programmatic stream
    // serialisation) start its prologue / weight prefetch on SMs as they free up.
    if (threadIdx.x == 0) griddep_launch_dependents();

    Sched sched;
    sched.k_tiles = args.k / kTileK;
    sched.n_tiles = (args.n + kTileN - 1) / kTileN;
    if (CL) sched.n_tiles /= 2; // unit space counts n-tile PAIRS (launcher ensures even)
    sched.m_tiles = GR ? group_tiles(table) : (args.m + NTOK - 1) / NTOK;
    sched.total_units = sched.k_tiles * sched.n_tiles * sched.m_tiles;
    sched.grid = CL ? gridDim.x / 2 : gridDim.x;
    sched.n_mul = CL ? 2 : 1;
    sched.n_add = cta_rank;
    sched.adj = args.cut_adj;
    const uint32_t u_begin = sched.begin(sched_id);
    const uint32_t u_end = sched.begin(sched_id + 1);

    if (warp == kProducerWarp && lane == 0) {
        prefetch_tensormap(&tmap_act);
        prefetch_tensormap(&tmap_out);
        for (int i = 0; i < C::kStages; ++i) {
            mbar_init(&bars->full[i], 1);
            mbar_init(&bars->full_act[i], 1);
            mbar_init(&bars->empty[i], C::kStageWarps);
            mbar_init(&bars->empty_act[i], CL ? 2 : C::kMmaWarps);
        }
        for (int i = 0; i < C::kAStages; ++i) {
            mbar_init(&bars->a_full[i], C::kStageWarps);
            mbar_init(&bars->a_empty[i], C::kMmaWarps);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars->acc_full[i], C::kMmaWarps);
            mbar_init(&bars->acc_empty[i], kNumEpilogueWarps * C::kEpiTeams);
        }
        mbar_init(&bars->part_full, 1);
        fence_mbar_init();
    }
    if (warp == kMmaWarp) tmem_alloc(&bars->tmem_base, 512);
    tc_fence_before();
    // The producer warp initialised the barriers itself, so it only signals the setup
    // barrier and starts streaming weights while the others wait for the TMEM base.
    if (CL) {
        // remote barriers must exist before the peer multicasts into them
        cluster_sync();
    } else if (warp == kProducerWarp) {
        __syncwarp();
        asm volatile("bar.arrive %0, %1;" ::"n"(kSetupBarId), "n"(kNumThreads) : "memory");
    } else {
        named_bar_sync(kSetupBarId, kNumThreads);
    }
    tc_fence_after();
    const uint32_t tmem = (!CL && warp == kProducerWarp) ? 0u : bars->tmem_base;
    const uint32_t tmem_a0 = tmem + C::kAccCols;
    if (threadIdx.x == 0) trace_stamp(args, 1);

    const uint32_t k_bytes_half = args.k / 2;

    if (warp < kFirstEpilogueWarp) setmaxnreg_dec<kRegsLight>();
    if (warp == kProducerWarp || warp == kActProducerWarp) {
        // ===================== TMA producers =====================
        // Two warps run the same stage loop, one per operand: warp 0 streams weights +
        // scales (-> full[s]), warp 2 the token tiles (-> full_act[s]).  The loops are
        // executed by the whole (converged) warp so that every value is warp-uniform; only
        // the async instructions are issued by one elected lane.
        //
        // Programmatic dependent launch: weights and scales are constants, so their warp
        // never waits for the grid dependency -- it fills the ring while the previous
        // kernel on the stream is still draining, and the dequant warps already fill the
        // TMEM A stages from it.  The token tile may be that kernel's output: its warp
        // starts with griddepcontrol.wait.  (With a single producer warp the ring-full of
        // weight requests -- ~0.2 us per stage of issue work -- sat in front of the wait;
        // a CTA that became resident late, behind the last CTAs of the previous grid,
        // asked for its first token tile 1.6 us after the dependency had resolved:
        // profiles/r01_percta_summary.txt.)
        const bool do_w = warp == kProducerWarp, do_act = !do_w;
        const uint64_t pol_stream = policy_evict_first();
        if (do_act) {
            griddep_wait();
            if (lane == 0) trace_stamp(args, 2);
        }
        uint32_t it = 0;
        for (uint32_t u = u_begin; u < u_end;) {
            const Segment g = make_segment(sched, u, u_end);
            const uint32_t rows = tile_rows(args.n, g.n_tile);
            const uint8_t *w_base = args.w, *sc_base = args.sc;
            uint32_t tok0 = g.m_tile * NTOK; // first token row of the tile
            if (GR) {
                const GroupEntry &ge = group_entry(table, g.m_tile);
                w_base = ge.w;
                sc_base = ge.sc;
                tok0 = ge.row0;
            }
            const uint8_t *w_tile = w_base + (size_t)g.n_tile * kTileN * k_bytes_half;
            const uint8_t *sc_tile =
                sc_base + (size_t)g.n_tile * kTileN * (args.k / 64) * C::kScPerSub;
            const uint32_t w_stage_bytes = C::kChunks * rows * 16;
            const uint32_t sc_stage_bytes = C::kSubs * rows * C::kScPerSub;
            const uint32_t n_stage = (g.kt1 - g.kt0) * C::kStagesPerUnit;
            const uint8_t *w_src = w_tile + (size_t)g.kt0 * rows * 128;
            const uint8_t *sc_src = sc_tile + (size_t)g.kt0 * rows * 4 * C::kScPerSub;
            int32_t k_slab = (int32_t)(g.kt0 * 4);
            for (uint32_t i = 0; i < n_stage; ++i, ++it) {
                const uint32_t s = it % C::kStages;
                const uint32_t ph = (it / C::kStages) & 1;
                if (it >= (uint32_t)C::kStages)
                    mbar_wait(do_w ? &bars->empty[s] : &bars->empty_act[s], ph ^ 1);
                if (elect_one()) {
                    uint8_t *st = stage_base + (size_t)s * C::kStageBytes;
                    trace_stage(args, it, do_w ? 0 : 1);
                    if (do_w) {
                        mbar_arrive_expect_tx(&bars->full[s], w_stage_bytes + sc_stage_bytes);
                        bulk_g2s_hint(st + C::kActBytes, w_src, w_stage_bytes,
                                      &bars->full[s], pol_stream);
                        if (PETIT_DBG(args.debug_flags, 8u)) // experiment: no scale copy
                            asm volatile("mbarrier.complete_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(
                                             smem_u32(&bars->full[s])),
                                         "r"(sc_stage_bytes)
                                         : "memory");
                        else
                        bulk_g2s_hint(st + C::kActBytes + C::kWBytes, sc_src,
                                      sc_stage_bytes, &bars->full[s], pol_stream);
                    } else {
                        // token tile: box {64 k, NTOK tokens, kSubs slabs}
                        mbar_arrive_expect_tx(&bars->full_act[s], C::kActBytes);
                        if (PETIT_DBG(args.debug_flags, 4u)) // experiment: no token-tile traffic
                            asm volatile("mbarrier.complete_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(
                                             smem_u32(&bars->full_act[s])),
                                         "r"((uint32_t)C::kActBytes)
                                         : "memory");
                        else if (CL) {
                            // my half of the token rows, one 128-byte-row slab per
                            // call, delivered to both CTAs of the cluster
#pragma unroll
                            for (int sl = 0; sl < C::kSubs; ++sl)
                                tma_load_3d_mc(st + sl * (NTOK * 128) +
                                                   cta_rank * (NTOK / 2) * 128,
                                               &tmap_act, &bars->full_act[s], 0,
                                               tok0 + cta_rank * (NTOK / 2),
                                               k_slab + sl, (uint16_t)3);
                        } else
                            tma_load_3d(st, &tmap_act, &bars->full_act[s], 0, tok0, k_slab);
                    }
                }
                __syncwarp();
                w_src += w_stage_bytes;
                sc_src += sc_stage_bytes;
                k_slab += C::kSubs;
            }
            u += g.kt1 - g.kt0;
        }
    } else if (warp == kMmaWarp || (C::kMmaWarps == 2 && warp == kMmaWarp2)) {
        // ===================== MMA issuer(s) =====================
        // Decode tiles: warp 1 issues the k-steps of the lower half of the accumulator chains,
        // warp 3 those of the upper half (a chain is only ever touched by one thread, so the
        // MMAs of a chain stay ordered); both commit to the stage barriers (count 2).
        constexpr uint32_t idesc = make_idesc_f16(
            C::kIsBf16 ? kFmtBF16 : kFmtF16, C::kIsBf16 ? kFmtBF16 : kFmtF16, 128, NTOK);
        constexpr int kHalfChains = C::kChains / C::kMmaWarps;
        const uint64_t bdesc0 = make_smem_desc_sw128(smem_u32(stage_base));
        auto mma_loop = [&](auto upper_tag) {
        constexpr bool kUpper = decltype(upper_tag)::value; // this warp owns the upper chains
        uint64_t bdesc_s = bdesc0;
        uint32_t a_tmem = tmem_a0;
        uint32_t s = 0, ph = 0, ta = 0, ta_ph = 0, seg = 0;
        for (uint32_t u = u_begin; u < u_end; ++seg) {
            const Segment g = make_segment(sched, u, u_end);
            const uint32_t acc = seg % C::kNumAcc;
            const uint32_t acc_ph = (seg / C::kNumAcc) & 1;
            mbar_wait(&bars->acc_empty[acc], acc_ph ^ 1);
            tc_fence_after();
            const uint32_t d_tmem = tmem + acc * C::kAccBufCols;
            const uint32_t n_stage = (g.kt1 - g.kt0) * C::kStagesPerUnit;
            for (uint32_t i = 0; i < n_stage; ++i) {
                mbar_wait(&bars->full_act[s], ph);  // token tile landed
#ifdef PETIT_DEBUG_HOOKS
                if (seg == 0 && i == 0 && lane == 0) trace_stamp(args, 3);
#endif
                mbar_wait(&bars->a_full[ta], ta_ph); // weights are in TMEM
                tc_fence_after();
                if (elect_one()) {
#pragma unroll
                    for (int j = 0; j < KS / 16; ++j) {
                        if ((PETIT_KO & 1) && j >= 4) continue; // experiment: fewer MMAs
                        const int chain = j % C::kChains;
                        if (C::kMmaWarps == 2 && (chain >= kHalfChains) != kUpper) continue;
                        const uint64_t bdesc =
                            bdesc_s + (uint64_t)(((j / 4) * (NTOK * 128) + (j % 4) * 32) >> 4);
                        mma_f16_ts(d_tmem + chain * NTOK, a_tmem + j * 8, bdesc, idesc,
                                   (i != 0 || j >= C::kChains) ? 1u : 0u);
                    }
                    tc_commit(&bars->a_empty[ta]);
                    if (CL)
                        tc_commit_mc(&bars->empty_act[s], (uint16_t)3);
                    else
                        tc_commit(&bars->empty_act[s]);
                    if (i + 1 == n_stage) tc_commit(&bars->acc_full[acc]);
                }
                __syncwarp();
                bdesc_s += (uint64_t)(C::kStageBytes >> 4);
                a_tmem += C::kACols;
                if (++s == (uint32_t)C::kStages) { s = 0; ph ^= 1; bdesc_s = bdesc0; }
                if (++ta == (uint32_t)C::kAStages) { ta = 0; ta_ph ^= 1; a_tmem = tmem_a0; }
            }
            u += g.kt1 - g.kt0;
        }
        };
        if (C::kMmaWarps == 2 && warp == kMmaWarp2)
            mma_loop(std::true_type{});
        else
            mma_loop(std::false_type{});
        if (lane == 0 && warp == kMmaWarp) trace_stamp(args, 5);
    } else if (warp >= kFirstDequantWarp &&
               (warp - kFirstDequantWarp) / 4 < (uint32_t)C::kUsedSlices) {
        // ===================== dequant warps =====================
        setmaxnreg_inc<kRegsDequant>();
        const uint32_t dw = warp - kFirstDequantWarp;
        const uint32_t quarter = warp % 4;     // TMEM lane quarter this warp may touch
        const uint32_t kslice = dw / 4;        // which slice of the stage's k range
        const uint32_t row = quarter * 32 + lane;
        constexpr int kMyChunks = C::kChunks / C::kActiveSlices;
        constexpr int kScBytesPerChunk = C::kScPerSub / 2; // NV: 2 bytes, MX: 1 byte
        const uint32_t group = kslice / C::kActiveSlices;  // which alternate stages are mine
        const uint32_t c0 = (kslice % C::kActiveSlices) * kMyChunks; // first chunk of this thread
        const uint32_t w_base = smem_u32(stage_base) + C::kActBytes;
        const uint32_t tmem_dst = tmem_a0 + ((quarter * 32) << 16) + c0 * 16;
        uint32_t s = 0, ph = 0, ta = 0, ta_ph = 1; // ta_ph: parity to wait on a_empty
        uint32_t it_dbg = 0;
        // The four k-slice warps of a lane quarter share one SM sub-partition and run
        // identical code; in lockstep they all hit the ALU-heavy (F2FP/LOP3) and the
        // FMA-heavy (IMAD.HI/HMUL2) parts of the loop body together and each pipe
        // idles half the time.  A one-off skew keeps them in different phases.
        if (args.skew_cycles) {
            const long long t0 = clock64();
            const long long wait = (long long)kslice * args.skew_cycles;
            while (clock64() - t0 < wait) {
            }
        }
        // Fast path (every n-tile has 128 rows -- all Llama shapes): the weight stream is one
        // continuous sequence of stages, nothing in it depends on which output tile a stage
        // belongs to, so the loop runs flat over this CTA's stages (no per-segment state), a
        // group steps straight to its own stages, and every shared-memory offset is an
        // immediate.  Ring state lives in running addresses (no multiplies / modulo).
        if (args.n % kTileN == 0) {
            constexpr uint32_t kG = C::kGroups;
            const uint32_t total = (u_end - u_begin) * C::kStagesPerUnit;
            const uint32_t bars_addr = smem_u32(bars);
            const uint32_t full_b = bars_addr + (uint32_t)offsetof(Barriers, full);
            const uint32_t aempty_b = bars_addr + (uint32_t)offsetof(Barriers, a_empty);
            constexpr uint32_t kFullToEmpty = (uint32_t)(offsetof(Barriers, empty) - offsetof(Barriers, full));
            constexpr int32_t kEmptyToFullA = (int32_t)offsetof(Barriers, a_full) - (int32_t)offsetof(Barriers, a_empty);
            const uint32_t lane_off = (c0 * kTileN + row) * 16;
            const uint32_t sc_lane_off = C::kWBytes + ((c0 / 2) * kTileN + row) * C::kScPerSub +
                                         (c0 & 1) * kScBytesPerChunk;
            const uint32_t st0 = w_base + lane_off, sc0 = w_base + sc_lane_off;
            const bool lane0 = lane == 0;
            // one stage of this thread: wait for the weights, load, wait for the TMEM slot,
            // convert + store, hand over
            auto stage_body = [&](uint32_t st_w, uint32_t st_sc, uint32_t fb, uint32_t ph2, uint32_t ab,
                                  uint32_t aph, uint32_t tm) {
                mbar_wait_addr(fb, ph2);
                uint4 q[kMyChunks];
#pragma unroll
                for (int ci = 0; ci < kMyChunks; ++ci) q[ci] = lds_v4(st_w + ci * (kTileN * 16));
                constexpr int kScLoads = kMyChunks >= 2 ? kMyChunks / 2 : 1;
                uint32_t scw[kScLoads];
#pragma unroll
                for (int p = 0; p < kScLoads; ++p) {
                    const uint32_t a = st_sc + p * (kTileN * C::kScPerSub);
                    if (kMyChunks >= 2)
                        scw[p] = C::kIsMx ? lds_u16(a) : lds_u32(a);
                    else
                        scw[p] = C::kIsMx ? lds_u8(a) : lds_u16(a);
                }
                // the previous occupant of this TMEM A stage must have been consumed
                mbar_wait_addr(ab, aph);
                tc_fence_after();
                // MXFP4 scales >= 2^-1 (e8m0 > 125) need a second exact multiply.  Real MX
                // weight scales are far below that, so the decision is taken once per stage for
                // the whole warp and the common case runs a loop body without the second
                // multiply (it used to be issued unconditionally: 64 of 366 instructions).
                bool any_two = false;
                if (C::kIsMx) {
                    bool mine = false;
#pragma unroll
                    for (int p = 0; p < kScLoads; ++p)
                        mine = mine || mx_needs_two_step(scw[p]) || mx_needs_two_step(scw[p] >> 8);
                    any_two = __any_sync(0xffffffffu, mine);
                }
                auto convert = [&](auto two_tag) {
                    constexpr bool kTwo = decltype(two_tag)::value;
#pragma unroll
                    for (int ci = 0; ci < kMyChunks; ++ci) {
                        const uint32_t bits = scw[ci / 2] >> ((ci & 1) * 8 * kScBytesPerChunk);
                        const uint32_t mult = chunk_multiplier<MODE>(bits, kTwo);
                        uint32_t out[16];
#if PETIT_KO & 2
#pragma unroll
                        for (int j = 0; j < 16; ++j) out[j] = q[ci].x + j;
#else
                        dequant_chunk<MODE>(q[ci], mult, kTwo, out);
#endif
#if PETIT_KO & 16
                        asm volatile("" ::"r"(out[0]), "r"(out[1]), "r"(out[2]), "r"(out[3]), "r"(out[4]),
                                     "r"(out[5]), "r"(out[6]), "r"(out[7]), "r"(out[8]), "r"(out[9]),
                                     "r"(out[10]), "r"(out[11]), "r"(out[12]), "r"(out[13]),
                                     "r"(out[14]), "r"(out[15]));
#else
                        tmem_st_x16(tm + ci * 16, out);
#endif
                    }
                };
                if (C::kIsMx && any_two)
                    convert(std::true_type{});
                else
                    convert(std::false_type{});
                if (!(PETIT_KO & 32)) tmem_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane0) {
                    mbar_arrive_addr((uint32_t)((int32_t)ab + kEmptyToFullA)); // a_full[slot]
                    mbar_arrive_addr(fb + kFullToEmpty);                        // empty[stage]
                }
            };
            constexpr bool kPeriodic = PETIT_PERIODIC && C::kStages == 6 && C::kAStages == 3 && kG == 2;
            if (kPeriodic) {
                // Group g takes stages g, g + 2, g + 4, ...: stage index mod 6 and TMEM slot mod 3
                // repeat every 3 iterations, and the a_empty parity of an iteration depends only
                // on its position r in that period (use count of the slot = (g + 2r) / 3 + 2q).
                // So: three copies of the body with constant offsets, one toggling bit.
                const uint32_t wg = st0 + group * C::kStageBytes, scg = sc0 + group * C::kStageBytes;
                const uint32_t fbg = full_b + group * 8;
                uint32_t ab_r[3], ap_r[3], tm_r[3];
#pragma unroll
                for (uint32_t r = 0; r < 3; ++r) {
                    const uint32_t i0 = group + 2 * r, slot = i0 % 3;
                    ab_r[r] = aempty_b + slot * 8;
                    ap_r[r] = ((i0 / 3) & 1u) ^ 1u;
                    tm_r[r] = tmem_dst + slot * C::kACols;
                }
                const uint32_t nj = total > group ? (total - group + 1) / 2 : 0;
                uint32_t j = 0, qpar = 0;
                for (; j + 3 <= nj; j += 3, qpar ^= 1) {
#pragma unroll
                    for (uint32_t r = 0; r < 3; ++r)
                        stage_body(wg + 2 * r * C::kStageBytes, scg + 2 * r * C::kStageBytes,
                                   fbg + 2 * r * 8, qpar, ab_r[r], ap_r[r], tm_r[r]);
                }
#pragma unroll
                for (uint32_t r = 0; r < 2; ++r)
                    if (j + r < nj)
                        stage_body(wg + 2 * r * C::kStageBytes, scg + 2 * r * C::kStageBytes,
                                   fbg + 2 * r * 8, qpar, ab_r[r], ap_r[r], tm_r[r]);
            } else {
            // position of this group's first stage
            uint32_t sidx = group % C::kStages, ph2 = 0, aidx = group % C::kAStages, aph = 1;
            uint32_t st_w = st0 + sidx * C::kStageBytes, st_sc = sc0 + sidx * C::kStageBytes;
            uint32_t fb = full_b + sidx * 8, ab = aempty_b + aidx * 8;
            uint32_t tm = tmem_dst + aidx * C::kACols;
            for (uint32_t it = group; it < total; it += kG) {
                stage_body(st_w, st_sc, fb, ph2, ab, aph, tm);
                // step to this group's next stage
                sidx += kG; st_w += kG * C::kStageBytes; st_sc += kG * C::kStageBytes; fb += kG * 8;
                if (sidx >= (uint32_t)C::kStages) {
                    sidx -= C::kStages; ph2 ^= 1;
                    st_w -= C::kStages * C::kStageBytes; st_sc -= C::kStages * C::kStageBytes;
                    fb -= C::kStages * 8;
                }
                aidx += kG; ab += kG * 8; tm += kG * C::kACols;
                if (aidx >= (uint32_t)C::kAStages) {
                    aidx -= C::kAStages; aph ^= 1;
                    ab -= C::kAStages * 8; tm -= C::kAStages * C::kACols;
                }
            }
            }
        } else
        for (uint32_t u = u_begin; u < u_end;) {
            const Segment g = make_segment(sched, u, u_end);
            const uint32_t rows = tile_rows(args.n, g.n_tile);
            // rows past the end of a cut n-tile re-read the last valid row: their
            // accumulator lanes are never stored, and no predication is needed.
            const uint32_t rrow = row < rows ? row : rows - 1;
            const uint32_t w_off = (c0 * rows + rrow) * 16;
            const uint32_t sc_off = C::kWBytes + ((c0 / 2) * rows + rrow) * C::kScPerSub +
                                    (c0 & 1) * kScBytesPerChunk;
            const uint32_t n_stage = (g.kt1 - g.kt0) * C::kStagesPerUnit;
            for (uint32_t i = 0; i < n_stage; ++i) {
                if (C::kGroups > 1 && (it_dbg % C::kGroups) != group) {
                    ++it_dbg;
                    if (++s == C::kStages) { s = 0; ph ^= 1; }
                    if (++ta == C::kAStages) { ta = 0; ta_ph ^= 1; }
                    continue;
                }
                const uint32_t st = w_base + s * C::kStageBytes;
                mbar_wait(&bars->full[s], ph);
                if (threadIdx.x == kFirstDequantWarp * 32) trace_stage(args, it_dbg, 2);
                uint4 q[kMyChunks];
#pragma unroll
                for (int ci = 0; ci < kMyChunks; ++ci) q[ci] = lds_v4(st + w_off + ci * rows * 16);
                // scale bytes: one 64-k slab (= 2 chunks) per load
                constexpr int kScLoads = kMyChunks >= 2 ? kMyChunks / 2 : 1;
                uint32_t scw[kScLoads];
#pragma unroll
                for (int p = 0; p < kScLoads; ++p) {
                    const uint32_t a = st + sc_off + p * rows * C::kScPerSub;
                    if (kMyChunks >= 2)
                        scw[p] = C::kIsMx ? lds_u16(a) : lds_u32(a);
                    else
                        scw[p] = C::kIsMx ? lds_u8(a) : lds_u16(a);
                }
                // the previous occupant of this TMEM A stage must have been consumed
                mbar_wait(&bars->a_empty[ta], ta_ph);
                tc_fence_after();
                if (threadIdx.x == kFirstDequantWarp * 32) trace_stage(args, it_dbg, 3);
#pragma unroll
                for (int ci = 0; ci < kMyChunks; ++ci) {
                    const uint32_t bits = scw[ci / 2] >> ((ci & 1) * 8 * kScBytesPerChunk);
                    bool two_step = false;
                    if (C::kIsMx) two_step = __any_sync(0xffffffffu, mx_needs_two_step(bits));
                    const uint32_t mult = chunk_multiplier<MODE>(bits, two_step);
                    uint32_t out[16];
                    if (PETIT_DBG(args.debug_flags, 2u)) { // experiment: no dequant math
#pragma unroll
                        for (int j = 0; j < 16; ++j) out[j] = q[ci].x + j;
                    } else
                    dequant_chunk<MODE>(q[ci], mult, two_step, out);
                    if (!PETIT_DBG(args.debug_flags, 16u)) // experiment: no TMEM stores
                    tmem_st_x16(tmem_dst + ta * C::kACols + ci * 16, out);
                }
                tmem_wait_st();
                tc_fence_before();
                __syncwarp();
                if (threadIdx.x == kFirstDequantWarp * 32) trace_stage(args, it_dbg, 4);
                ++it_dbg;
                if (lane == 0) {
                    mbar_arrive(&bars->a_full[ta]);
                    mbar_arrive(&bars->empty[s]);
                }
                if (++s == C::kStages) { s = 0; ph ^= 1; }
                if (++ta == C::kAStages) { ta = 0; ta_ph ^= 1; }
            }
            u += g.kt1 - g.kt0;
        }
        if (threadIdx.x == kFirstDequantWarp * 32) trace_stamp(args, 4);
    } else if ((warp >= kFirstEpilogueWarp && warp < kFirstDequantWarp) ||
               (C::kEpiTeams > 1 && warp >= kFirstDequantWarp + 4 * C::kUsedSlices)) {
        // ===================== epilogue warps =====================
        setmaxnreg_inc<kRegsDequant>();
        // team 0 = warps 4-7; with kEpiTeams == 3 the idle dequant warps 16-19 / 20-23 are
        // teams 1 / 2.  A team's four warps cover the four TMEM lane quarters.
        const uint32_t quarter = warp % 4;
        const uint32_t team = warp < kFirstDequantWarp
                                  ? 0u
                                  : 1u + (warp - kFirstDequantWarp - 4 * C::kUsedSlices) / 4;
        const uint32_t ew_tid = (warp % 4) * 32 + lane; // 0..127 inside the team
        const bool lead = team == 0 && ew_tid == 0;      // the one thread that polls / publishes
        constexpr int kAllEpiThreads = kNumEpilogueWarps * 32 * C::kEpiTeams;
        const int team_bar = kTeamBarId0 + (int)team;
        uint8_t *team_stage = out_stage + team * (C::kOutBufs * C::kOutStageBytes);
        bool ring_ready = false;
        const uint32_t row = quarter * 32 + lane;
        const uint32_t lane_base = (quarter * 32) << 16;
        griddep_wait(); // global_scale, workspace and C may depend on the previous kernel
        float gs = GR ? 0.f : *args.global_scale;
        gs *= epilogue_factor<MODE>(); // power of two folded out of the A operand
        uint32_t ar_epoch = 0;
        if (AR)
            asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(ar_epoch) : "l"(args.ar_state) : "memory");
        const uint32_t sched_tiles_n = (args.n + kTileN - 1) / kTileN;
        uint32_t seg = 0;
        uint32_t out_buf = 0; // staging buffer the next 16-token group goes to
        for (uint32_t u = u_begin; u < u_end; ++seg) {
            const Segment g = make_segment(sched, u, u_end);
            const uint32_t rows = tile_rows(args.n, g.n_tile);
            const uint32_t acc = seg % C::kNumAcc;
            const uint32_t acc_ph = (seg / C::kNumAcc) & 1;
            const bool full_k = g.kt0 == 0 && g.kt1 == sched.k_tiles;
            uint32_t m0 = g.m_tile * NTOK;
            uint32_t m_valid = args.m - m0 < (uint32_t)NTOK ? args.m - m0 : NTOK;
            if (GR) { // this tile's row block and its group's scale
                const GroupEntry &ge = group_entry(table, g.m_tile);
                m0 = ge.row0;
                m_valid = ge.rows;
                gs = __ldg(ge.gs) * epilogue_factor<MODE>();
            }

            // Split tiles (stream-K): the CTA that owns the FIRST k-part of a tile
            // reaches it as the last segment of its range, after every other
            // contributor (which meets the tile at the START of its range) has
            // published its fp32 partial.  So that CTA is the reducer: it adds the
            // published partials to its own accumulator in CTA order (deterministic)
            // and writes the output; contributors never wait.
            const bool is_reducer = !full_k && g.kt0 == 0;
            const bool is_contrib = !full_k && g.kt0 != 0;
            float *slot = args.ws_partials + (size_t)blockIdx.x * (kTileN * NTOK);
            // ids below are scheduling units (clusters if CL); the contributor of unit b to
            // THIS CTA's tile is the CTA of the same cluster rank, i.e. slot b * n_mul + n_add
            uint32_t b_first = sched_id, b_last = sched_id;
            if (is_reducer) b_last = sched.owner(g.tile * sched.k_tiles + sched.k_tiles - 1);
            const uint32_t out_tile = g.n_tile * sched.m_tiles + g.m_tile;

            // Reducer: contributors that met the tile at the start of their range published
            // long ago, so their partials for the first 16 tokens are summed (in CTA order)
            // into this thread's shared-memory slots while the MMAs of this last segment are
            // still running; the tail after acc_full is then TMEM read + add + store.
            const uint32_t pre_addr = pre_smem + row * 4; // + j * 512: this thread's 16 sums
            // A tile split over many CTAs (small TP shards: 10 n-tiles on 148 SMs) would cost
            // one L2 round trip per contributor in the register path below; from 4
            // contributors on, the first 16 tokens go through the ring like the rest.
            constexpr uint32_t kRingFit = (uint32_t)(C::kStages * C::kStageBytes) / (NTOK * kTileN * 4);
            const uint32_t ring_from = (is_reducer && b_last - b_first > 3u && b_last - b_first <= kRingFit) ? 0u : 16u;
            const bool last_seg = u + (g.kt1 - g.kt0) >= u_end;
            if (lead && last_seg) trace_stamp(args, 11);
            if (is_reducer) {
                if (lead) {
                    // The contributors are CTAs with higher block ids.  They never wait for
                    // anyone, so they publish as soon as they are resident -- which needs the
                    // whole grid (<= one CTA per SM) to become co-resident.  Another grid that
                    // holds SMs and itself waits (two stream-K GEMMs interleaved by a
                    // high-priority stream) could keep them out for ever: a watchdog turns that
                    // hang into a reported error (petit_workspace_status) and the CTA goes on
                    // with what it has.
                    const uint32_t need = b_last - b_first;
                    uint32_t seen, spins = 0;
                    unsigned long long t_start = 0;
                    for (;;) {
                        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];"
                                     : "=r"(seen)
                                     : "l"(args.ws_counters + out_tile)
                                     : "memory");
                        if (seen >= need) break;
                        if ((++spins & 0x3ff) == 0) {
                            unsigned long long now;
                            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                            if (t_start == 0) t_start = now;
                            if (now - t_start > args.watchdog_ns) {
                                atomicExch(args.ws_status, 1u + out_tile);
                                break;
                            }
                        }
                    }
                    if (last_seg) trace_stamp(args, 12);
                }
                named_bar_sync(kEpilogueBarId, kAllEpiThreads);
#pragma unroll 1
                // Two contributors per round trip: all loads of a pair are in flight before
                // the first add; the sum order stays CTA order.  (A reducer whose last
                // contributor publishes at the very end has these L2 round trips on the
                // kernel's critical path: profiles/r01_percta_summary.txt, `down`.)
                for (uint32_t b = b_first + 1; b <= b_last && ring_from != 0 && team == 0; b += 2) {
                    const float *p = args.ws_partials +
                                     (size_t)(b * sched.n_mul + sched.n_add) * (kTileN * NTOK) + row;
                    const bool two = b + 1 <= b_last;
                    const float *p2 = p + (size_t)sched.n_mul * (kTileN * NTOK);
                    float x[16], y[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        x[j] = (uint32_t)j < m_valid ? __ldcg(p + (size_t)j * kTileN) : 0.f;
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        y[j] = (two && (uint32_t)j < m_valid) ? __ldcg(p2 + (size_t)j * kTileN) : 0.f;
                    const bool first = b == b_first + 1;
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        float acc = first ? 0.f : lds_f32(pre_addr + j * (kTileN * 4));
                        acc += x[j];
                        acc += y[j];
                        sts_f32(pre_addr + j * (kTileN * 4), acc);
                    }
                }
            }
            if (lead && last_seg) trace_stamp(args, 13);
            while (!mbar_try_wait(&bars->acc_full[acc], acc_ph)) __nanosleep(32);
            tc_fence_after();
            if (lead && last_seg) trace_stamp(args, 6);
            // Reducer, tokens 16.. : the reducer segment is the LAST of this CTA's range and
            // its MMAs are complete, so the whole stage ring is idle -- the contributors'
            // partial tiles (tokens 16..m_valid) are pulled into it with one bulk copy each
            // (one L2 round trip in total instead of one per 16-token group).
            const uint32_t n_ring = (is_reducer && m_valid > ring_from)
                                        ? (b_last - b_first < kRingFit ? b_last - b_first : kRingFit)
                                        : 0u;
            if (n_ring && lead) {
                const uint32_t bytes = (m_valid - ring_from) * (kTileN * 4);
                mbar_arrive_expect_tx(&bars->part_full, n_ring * bytes);
                for (uint32_t i = 0; i < n_ring; ++i)
                    bulk_g2s(stage_base + (size_t)i * (NTOK * kTileN * 4) + ring_from * kTileN * 4,
                             args.ws_partials +
                                 (size_t)((b_first + 1 + i) * sched.n_mul + sched.n_add) *
                                     (kTileN * NTOK) +
                                 ring_from * kTileN,
                             bytes, &bars->part_full);
            }
            if (lead && seg == 1) trace_stamp(args, 9); // a mid-kernel tile: epilogue begin
#pragma unroll 1
            for (int c0 = (int)team * 16; c0 < NTOK; c0 += 16 * C::kEpiTeams) {
                if ((uint32_t)c0 >= m_valid) break; // tokens beyond M are never stored
                float v[16];
                {
                    uint32_t r0[16];
                    tmem_ld_x16(tmem + lane_base + acc * C::kAccBufCols + c0, r0);
                    tmem_wait_ld();
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r0[j]);
                }
                if (lead && last_seg && c0 == 0) trace_stamp(args, 14);
#pragma unroll
                for (int ch = 1; ch < C::kChains; ++ch) {
                    uint32_t r1[16];
                    tmem_ld_x16(tmem + lane_base + acc * C::kAccBufCols + ch * NTOK + c0, r1);
                    tmem_wait_ld();
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] += __uint_as_float(r1[j]);
                }
                if (is_contrib) {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if ((uint32_t)(c0 + j) < m_valid)
                            __stcg(&slot[(size_t)(c0 + j) * kTileN + row], v[j]);
                    continue;
                }
                if (is_reducer && (uint32_t)c0 < ring_from) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] += lds_f32(pre_addr + j * (kTileN * 4));
                } else if (is_reducer && !PETIT_DBG(args.debug_flags, 32u)) {
                    if (n_ring) {
                        if (!ring_ready) {
                            while (!mbar_try_wait(&bars->part_full, 0)) __nanosleep(32);
                            ring_ready = true;
                        }
#pragma unroll 1
                        for (uint32_t i = 0; i < n_ring; ++i) {
                            const uint32_t src = smem_u32(stage_base) + i * (NTOK * kTileN * 4) +
                                                 (uint32_t)c0 * (kTileN * 4) + row * 4;
                            // all 16 loads first, then the adds; tokens >= m_valid read stale
                            // ring bytes into lanes that the TMA store clips
                            uint32_t x[16];
#pragma unroll
                            for (int j = 0; j < 16; ++j) x[j] = lds_u32(src + j * (kTileN * 4));
#pragma unroll
                            for (int j = 0; j < 16; ++j) v[j] += __uint_as_float(x[j]);
                        }
                    }
                    // partial tiles that did not fit the ring (tile split over many CTAs):
                    // straight from L2, in CTA order like the rest
#pragma unroll 1
                    for (uint32_t bb = b_first + 1 + n_ring; bb <= b_last; ++bb) {
                        const float *p = args.ws_partials +
                                         (size_t)(bb * sched.n_mul + sched.n_add) * (kTileN * NTOK) +
                                         (size_t)c0 * kTileN + row;
                        float x[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            x[j] = (uint32_t)(c0 + j) < m_valid ? __ldcg(p + (size_t)j * kTileN) : 0.f;
#pragma unroll
                        for (int j = 0; j < 16; ++j) v[j] += x[j];
                    }
                }
                // Fused epilogue terms (extends WriteResult, qgemm.cuh:146-156): the final owner of
                // a tile adds bias[n] and residual[m, n] in fp32 before the one rounding to the
                // output type.  (Under the fused all-reduce they go into THIS rank's partial: a
                // row-parallel layer passes them on one rank only, as frameworks do with bias.)
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] *= gs;
                if (args.bias != nullptr || args.residual != nullptr) {
                    const uint32_t col = g.n_tile * kTileN + row;
                    if (row < rows) {
                        if (args.bias != nullptr) {
                            const uint16_t bb = static_cast<const uint16_t *>(args.bias)[col];
                            const float bv = C::kIsBf16 ? __uint_as_float((uint32_t)bb << 16)
                                                        : __half2float(__ushort_as_half(bb));
#pragma unroll
                            for (int j = 0; j < 16; ++j) v[j] += bv;
                        }
                        if (args.residual != nullptr) {
                            const uint16_t *rp = static_cast<const uint16_t *>(args.residual) +
                                                 (size_t)(m0 + c0) * args.n + col;
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                if ((uint32_t)(c0 + j) < m_valid) {
                                    const uint16_t rb = rp[(size_t)j * args.n];
                                    v[j] += C::kIsBf16 ? __uint_as_float((uint32_t)rb << 16)
                                                       : __half2float(__ushort_as_half(rb));
                                }
                        }
                    }
                }
                if (AR) {
                    // ---- fused all-reduce (row-parallel GEMM): v[] holds this rank's partial.
                    // Every rank finishes the same tile at about the same time (same shapes,
                    // same schedule).  16-bit values travel as 16-byte packets {4 B data, epoch,
                    // 4 B data, epoch} -- each 8-byte half validates itself, so no fence or flag
                    // write is needed -- into the destination rank's receive buffer
                    // [parity][source rank][slot]; ranks' values are always added in rank order
                    // in fp32, so every rank ends up with the same bits.
                    //  one-shot (world <= 4): push the partial to every peer, sum all partials.
                    //  two-shot (world 8): reduce-scatter + all-gather inside every tile --
                    //    rank r reduces rows [r * 128 / world, (r + 1) * 128 / world) of EVERY
                    //    tile: a thread pushes its row's partial to the row's reducer and waits
                    //    for the finished row, the reducer's threads sum the peers' partials and
                    //    push the finished rows to everyone.  An SM sustains only ~10 GB/s of
                    //    NVLink stores (measured: one CTA pushing a finished 8 KB tile to 7 peers
                    //    took 5-10 us, the one-shot exchange 16 us per GEMM at 8 ranks), so the
                    //    bytes have to be few (4x fewer than one-shot at 8 ranks) AND spread
                    //    over all the CTAs that finish tiles.
                    // Two buffer parities alternate per call: a rank can only get one call ahead
                    // of a peer (it needs that peer's packets to finish a call).
                    // Epoch 0 is never used: a slot no call has written yet is all zero bytes,
                    // i.e. a valid packet of epoch 0 holding 0, which a reader would take for a
                    // peer's partial.  So the call counter state[0] runs modulo kArCallPeriod =
                    // 2^32 - 2 and the epochs run 1 .. 2^32 - 2; the period is even, so the
                    // parity still alternates from one call to the next across the wrap.
                    const uint32_t epoch = ar_epoch + 1;
                    const uint32_t n_slots = sched_tiles_n * (kArMaxTokens / 16);
                    const uint32_t slot = g.n_tile * (kArMaxTokens / 16) + (m0 + (uint32_t)c0) / 16;
                    const size_t src_stride = (size_t)n_slots * kArSlotBytes;
                    const size_t par_off = (size_t)(epoch & 1) * kArMaxWorld * src_stride;
                    const size_t my_off = par_off + (size_t)args.ar_rank * src_stride +
                                          (size_t)slot * kArSlotBytes + row * 16;
                    const uint8_t *my_recv = nullptr; // (constant indices: no local copy of the array)
#pragma unroll
                    for (uint32_t p = 0; p < kArMaxWorld; ++p)
                        if (p == args.ar_rank) my_recv = args.ar_recv[p];
                    const uint8_t *rbase = my_recv + par_off + (size_t)slot * kArSlotBytes + row * 16;
                    const uint32_t all_mask = (1u << args.ar_world) - 1u;
                    const uint32_t me_bit = 1u << args.ar_rank;
                    const bool two_shot = args.ar_two_shot != 0; // host: only if 128 % world == 0
                    const uint32_t owner = two_shot ? row / (kTileN / args.ar_world) : args.ar_rank;
                    uint32_t res[8]; // the tile's 16 tokens of this row as 16-bit pairs
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        res[j] = (uint32_t)to_bits16<C::kIsBf16>(v[2 * j]) |
                                 ((uint32_t)to_bits16<C::kIsBf16>(v[2 * j + 1]) << 16);
                    uint32_t spins = 0;
                    unsigned long long t_start = 0;
                    bool gave_up = false;
                    auto send = [&](uint32_t to_mask) {
#pragma unroll
                        for (uint32_t p = 0; p < kArMaxWorld; ++p) {
                            if (!((to_mask >> p) & 1u)) continue;
                            uint8_t *dst = args.ar_recv[p] + my_off;
#pragma unroll
                            for (int qd = 0; qd < 4; ++qd)
                                asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1, %2, %3, %2};" ::"l"(
                                                 dst + qd * 2048),
                                             "r"(res[2 * qd]), "r"(epoch), "r"(res[2 * qd + 1])
                                             : "memory");
                        }
                    };
                    // wait for packet row qd of the (up to four) ranks base .. base + 3 that are in
                    // from_mask; all loads of an attempt are in flight together (one L2 round
                    // trip per attempt).  Four at a time keeps the epilogue warps inside their
                    // 88 registers.
                    auto wait_row4 = [&](uint32_t from_mask, uint32_t base, int qd, uint32_t (&x)[4],
                                         uint32_t (&y)[4]) {
                        const uint8_t *src = rbase + (size_t)base * src_stride + qd * 2048;
                        for (;;) {
                            uint32_t fx[4], fy[4];
#pragma unroll
                            for (uint32_t i = 0; i < 4; ++i)
                                if ((from_mask >> (base + i)) & 1u)
                                    asm volatile("ld.relaxed.sys.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                                                 : "=r"(x[i]), "=r"(fx[i]), "=r"(y[i]), "=r"(fy[i])
                                                 : "l"(src + (size_t)i * src_stride)
                                                 : "memory");
                            bool ready = true;
#pragma unroll
                            for (uint32_t i = 0; i < 4; ++i)
                                if ((from_mask >> (base + i)) & 1u)
                                    ready = ready && fx[i] == epoch && fy[i] == epoch;
                            if (ready || gave_up) break;
                            if ((++spins & 0xff) == 0) {
                                unsigned long long now;
                                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                                if (t_start == 0) t_start = now;
                                if (now - t_start > args.watchdog_ns) {
                                    atomicExch(args.ar_state + 2, 1u);
                                    gave_up = true;
                                }
                            }
                        }
                    };
                    if (lead) trace_stamp(args, 11); // partial ready
                    // phase A: partial -> the row's reducer (two-shot) / every peer (one-shot)
                    if (!two_shot)
                        send(all_mask & ~me_bit);
                    else if (owner != args.ar_rank)
                        send(1u << owner);
                    if (lead) trace_stamp(args, 12);
                    if (owner == args.ar_rank) {
                        // phase B: reducer of this row (every thread in one-shot mode)
                        const uint32_t from = all_mask & ~me_bit;
#pragma unroll
                        for (int qd = 0; qd < 4; ++qd) {
                            float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
                            for (uint32_t base = 0; base < kArMaxWorld; base += 4) {
                                if (base >= args.ar_world) continue;
                                uint32_t x[4], y[4];
                                if ((from >> base) & 0xfu) wait_row4(from, base, qd, x, y);
#pragma unroll
                                for (uint32_t i = 0; i < 4; ++i) {
                                    const uint32_t p = base + i;
                                    if (p >= args.ar_world) continue;
                                    const uint32_t lo = p == args.ar_rank ? res[2 * qd] : x[i];
                                    const uint32_t hi = p == args.ar_rank ? res[2 * qd + 1] : y[i];
                                    if (C::kIsBf16) {
                                        s0 += __uint_as_float(lo << 16);
                                        s1 += __uint_as_float(lo & 0xffff0000u);
                                        s2 += __uint_as_float(hi << 16);
                                        s3 += __uint_as_float(hi & 0xffff0000u);
                                    } else {
                                        const __half2 h0 = *reinterpret_cast<const __half2 *>(&lo);
                                        const __half2 h1 = *reinterpret_cast<const __half2 *>(&hi);
                                        s0 += __low2float(h0);
                                        s1 += __high2float(h0);
                                        s2 += __low2float(h1);
                                        s3 += __high2float(h1);
                                    }
                                }
                            }
                            res[2 * qd] = (uint32_t)to_bits16<C::kIsBf16>(s0) |
                                          ((uint32_t)to_bits16<C::kIsBf16>(s1) << 16);
                            res[2 * qd + 1] = (uint32_t)to_bits16<C::kIsBf16>(s2) |
                                              ((uint32_t)to_bits16<C::kIsBf16>(s3) << 16);
                        }
                        if (lead) trace_stamp(args, 13); // all partials received and summed
                        if (two_shot) send(all_mask & ~me_bit); // the finished tile
                        if (lead) trace_stamp(args, 14);
                    } else {
                        // phase C: wait for the finished row from its reducer
                        const uint32_t base = owner & ~3u;
#pragma unroll
                        for (int qd = 0; qd < 4; ++qd) {
                            uint32_t x[4], y[4];
                            wait_row4(1u << owner, base, qd, x, y);
#pragma unroll
                            for (uint32_t i = 0; i < 4; ++i)
                                if (base + i == owner) {
                                    res[2 * qd] = x[i];
                                    res[2 * qd + 1] = y[i];
                                }
                        }
                        if (lead) trace_stamp(args, 14); // finished tile received
                    }
                    uint16_t *stg = reinterpret_cast<uint16_t *>(team_stage + out_buf * C::kOutStageBytes);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        stg[(2 * j) * kTileN + row] = (uint16_t)(res[j] & 0xffffu);
                        stg[(2 * j + 1) * kTileN + row] = (uint16_t)(res[j] >> 16);
                    }
                    fence_proxy_async();
                    if (ew_tid == 0) bulk_wait_group_read<C::kOutBufs - 2>();
                    named_bar_sync(team_bar, kNumEpilogueWarps * 32);
                    if (ew_tid == 0) {
                        tma_store_2d(&tmap_out, stg, (int)(g.n_tile * kTileN), (int)(m0 + c0));
                        bulk_commit_group();
                    }
                    out_buf = out_buf == C::kOutBufs - 1 ? 0 : out_buf + 1;
                } else if (args.act_silu_mul) {
                    // ---- fused SiLU(gate) * up (the MLP's gate_up projection; rows of every
                    // 128-row tile were interleaved at weight-load time: 0-63 gate, 64-127 the
                    // matching up rows).  Same arithmetic as the unfused path the frameworks run
                    // (GEMM output rounded to 16 bit, silu in fp32 rounded to 16 bit, product
                    // rounded to 16 bit), so the result is the same bits; output tile is
                    // [16 tokens][64 columns] of c[m, n / 2].
                    uint16_t *stg = reinterpret_cast<uint16_t *>(team_stage + out_buf * C::kOutStageBytes);
                    if (ew_tid == 0) bulk_wait_group_read<C::kOutBufs - 2>();
                    named_bar_sync(team_bar, kNumEpilogueWarps * 32); // buffer drained
                    if (row >= 64) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) stg[j * 64 + (row - 64)] = to_bits16<C::kIsBf16>(v[j]);
                    }
                    named_bar_sync(team_bar, kNumEpilogueWarps * 32); // up rows visible
                    uint16_t r16[16];
                    if (row < 64) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const uint16_t ub = stg[j * 64 + row];
                            const uint16_t gb = to_bits16<C::kIsBf16>(v[j]);
                            const float gf = C::kIsBf16 ? __uint_as_float((uint32_t)gb << 16)
                                                        : __half2float(__ushort_as_half(gb));
                            const float uf = C::kIsBf16 ? __uint_as_float((uint32_t)ub << 16)
                                                        : __half2float(__ushort_as_half(ub));
                            const uint16_t sb = to_bits16<C::kIsBf16>(gf / (1.0f + expf(-gf)));
                            const float sf = C::kIsBf16 ? __uint_as_float((uint32_t)sb << 16)
                                                        : __half2float(__ushort_as_half(sb));
                            r16[j] = to_bits16<C::kIsBf16>(sf * uf);
                        }
                    }
                    named_bar_sync(team_bar, kNumEpilogueWarps * 32); // up rows consumed
                    if (row < 64) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) stg[j * 64 + row] = r16[j];
                    }
                    fence_proxy_async();
                    named_bar_sync(team_bar, kNumEpilogueWarps * 32);
                    if (GR && m_valid - (uint32_t)c0 < 16u) {
                        // (grouped: the rows behind the group's last token are another group's)
                        const uint32_t j = ew_tid / 8, chunk = ew_tid % 8;
                        if ((uint32_t)c0 + j < m_valid)
                            *reinterpret_cast<uint4 *>(static_cast<uint16_t *>(args.c) +
                                                       (size_t)(m0 + c0 + j) * (args.n / 2) +
                                                       g.n_tile * 64 + chunk * 8) =
                                *reinterpret_cast<const uint4 *>(stg + j * 64 + chunk * 8);
                    } else if (ew_tid == 0) {
                        // tmap_out describes c[m, n / 2] with [16][64] boxes in this mode
                        tma_store_2d(&tmap_out, stg, (int)(g.n_tile * 64), (int)(m0 + c0));
                        bulk_commit_group();
                    }
                    out_buf = out_buf == C::kOutBufs - 1 ? 0 : out_buf + 1;
                } else if (!PETIT_DBG(args.debug_flags, 64u)) {
                    // [16 tokens][128 rows] 16-bit staging tile -> one TMA store; the tensor
                    // map clips tokens >= M and rows >= N.  Three buffers in rotation: the
                    // wait below (before the barrier) leaves only the previous group's store
                    // in flight, so the buffer the NEXT group fills is known to be drained.
                    uint16_t *stg = reinterpret_cast<uint16_t *>(team_stage + out_buf * C::kOutStageBytes);
#pragma unroll
                    for (int j = 0; j < 16; ++j) stg[j * kTileN + row] = to_bits16<C::kIsBf16>(v[j]);
                    if (!PETIT_DBG(args.debug_flags, 256u)) fence_proxy_async();
                    if (ew_tid == 0 && !PETIT_DBG(args.debug_flags, 128u))
                        bulk_wait_group_read<C::kOutBufs - 2>();
                    named_bar_sync(team_bar, kNumEpilogueWarps * 32);
                    if (GR && m_valid - (uint32_t)c0 < 16u) {
                        // the rows behind a group's last token belong to the next group: no
                        // TMA box here, 16-byte stores of the valid tokens only (a thread takes
                        // chunk ew_tid % 16 of tokens ew_tid / 16 and + 8)
                        const uint32_t chunk = ew_tid % 16;
#pragma unroll
                        for (uint32_t j = ew_tid / 16; j < 16; j += 8)
                            if ((uint32_t)c0 + j < m_valid && chunk * 8 < rows)
                                *reinterpret_cast<uint4 *>(
                                    static_cast<uint16_t *>(args.c) + (size_t)(m0 + c0 + j) * args.n +
                                    g.n_tile * kTileN + chunk * 8) =
                                    *reinterpret_cast<const uint4 *>(stg + j * kTileN + chunk * 8);
                    } else if (ew_tid == 0 && !PETIT_DBG(args.debug_flags, 512u)) {
                        tma_store_2d(&tmap_out, stg, (int)(g.n_tile * kTileN), (int)(m0 + c0));
                        bulk_commit_group();
                    }
                    out_buf = out_buf == C::kOutBufs - 1 ? 0 : out_buf + 1;
                }
                if (lead && last_seg && c0 == 0) trace_stamp(args, 15);
            }
            // accumulator drained -> MMA may reuse it
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->acc_empty[acc]);
            if (lead && seg == 1) trace_stamp(args, 10); // ... and end

            if (is_contrib) {
                // publish: CTA barrier, then one release-increment of the tile counter
                named_bar_sync(kEpilogueBarId, kAllEpiThreads);
                if (lead)
                    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(
                                     args.ws_counters + out_tile)
                                 : "memory");
            } else if (is_reducer) {
                named_bar_sync(kEpilogueBarId, kAllEpiThreads);
                if (lead) args.ws_counters[out_tile] = 0; // self-cleaning
            }
            u += g.kt1 - g.kt0;
        }
        // staging smem must outlive the read of this team's last TMA store
        if (ew_tid == 0) bulk_wait_group_read<0>();
    }

    if (threadIdx.x == kFirstEpilogueWarp * 32) trace_stamp(args, 7);
    tc_fence_before();
    if (CL)
        cluster_sync(); // the peer may still multicast into / arrive on this CTA's smem
    else
        __syncthreads();
    if (threadIdx.x == 0) trace_stamp(args, 8);
    if (warp == kMmaWarp) tmem_dealloc(tmem, 512);
    // fused all-reduce: the last CTA to exit advances the call counter (every CTA read it at its
    // start; the next launch reads it after this grid has completed), modulo kArCallPeriod so
    // that the epoch (counter + 1) is never 0 -- see the packet format above
    if (AR && threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(args.ar_state + 1, 1u) == gridDim.x - 1) {
            args.ar_state[1] = 0;
            const uint32_t next = args.ar_state[0] + 1;
            args.ar_state[0] = next == kArCallPeriod ? 0u : next;
        }
    }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                  const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) !=
                cudaSuccess ||
            qres != cudaDriverEntryPointSuccess)
            return nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// Stream-K range cuts (decode tiles): equal ranges do not finish together, for two reasons.
//  (1) Roles.  A CTA whose whole range lies inside one output tile publishes its partial at the
//      very end of its run -- exactly when the CTA that reduces the tile (the owner of the tile's
//      first k-part, which meets the tile LAST) wants it: the reducer then sits through publish
//      + poll + read (~2 us, most of the tail of qkv / o / down at M <= 16).
//  (2) Arrival.  Behind another grid (programmatic dependent launch) the CTAs become resident in
//      block-id order over ~3 us as the previous grid drains; until griddepcontrol.wait returns
//      they dequantise ahead (smem ring + TMEM A stages = ~4.5 units), so the last block ids
//      start with up to that much less done and finish last (profiles/r02_percta_summary.txt:
//      dequant_done +0.5 / +0.9 / +1.9 us for block ids 112.. / 128.. / 144.. on qkv).
// Model (quarter units): CTA i starts at start[i] = late * profile(i / grid), a unit costs 1,
// a partial is usable `lat` units after its segment ended.  The cuts start from the
// water-filling solution for start[] and a local search over single-unit moves of the cut
// points minimises the largest modelled finish time (then the sum of squares).  Result cached
// per (units, k_tiles, grid, lat, late); adj[b] = cut[b] - units * b / grid.
// PETIT_TILT_UNITS / PETIT_TILT_LATE (units; 0 = off) override lat / late.
struct CutKey {
    uint32_t units, k_tiles, grid;
    int lat, late;
    bool operator<(const CutKey &o) const {
        return std::tie(units, k_tiles, grid, lat, late) <
               std::tie(o.units, o.k_tiles, o.grid, o.lat, o.late);
    }
};
struct CutAdj { int8_t v[kMaxGrid + 4]; };

// share of the head start a CTA at relative block id r lacks (measured, see above)
double late_profile(double r) {
    const double xs[] = {0.0, 0.6, 0.8, 0.92, 1.0}, ys[] = {0.0, 0.0, 0.2, 0.5, 1.0};
    for (int i = 1; i < 5; ++i)
        if (r <= xs[i]) return ys[i - 1] + (ys[i] - ys[i - 1]) * (r - xs[i - 1]) / (xs[i] - xs[i - 1]);
    return 1.0;
}

void tilt_cuts(uint32_t units, uint32_t k_tiles, uint32_t grid, int lat, int late, int8_t *adj) {
    static std::mutex mu;
    static std::map<CutKey, CutAdj> cache;
    const CutKey key{units, k_tiles, grid, lat, late};
    {
        std::lock_guard<std::mutex> lock(mu);
        auto it = cache.find(key);
        if (it != cache.end()) {
            std::memcpy(adj, it->second.v, sizeof(it->second.v));
            return;
        }
    }
    constexpr int64_t Q = 4; // model resolution: quarter units
    std::vector<int64_t> base(grid + 1), cut(grid + 1), start(grid), fin(grid), pre(grid + 1), suf(grid + 2);
    for (uint32_t b = 0; b <= grid; ++b) base[b] = (int64_t)((uint64_t)units * b / grid);
    double start_sum = 0;
    for (uint32_t i = 0; i < grid; ++i) {
        start[i] = (int64_t)(Q * late * late_profile((i + 0.5) / grid) + 0.5);
        start_sum += (double)start[i];
    }
    {   // water filling: everybody finishes at `level`
        const double level = ((double)Q * units + start_sum) / grid;
        double acc = 0;
        cut[0] = 0;
        for (uint32_t i = 0; i < grid; ++i) {
            acc += (level - (double)start[i]) / Q;
            int64_t c = (int64_t)(acc + 0.5);
            c = std::max(c, cut[i] + 1);                                  // >= 1 unit each
            c = std::min(c, (int64_t)units - (int64_t)(grid - 1 - i));     // ... also for the rest
            c = std::min(std::max(c, base[i + 1] - 100), base[i + 1] + 100);
            cut[i + 1] = c;
        }
        cut[grid] = units;
    }
    const int64_t lat_q = Q * lat;
    // modelled finish time of CTA i
    auto fin_of = [&](uint32_t i) {
        const int64_t len = cut[i + 1] - cut[i];
        int64_t f = start[i] + Q * len;
        if (len > 0 && lat > 0) {
            const int64_t head = (cut[i + 1] - 1) / k_tiles * k_tiles, tile_end = head + k_tiles;
            if (head >= cut[i] && tile_end > cut[i + 1]) // reducer of a tile that goes on
                for (uint32_t j = i + 1; j < grid && cut[j] < tile_end; ++j) {
                    const int64_t seg_end = (cut[j + 1] < tile_end ? cut[j + 1] : tile_end) - cut[j];
                    f = std::max(f, start[j] + Q * seg_end + lat_q);
                }
        }
        return f;
    };
    for (int iter = 0; iter < 400; ++iter) {
        int64_t worst = 0, sumsq = 0, min_len = units;
        for (uint32_t i = 0; i < grid; ++i) {
            fin[i] = fin_of(i);
            sumsq += fin[i] * fin[i];
            min_len = std::min(min_len, cut[i + 1] - cut[i]);
        }
        pre[0] = 0;
        for (uint32_t i = 0; i < grid; ++i) pre[i + 1] = std::max(pre[i], fin[i]);
        suf[grid] = suf[grid + 1] = 0;
        for (uint32_t i = grid; i-- > 0;) suf[i] = std::max(suf[i + 1], fin[i]);
        worst = pre[grid];
        // moving cut b changes CTAs b - 1 and b and the reducers that count them as contributors:
        // at most `span` CTAs back
        const uint32_t span = (uint32_t)std::min<int64_t>(grid, k_tiles / std::max<int64_t>(min_len, 1) + 2);
        int best_b = -1, best_d = 0;
        int64_t bw = worst, bs = sumsq;
        for (uint32_t b = 1; b < grid; ++b)
            for (int d = -1; d <= 1; d += 2) {
                const int64_t nc = cut[b] + d;
                if (nc < cut[b - 1] + 1 || nc > cut[b + 1] - 1 || nc - base[b] > 100 || nc - base[b] < -100)
                    continue;
                const uint32_t lo = b > span ? b - span : 0;
                cut[b] = nc;
                int64_t w = std::max(pre[lo], suf[b + 1]), sq = sumsq;
                for (uint32_t i = lo; i <= b; ++i) {
                    const int64_t f = fin_of(i);
                    w = std::max(w, f);
                    sq += f * f - fin[i] * fin[i];
                }
                cut[b] = nc - d;
                if (w < bw || (w == bw && sq < bs)) {
                    bw = w;
                    bs = sq;
                    best_b = (int)b;
                    best_d = d;
                }
            }
        if (best_b < 0) break;
        cut[best_b] += best_d;
    }
    CutAdj out;
    std::memset(out.v, 0, sizeof(out.v));
    for (uint32_t b = 0; b <= grid; ++b) out.v[b] = (int8_t)(cut[b] - base[b]);
    std::memcpy(adj, out.v, sizeof(out.v));
    std::lock_guard<std::mutex> lock(mu);
    cache[key] = out;
}

template <int MODE, int NTOK, int KS, bool CL = false, bool AR = false, bool GR = false>
int launch_variant(const GemmArgs &args, int num_sms, cudaStream_t stream,
                   const GroupTable *table = nullptr) {
    using C = Cfg<MODE, NTOK, KS>;
    EncodeTiledFn encode = get_encode_fn();
    if (!encode) return kLaunchCudaError;

    // activations [M, K] 16-bit row-major viewed as (64, M, K/64)
    CUtensorMap tmap;
    const cuuint64_t dims[3] = {64, args.m, args.k / 64};
    const cuuint64_t strides[2] = {(cuuint64_t)args.k * 2, 128};
    const cuuint32_t box[3] = {64, (cuuint32_t)(CL ? NTOK / 2 : NTOK), (cuuint32_t)(CL ? 1 : C::kSubs)};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = encode(&tmap,
                        C::kIsBf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                   : CU_TENSOR_MAP_DATA_TYPE_FLOAT16,
                        3, const_cast<void *>(args.a), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return kLaunchCudaError;
    // output [M, N] 16-bit row-major; the epilogue stores [16 tokens][128 rows] boxes
    CUtensorMap tmap_out;
    // (fused SiLU * mul: c is [M, N / 2] and a tile stores a [16 tokens][64 columns] box)
    const cuuint64_t out_n = args.act_silu_mul ? args.n / 2 : args.n;
    const cuuint64_t odims[2] = {out_n, args.m};
    const cuuint64_t ostrides[1] = {out_n * 2};
    const cuuint32_t obox[2] = {args.act_silu_mul ? 64u : kTileN, 16};
    r = encode(&tmap_out, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, args.c, odims, ostrides, obox, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
               CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return kLaunchCudaError;

    static std::atomic<bool> attr_set[64]; // per instantiation, per device (zero-initialised)
    auto kern = fp4_gemm_kernel<MODE, NTOK, KS, CL, AR, GR>;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return kLaunchCudaError;
    if (!attr_set[dev & 63].load(std::memory_order_acquire)) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 C::kSmemBytes) != cudaSuccess)
            return kLaunchCudaError;
        attr_set[dev & 63].store(true, std::memory_order_release);
    }
    const uint64_t n_tiles = (args.n + kTileN - 1) / kTileN;
    const uint64_t m_tiles = GR ? table->tiles : (args.m + NTOK - 1) / NTOK;
    const uint64_t units = (CL ? n_tiles / 2 : n_tiles) * m_tiles * (args.k / kTileK);
    unsigned grid = (unsigned)(units < (uint64_t)num_sms ? units : (uint64_t)num_sms);
    bool whole_tiles = false; // one whole tile per CTA: the cuts must stay on tile boundaries
    // Small shards (TP-8 o_proj: 64 tiles x 4 k-tiles on 148 SMs): with < ~2 units per SM every
    // tile would be cut between CTAs that all finish together, and the split-tile hand-shake
    // (~2 us) would be most of the launch.  One whole tile per CTA on fewer SMs is faster there
    // (PETIT_WHOLE_TILES=0 turns the rule off for A/B runs).
    if (!CL && NTOK <= 64) {
        static const int whole = [] {
            const char *e = std::getenv("PETIT_WHOLE_TILES");
            return e ? std::atoi(e) : 1;
        }();
        const uint64_t tiles = n_tiles * m_tiles, k_tiles = args.k / kTileK;
        if (whole && tiles <= (uint64_t)num_sms && tiles * 3 >= (uint64_t)num_sms && k_tiles <= 6) {
            grid = (unsigned)tiles;
            whole_tiles = true;
        }
    }
    if (CL) {
        const uint64_t clusters = units < (uint64_t)(num_sms / 2) ? units : (uint64_t)(num_sms / 2);
        grid = (unsigned)clusters * 2;
    }
    if (m_tiles * n_tiles > kMaxTiles || grid > kMaxGrid || units >= (1ull << 31))
        return kLaunchBadShape;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kNumThreads);
    cfg.dynamicSmemBytes = C::kSmemBytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = args.use_pdl ? 1 : 0;
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = 2;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = CL ? 2 : 1;
    GemmArgs largs = args;
    std::memset(largs.cut_adj, 0, sizeof(largs.cut_adj));
    // Not for whole-tile grids, and not for small shards (< 8 units per CTA): there the model's
    // few units of latency are most of a range, and the TP-8 step got slower with it (o_proj +
    // all-reduce 24 -> 38 us when its whole-tile grid was cut up again).
    if (!CL && NTOK <= 64 && grid > 1 && !whole_tiles && units >= 8ull * grid) {
        static const int lat_env = [] {
            const char *e = std::getenv("PETIT_TILT_UNITS");
            return e ? std::atoi(e) : -1;
        }();
        static const int late_env = [] {
            const char *e = std::getenv("PETIT_TILT_LATE");
            return e ? std::atoi(e) : -1;
        }();
        const int lat = lat_env >= 0 ? lat_env : (NTOK <= 32 ? 5 : 3);
        // the head start is worth ~4.5 units of a 16-token tile; only launches chained by
        // programmatic dependent launch see it
        // (the arrival term is only measured for plain GEMMs: none under the fused all-reduce)
        const int late = (!args.use_pdl || AR) ? 0 : (late_env >= 0 ? late_env : (NTOK <= 32 ? 4 : 3));
        if (lat > 0 || late > 0)
            tilt_cuts((uint32_t)units, (uint32_t)(args.k / kTileK), grid, lat, late, largs.cut_adj);
    }
    cudaError_t e;
    if constexpr (GR)
        e = cudaLaunchKernelEx(&cfg, kern, tmap, tmap_out, largs, *table);
    else
        e = cudaLaunchKernelEx(&cfg, kern, tmap, tmap_out, largs, NoGroups{});
    return e == cudaSuccess ? kLaunchOk : kLaunchCudaError;
}

template <int MODE> int launch_grouped_mode(const GemmArgs &args, int ntok, const GroupTable &table,
                                            int num_sms, cudaStream_t stream) {
    switch (ntok) {
    case 16: return launch_variant<MODE, 16, 256, false, false, true>(args, num_sms, stream, &table);
    case 32: return launch_variant<MODE, 32, 256, false, false, true>(args, num_sms, stream, &table);
    case 64: return launch_variant<MODE, 64, PETIT_KS_64, false, false, true>(args, num_sms, stream, &table);
    default: return kLaunchNoKernel;
    }
}

template <int MODE> int launch_mode(const GemmArgs &args, int ntok, int num_sms,
                                    cudaStream_t stream) {
    // 2-CTA multicast clusters need an even number of n-tiles (pairs) and enough tokens
    // for the shared tile to matter
    const uint32_t n_tiles = (args.n + kTileN - 1) / kTileN;
    const bool cluster_ok = args.use_cluster && n_tiles % 2 == 0 && args.n % kTileN == 0;
    if (args.ar_world > 1) { // fused all-reduce: decode tiles only (m <= 64, checked by the C ABI)
        switch (ntok) {
        case 16: return launch_variant<MODE, 16, 256, false, true>(args, num_sms, stream);
        case 32: return launch_variant<MODE, 32, 256, false, true>(args, num_sms, stream);
        case 64: return launch_variant<MODE, 64, PETIT_KS_64, false, true>(args, num_sms, stream);
        default: return kLaunchNoKernel;
        }
    }
    switch (ntok) {
    case 16: return launch_variant<MODE, 16, 256>(args, num_sms, stream);
    case 32: return launch_variant<MODE, 32, 256>(args, num_sms, stream);
    case 64: return launch_variant<MODE, 64, PETIT_KS_64>(args, num_sms, stream);
    case 128:
        return cluster_ok ? launch_variant<MODE, 128, 128, true>(args, num_sms, stream)
                          : launch_variant<MODE, 128, 128>(args, num_sms, stream);
    case 256:
        return cluster_ok ? launch_variant<MODE, 256, 64, true>(args, num_sms, stream)
                          : launch_variant<MODE, 256, 64>(args, num_sms, stream);
    default: return kLaunchNoKernel;
    }
}

} // namespace

void debug_stream_k_cuts(uint32_t units, uint32_t k_tiles, uint32_t grid, int lat, int late,
                          int8_t *adj) {
    std::memset(adj, 0, kMaxGrid + 4);
    if (lat > 0 || late > 0) tilt_cuts(units, k_tiles, grid, lat, late, adj); // as the launcher
}

size_t workspace_partials_bytes() {
    return (size_t)kMaxGrid * kTileN * 256 * sizeof(float);
}
size_t workspace_counters_bytes() { return ((size_t)kMaxTiles + 1) * sizeof(unsigned); }

int launch_grouped(int mode, int ntok, const GemmArgs &args, const GroupTable &table, int num_sms,
                   cudaStream_t stream) {
    if (table.tiles == 0 || table.tiles > kMaxGroupTiles || args.ar_world > 1 || args.bias ||
        args.residual)
        return kLaunchBadShape;
    switch (mode) {
    case kModeNvF16: return launch_grouped_mode<kModeNvF16>(args, ntok, table, num_sms, stream);
    case kModeNvBf16: return launch_grouped_mode<kModeNvBf16>(args, ntok, table, num_sms, stream);
    case kModeMxBf16: return launch_grouped_mode<kModeMxBf16>(args, ntok, table, num_sms, stream);
    case kModeNvF16N: return launch_grouped_mode<kModeNvF16N>(args, ntok, table, num_sms, stream);
    default: return kLaunchNoKernel;
    }
}

int launch(int mode, int ntok, const GemmArgs &args, int num_sms, cudaStream_t stream) {
    switch (mode) {
    case kModeNvF16: return launch_mode<kModeNvF16>(args, ntok, num_sms, stream);
    case kModeNvBf16: return launch_mode<kModeNvBf16>(args, ntok, num_sms, stream);
    case kModeMxBf16: return launch_mode<kModeMxBf16>(args, ntok, num_sms, stream);
    case kModeNvF16N: return launch_mode<kModeNvF16N>(args, ntok, num_sms, stream);
    default: return kLaunchNoKernel;
    }
}

} // namespace petit::gemm
