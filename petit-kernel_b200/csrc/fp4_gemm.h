// Internal interface between the C ABI (capi.cu) and the GEMM kernels.
#pragma once

#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace petit::gemm {

// kModeNvF16N: fp16 activations on weights repacked in the fp16-native layout (native nibble
// order inside a word: cvt.rn.f16x2.e2m1x2 converts a pair with one instruction).
enum : int { kModeNvF16 = 0, kModeNvBf16 = 1, kModeMxBf16 = 2, kModeNvF16N = 3 };
enum : int { kLaunchOk = 0, kLaunchBadShape = 1, kLaunchNoKernel = 2, kLaunchCudaError = 3 };

constexpr unsigned kMaxGrid = 160;         // >= SM count of any sm_100 part
constexpr unsigned kMaxTiles = 1u << 20;   // (n-tiles x token-tiles) upper bound

struct GemmArgs {
    const void *a;          // [m, k] 16-bit row-major
    const uint8_t *w;       // packed fp4 (layout.cuh)
    const uint8_t *sc;      // packed scales
    const float *global_scale; // device pointer
    void *c;                // [m, n] 16-bit row-major
    const void *bias;       // optional [n] in the output type: added in fp32 before rounding
    const void *residual;   // optional [m, n] in the output type: added in fp32 before rounding
    uint32_t act_silu_mul;  // 1: rows 0-63 of every n-tile are gate rows, 64-127 the matching up
                            // rows; c is [m, n / 2] = silu(gate) * up
    float *ws_partials;     // stream-K partial tiles
    unsigned *ws_counters;  // per-tile arrival counters (zero between launches)
    unsigned *ws_status;    // sticky: != 0 once a split-tile reducer gave up waiting (watchdog)
    unsigned long long watchdog_ns; // how long a reducer polls for its contributors
    uint32_t m, n, k;
    uint32_t debug_flags;   // experiments only (PETIT_DEBUG_FLAGS); 0 in production
    uint32_t use_cluster;   // allow the 2-CTA multicast variant for 128/256-token tiles
    uint32_t use_pdl;       // launch with programmatic stream serialisation
    uint32_t skew_cycles;   // initial phase skew between k-slice warps (tuning knob)
    unsigned long long *trace; // optional [grid][16] globaltimer stamps (debug), else null
    // Stream-K range cuts: CTA b owns units [total * b / grid + cut_adj[b], total * (b + 1) / grid
    // + cut_adj[b + 1]).  All zero = equal ranges; the launcher shortens the ranges of CTAs that a
    // split-tile reducer would otherwise wait for (fp4_gemm.cu, tilt_cuts).
    int8_t cut_adj[kMaxGrid + 4];
    // Fused all-reduce of a row-parallel (K-split) GEMM over NVLink peer memory (ar_world > 1):
    // the CTA that finishes an output tile pushes its 16-bit partial to every peer's receive
    // buffer as self-validating {data, epoch} packets and sums the peers' packets of the same
    // tile in rank order before it stores the tile (see fp4_gemm.cu, "fused all-reduce").
    uint32_t ar_world, ar_rank;
    uint32_t ar_two_shot;      // 0: every rank sums every row; 1: row r of a tile is reduced by
                               //    rank r / (128 / world)
    uint8_t *ar_recv[8];       // rank p's receive buffer as mapped in this process
    unsigned *ar_state;        // local device words: [0] call counter (epoch - 1), [1] exited-CTA
                               // counter, [2] status
};

// Receive-buffer geometry of the fused all-reduce: [parity 2][source rank 8][slot][8 KB], one slot
// per (n-tile, 16-token group); at most 64 tokens.
constexpr unsigned kArMaxWorld = 8;
constexpr unsigned kArMaxTokens = 64;
constexpr unsigned kArSlotBytes = 8192;
// The call counter ar_state[0] wraps at this (even) period, so the epoch is never 0.
constexpr unsigned kArCallPeriod = 0xFFFFFFFEu;
inline size_t ar_recv_bytes(unsigned n) {
    return (size_t)2 * kArMaxWorld * ((n + 127) / 128) * (kArMaxTokens / 16) * kArSlotBytes;
}

// Grouped (MoE) GEMM in one launch: the activations / outputs of all groups are the row
// blocks of ONE [total_rows, k] / [total_rows, n] tensor (tokens sorted by expert), and the
// unit space of the stream-K schedule runs over the token tiles of all groups; entry t says
// which rows token tile t covers and whose weights it multiplies.
struct GroupEntry {
    const uint8_t *w;   // packed weights of the tile's group
    const uint8_t *sc;  // packed scales
    const float *gs;    // the group's global scale (device)
    uint32_t row0;      // first row of the tile in the concatenated activations / output
    uint32_t rows;      // valid rows (1 .. ntok)
};
constexpr unsigned kMaxGroupTiles = 96; // 3 KB of kernel parameters
struct GroupTable {
    uint32_t tiles;
    uint32_t pad;
    GroupEntry e[kMaxGroupTiles];
};

// test hook: the range cuts the launcher would use; adj must hold kMaxGrid + 4 entries
void debug_stream_k_cuts(uint32_t units, uint32_t k_tiles, uint32_t grid, int lat, int late,
                         int8_t *adj);

size_t workspace_partials_bytes();
size_t workspace_counters_bytes(); // kMaxTiles counters + the status word (last)

// ntok: tokens per MMA (16, 32, 64, 128, 256).
int launch(int mode, int ntok, const GemmArgs &args, int num_sms, cudaStream_t stream);
// args.a / args.c: the concatenated tensors, args.m: their rows; args.w / sc / global_scale
// are ignored (per tile in `table`); ntok 16, 32 or 64; SiLU * mul is the only fused epilogue
// (no bias / residual: they would be per group), no all-reduce.
int launch_grouped(int mode, int ntok, const GemmArgs &args, const GroupTable &table, int num_sms,
                   cudaStream_t stream);

} // namespace petit::gemm
