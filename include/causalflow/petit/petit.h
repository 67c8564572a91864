/*
 * petit.h -- C ABI of the B200 (sm_100a) FP4-weight x 16-bit-activation GEMM.
 *
 * This is the drop-in boundary.  Every entry point replaces one function of the
 * reference's C++ API (all citations into /root/reference):
 *
 *   petit_gemm_nvfp4_a16        <- fp4::GemmFp4Fp16Grid      lib/gemm/rocm/quantization/gemm.h:120-124
 *   petit_gemm_mxfp4_a16        <- fp4::GemmMxFp4Fp16Grid    gemm.h:126-130
 *   petit_get_solutions         <- fp4::GemmGetSolutions     gemm.h:132-133
 *   petit_get_default_solution  <- fp4::ChooseDefaultFp4Fp16Solution  fp4/algo_chooser.cc:64-132
 *   petit_tune_table_*          (feeds `bench_matmul -algo tune` results, tools/benchmarks/matmul/main.cc:269-325,
 *                                back to the default chooser; no reference equivalent)
 *   petit_repack_fp4_weights    <- fp4::RepackNvFp4ToPetitFp4Weights  gemm.h:135-137
 *   petit_repack_nvfp4_scales   <- fp4::RepackNvFp4ToPetitFp4Scales   gemm.h:139-141
 *   petit_repack_mxfp4_scales   <- fp4::RepackMxFp4ToPetitFp4Scales   gemm.h:143-145
 *   petit_dequant_nvfp4         <- fp4::DequantNvFp4         fp4/quantization_utils.cu:614-645
 *   petit_dequant_mxfp4         <- fp4::DequantMxFp4         fp4/gemm_fp4.h:19-21
 *   petit_dequant_packed_nvfp4  <- fp4::DequantPetitFp4      fp4/gemm_fp4.h:11-13
 *   petit_dequant_packed_mxfp4  <- fp4::DequantPetitMxFp4    fp4/gemm_fp4.h:15-17
 *   petit_unpack_fp4_weights    (inverse of the repack; round-trip test hook, no reference equivalent)
 *   petit_hal_*                 <- hal::Device               lib/hal/device.h:8-34
 *
 * Differences from the reference, all deliberate:
 *   - hipStream_t -> cudaStream_t; `unsigned*` payload pointers -> `void*`.
 *   - the repack functions return an int status (the reference returns void and
 *     never checks the launch, gemm.h:135-145).
 *   - the packed layouts are Blackwell tile layouts (see DESIGN.md); they are
 *     opaque to callers exactly as the reference's are.
 *   - the GEMM moves every operand with TMA: the activation, output, packed weight
 *     and packed scale base addresses must be 16-byte aligned (else
 *     PETIT_ERROR_PROBLEM_SHAPE); rows need no padding.
 *
 * Semantics kept from the reference:
 *   - return 0 on success, PETIT_ERROR_PROBLEM_SHAPE (1), PETIT_ERROR_KERNEL_SHAPE (2)
 *     (gemm.h:107-108); petit_get_solutions returns -1 for an unsupported b_type
 *     (fp4/algo_chooser.cc:20-23); the dequant hooks return -1 on a bad shape or
 *     type (fp4/quantization_utils.cu:619-621,642).
 *   - m == 0 || n == 0 || k == 0 is a successful no-op (fp4/gemm_fp4_fp16_grid.cc:42-44).
 *   - solution_id == (uint64_t)-1 selects the default solution
 *     (fp4/gemm_fp4_fp16_grid.cc:46-52); other values must come from
 *     petit_get_solutions.
 *   - global_scale is a DEVICE pointer, dereferenced inside the kernel
 *     (fp4/gemm_fp4_fp16_grid.cuh:469-470): no host sync, CUDA-graph safe.
 *   - everything is asynchronous on the caller's stream; the library owns no
 *     streams.  MXFP4 requires bf16 activations/outputs
 *     (fp4/gemm_fp4_fp16_grid.cc:60-63).
 *
 * There is no CPU fallback: every function fails (nonzero / CUDA error) when no
 * sm_100 device is present.
 */
#ifndef CAUSALFLOW_PETIT_PETIT_H_
#define CAUSALFLOW_PETIT_PETIT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* cudaStream_t without pulling in the CUDA headers. */
typedef struct CUstream_st *petit_stream_t;

/* Same enumerators, same values as the reference's C++ DataType
 * (lib/gemm/rocm/quantization/types.h:4-13). */
typedef enum PetitDataType {
    PETIT_DTYPE_INT4 = 0,
    PETIT_DTYPE_FP8_E4M3 = 1,
    PETIT_DTYPE_FP8_E8M0 = 2,
    PETIT_DTYPE_FP4_E2M1 = 3,
    PETIT_DTYPE_FP16 = 4,
    PETIT_DTYPE_BF16 = 5,
    PETIT_DTYPE_FP8_E5M2_FNUZ = 6,
    PETIT_DTYPE_MXFP4_E2M1 = 7
} PetitDataType;

/* gemm.h:107-108 */
#define PETIT_OK 0
#define PETIT_ERROR_PROBLEM_SHAPE 1
#define PETIT_ERROR_KERNEL_SHAPE 2
/* Not in the reference: a CUDA runtime/driver failure (launch error, no device). */
#define PETIT_ERROR_CUDA 3

/* gemm.h:112-117.  require_high_precision is the gfx90a denormal workaround
 * (lib/pybind/fp4.cc:24-34); it is accepted and ignored on B200, where the one
 * code path is exact. */
typedef struct PetitSolutionHints {
    int32_t a_type; /* PetitDataType: FP16 or BF16 */
    int32_t b_type; /* PetitDataType: FP4_E2M1 (NVFP4) or MXFP4_E2M1 */
    int32_t c_type; /* PetitDataType: must equal a_type */
    int32_t require_high_precision;
} PetitSolutionHints;

#define PETIT_SOLUTION_AUTO ((uint64_t)-1)

/* C[m,n] (a_type) = A[m,k] (a_type, row-major) x dequant(B)[n,k]^T x *global_scale.
 * b / scales are the outputs of petit_repack_fp4_weights / petit_repack_nvfp4_scales.
 * Requires k % 256 == 0 and n % 16 == 0 (lib/pybind/fp4.cc:40-43,82-86).
 * Ordering: the GEMM is launched with programmatic dependent launch and starts streaming
 * b / scales while the previous kernel on the stream drains; a, global_scale and c are
 * touched only after that kernel has completed.  b / scales must therefore be complete before
 * the kernel that precedes the GEMM on the stream was launched -- true for weights, which
 * are constants; a GEMM that directly follows a petit_repack_* call on the same stream is
 * ordered behind it by the library; anything else that rewrites weights immediately before a
 * GEMM sets PETIT_PDL=0. */
int petit_gemm_nvfp4_a16(void *c, const void *a, const void *b, const void *scales,
                         const float *global_scale_dev, unsigned m, unsigned n, unsigned k,
                         const PetitSolutionHints *hints, uint64_t solution_id,
                         petit_stream_t stream);

/* Same for MXFP4 (group-32 e8m0 scales from petit_repack_mxfp4_scales); bf16 only. */
int petit_gemm_mxfp4_a16(void *c, const void *a, const void *b, const void *scales,
                         const float *global_scale_dev, unsigned m, unsigned n, unsigned k,
                         const PetitSolutionHints *hints, uint64_t solution_id,
                         petit_stream_t stream);

/* Two-call enumeration (fp4/algo_chooser.cc:14-62): sols may be NULL; *n_sols is the
 * capacity on entry (ignored when sols is NULL) and the number of applicable
 * solutions on return.  The values are SolutionId::Repr()-style 64-bit ids. */
int petit_get_solutions(const PetitSolutionHints *hints, unsigned m, unsigned n, unsigned k,
                        uint64_t *sols, unsigned *n_sols);

/* The solution a GEMM call with solution_id == PETIT_SOLUTION_AUTO uses for this problem: the
 * tuned-solution table first, then the built-in rule (the role of
 * ChooseDefaultFp4Fp16Solution, fp4/algo_chooser.cc:64-132).  Pure host code; returns 0,
 * PETIT_ERROR_PROBLEM_SHAPE for shapes/types no kernel takes, -1 for an unsupported b_type. */
int petit_get_default_solution(const PetitSolutionHints *hints, unsigned m, unsigned n,
                               unsigned k, uint64_t *solution_id);

/* Tuned-solution table (SURVEY section 8 row f1: what `bench_matmul -algo tune` finds, fed
 * back to the default chooser; the reference's README tells users to autotune but gives the
 * result nowhere to live).  An entry applies to an exact (a_type, b_type, m, n, k).
 *   petit_tune_table_set    add / replace one entry; solution_id must come from
 *                           petit_get_solutions for the same hints (else
 *                           PETIT_ERROR_KERNEL_SHAPE); PETIT_SOLUTION_AUTO removes the entry
 *   petit_tune_table_load   text file, one entry per line:
 *                           "<nvfp4|mxfp4> <bf16|fp16> <m> <n> <k> <16 hex digits>" (the id as
 *                           bench_matmul prints it: its 8 bytes, little endian); '#' starts a
 *                           comment.  Returns the number of entries read, -1 if the file
 *                           cannot be read or a line is malformed (nothing is added then).
 *   petit_tune_table_clear  forget everything (also what was loaded from $PETIT_TUNE_TABLE,
 *                           which is read once, before the first lookup). */
int petit_tune_table_set(const PetitSolutionHints *hints, unsigned m, unsigned n, unsigned k,
                         uint64_t solution_id);
int petit_tune_table_load(const char *path);
void petit_tune_table_clear(void);

/* in: u32 [out_chan, in_chan/8] row-major, nibble i of a word = element 8w+i;
 * out: in_chan*out_chan/2 bytes in the packed tile layout. */
int petit_repack_fp4_weights(uint32_t *out, const uint32_t *in, unsigned in_chan,
                             unsigned out_chan, petit_stream_t stream);
int petit_unpack_fp4_weights(uint32_t *out, const uint32_t *in_packed, unsigned in_chan,
                             unsigned out_chan, petit_stream_t stream);

/* in: e4m3 bytes [out_chan, in_chan/16]; out: same byte count, tile layout, each
 * byte re-encoded as unsigned E5M3 (exact for every positive finite e4m3). */
int petit_repack_nvfp4_scales(void *out, const void *in, unsigned in_chan, unsigned out_chan,
                              petit_stream_t stream);
/* in: e8m0 bytes [out_chan, in_chan/32]; out: same bytes, tile layout. */
int petit_repack_mxfp4_scales(void *out, const void *in, unsigned in_chan, unsigned out_chan,
                              petit_stream_t stream);

/* Dense dequantisation hooks: out is 16-bit [n, k] row-major =
 * (16-bit)(e2m1 * scale) * (16-bit)global_scale.  out_type is FP16 or BF16 (MXFP4:
 * BF16 only).  The _packed variants read the repacked layouts. */
int petit_dequant_nvfp4(void *out, const void *w, const void *scales, float global_scale,
                        int out_type, unsigned k, unsigned n, petit_stream_t stream);
int petit_dequant_mxfp4(void *out, const void *w, const void *scales, float global_scale,
                        int out_type, unsigned k, unsigned n, petit_stream_t stream);
int petit_dequant_packed_nvfp4(void *out, const void *w_packed, const void *scales_packed,
                               float global_scale, int out_type, unsigned k, unsigned n,
                               petit_stream_t stream);
int petit_dequant_packed_mxfp4(void *out, const void *w_packed, const void *scales_packed,
                               float global_scale, int out_type, unsigned k, unsigned n,
                               petit_stream_t stream);

/* Thin device shim (lib/hal/device.h:8-34).  CUDA only; returns 0 or a cudaError_t. */
int petit_hal_device_count(int *count);
int petit_hal_set_device(int device);
int petit_hal_malloc(void **ptr, size_t bytes);
int petit_hal_free(void *ptr);
int petit_hal_memset(void *ptr, int value, size_t bytes);
int petit_hal_copy_to_device(void *dst, const void *src, size_t bytes);
int petit_hal_copy_to_host(void *dst, const void *src, size_t bytes);
int petit_hal_synchronize(void);

/* Tensor-parallel extension (SURVEY section 8 rows e/f2; no reference counterpart): one-shot
 * all-reduce (sum) of a small 16-bit tensor over peer-mapped (symmetric) memory.
 * peer_bufs[r] / peer_pads[r] are THIS process's mappings of rank r's data buffer and
 * signal pad (petit_allreduce_pad_bytes() bytes, zeroed once, then owned by this
 * function); epoch is a local zero-initialised device buffer of
 * petit_allreduce_epoch_bytes().  Every rank must call it with the same numel, in the
 * same order per pad.  out must not alias the local buffer.  dtype: PETIT_DTYPE_BF16/FP16;
 * numel % 8 == 0; world <= 8.  `end_barrier` is a bit set:
 *   PETIT_ALLREDUCE_END_BARRIER: the local buffer may be overwritten as soon as the call has
 *     completed on the stream; without it (one NVLink round trip less) only after the NEXT
 *     call of this group has completed, i.e. the caller alternates between two buffers
 *     (each with its own pad and epoch) and issues at least one call on a buffer's pad
 *     between a read of the buffer and its next overwrite (a CUDA graph that holds a single
 *     call must therefore set the bit);
 *   PETIT_ALLREDUCE_FENCED (or env PETIT_AR_FENCED=1): the peer flags use a
 *     fence.acq_rel.sys release/acquire pattern instead of relaxed system-scope accesses
 *     (+~4 us per barrier; see csrc/allreduce.cu for what the relaxed protocol relies on).
 * A peer that does not arrive within PETIT_AR_TIMEOUT_MS (default 4000) makes the kernel
 * give up without reducing; petit_allreduce_status (synchronises the stream) then returns
 * 1 + the rank that was missing, 0 if every call so far completed, -1 on a CUDA error. */
#define PETIT_ALLREDUCE_END_BARRIER 1
#define PETIT_ALLREDUCE_FENCED 2
size_t petit_allreduce_pad_bytes(void);
size_t petit_allreduce_epoch_bytes(void);
int petit_allreduce_status(const void *epoch, petit_stream_t stream);
int petit_allreduce_oneshot(void *out, const void *const *peer_bufs, void *const *peer_pads,
                            void *epoch, int rank, int world, size_t numel, int dtype,
                            int end_barrier, petit_stream_t stream);

/* Row-parallel (K-split) GEMM fused with the all-reduce of its output (SURVEY section 8 row f2;
 * no reference counterpart): C = sum over ranks of (A_r x dequant(B_r)^T x global_scale), the
 * same bits on every rank.  The CTA that finishes an output tile pushes its 16-bit partial into
 * every peer's receive buffer over NVLink (self-validating {data, epoch} packets, no fence, no
 * separate collective launch) and adds the peers' packets of that tile in rank order in fp32.
 *   recv[r]: THIS process's mapping of rank r's receive buffer (symmetric / peer-mapped
 *     memory, petit_fused_allreduce_recv_bytes(n) bytes, zeroed once before the first call
 *     by its owner, then owned by these functions; recv[rank] is the local buffer);
 *   state: local device words (petit_fused_allreduce_state_bytes(), zeroed once).
 * Every rank calls it for every GEMM of the group, in the same order, with the same m <= 64,
 * n and solution id (the call is CUDA-graph capturable; the call counter lives in `state`).
 * A peer that does not deliver within PETIT_WATCHDOG_MS makes the waiting CTA go on without
 * it; petit_fused_allreduce_status (synchronises the stream) then returns 1 (it does not say
 * which peer was missing), else 0 (-1: CUDA error). */
typedef struct PetitFusedAllReduce {
    int32_t world, rank;
    void *recv[8];
    void *state;
} PetitFusedAllReduce;
int petit_gemm_nvfp4_a16_allreduce(void *c, const void *a, const void *b, const void *scales,
                                   const float *global_scale_dev, unsigned m, unsigned n,
                                   unsigned k, const PetitSolutionHints *hints,
                                   uint64_t solution_id, const PetitFusedAllReduce *ar,
                                   petit_stream_t stream);
int petit_gemm_mxfp4_a16_allreduce(void *c, const void *a, const void *b, const void *scales,
                                   const float *global_scale_dev, unsigned m, unsigned n,
                                   unsigned k, const PetitSolutionHints *hints,
                                   uint64_t solution_id, const PetitFusedAllReduce *ar,
                                   petit_stream_t stream);
/* Fused epilogue (SURVEY section 8 rows f2/f3; extends WriteResult, qgemm.cuh:95-192): what the
 * callers of the reference do right after the GEMM -- `output.add_(bias)`, the residual add --
 * happens on the fp32 accumulator before the single rounding to the output type:
 *     C[m, n] = round(acc[m, n] * global_scale + bias[n] + residual[m, n])
 * bias: [n], residual: [m, n] row-major, both in the output type, either may be NULL;
 * residual may alias c.  `ar` may be NULL (plain GEMM) or a fused all-reduce context; then bias /
 * residual are added to THIS rank's partial, i.e. a row-parallel layer passes them on one rank
 * only.
 * activation = PETIT_ACT_SILU_MUL fuses the MLP's act-and-mul into the gate_up projection:
 *     C[m, i] = round(round(silu(G[m, i])) * U[m, i]),  G / U the rounded GEMM outputs,
 * the arithmetic of the unfused path (GEMM, then silu_and_mul), so the same bits.  C is
 * [m, n / 2].  The weight rows must have been interleaved per 128-row tile BEFORE repacking:
 * rows [128 t, 128 t + 64) = gate rows [64 t, 64 t + 64), rows [128 t + 64, 128 t + 128) = up
 * rows [64 t, 64 t + 64) (petit_kernel.petit_utils.interleave_gate_up does it; bias, if any, is
 * indexed in that row order).  Needs n % 128 == 0, no residual, no all-reduce. */
#define PETIT_ACT_NONE 0
#define PETIT_ACT_SILU_MUL 1
typedef struct PetitEpilogue {
    const void *bias;
    const void *residual;
    int32_t activation;
    int32_t weight_layout; /* PETIT_WEIGHT_LAYOUT_*: how b was repacked (below) */
} PetitEpilogue;

/* Packed weight layouts.  petit_repack_fp4_weights produces the DEFAULT layout, whose in-word
 * bit order is native to bf16 (one shift + one LOP3 per pair of weights) and which every
 * activation type can use.  For fp16 activations the F16_NATIVE variant -- same tiles, words in
 * the native nibble order -- lets the kernel convert a pair with a single cvt.rn.f16x2.e2m1x2
 * (2 instead of ~5 instructions per pair: fp16 decode is then HBM-bound).  It is only valid
 * with NVFP4 weights and fp16 activations, and must be named in PetitEpilogue.weight_layout of
 * the petit_gemm_nvfp4_a16_ex call (the Python ops carry it in the packed tensor's shape). */
#define PETIT_WEIGHT_LAYOUT_DEFAULT 0
#define PETIT_WEIGHT_LAYOUT_F16_NATIVE 1
int petit_repack_fp4_weights_layout(uint32_t *out, const uint32_t *in, unsigned in_chan,
                                    unsigned out_chan, int weight_layout, petit_stream_t stream);
int petit_unpack_fp4_weights_layout(uint32_t *out, const uint32_t *in_packed, unsigned in_chan,
                                    unsigned out_chan, int weight_layout, petit_stream_t stream);
int petit_dequant_packed_nvfp4_layout(void *out, const void *w_packed, const void *scales_packed,
                                      float global_scale, int out_type, unsigned k, unsigned n,
                                      int weight_layout, petit_stream_t stream);
int petit_gemm_nvfp4_a16_ex(void *c, const void *a, const void *b, const void *scales,
                            const float *global_scale_dev, unsigned m, unsigned n, unsigned k,
                            const PetitSolutionHints *hints, uint64_t solution_id,
                            const PetitEpilogue *epilogue, const PetitFusedAllReduce *ar,
                            petit_stream_t stream);
int petit_gemm_mxfp4_a16_ex(void *c, const void *a, const void *b, const void *scales,
                            const float *global_scale_dev, unsigned m, unsigned n, unsigned k,
                            const PetitSolutionHints *hints, uint64_t solution_id,
                            const PetitEpilogue *epilogue, const PetitFusedAllReduce *ar,
                            petit_stream_t stream);

/* Grouped (MoE) GEMM (SURVEY section 8 row f4; the reference has no grouped entry point): one
 * call for `num_groups` independent problems C_g[m_g, n] = A_g[m_g, k] x dequant(B_g)^T x gs_g
 * with a common n, k and type -- the token-grouped expert GEMMs of an MoE layer (tokens sorted
 * by expert, m_g = tokens routed to expert g, groups with m_g == 0 are skipped).
 * ONE launch serves all groups when their activations and outputs are consecutive row blocks
 * of one tensor (a_{g+1} == a_g + m_g * k elements, c likewise -- what "tokens sorted by expert"
 * gives), the token tile is a decode tile (AUTO: 16 / 32 / 64 tokens by the largest m_g; an
 * explicit solution id must name such a tile) and the groups make at most 96 token tiles: the
 * persistent stream-K schedule then runs over the (n-tile, token-tile, k) units of all experts,
 * every SM streams an equal share of all experts' weights, and there is one launch floor
 * instead of one per expert (8 Mixtral-size experts at 16 tokens: 103 vs 140 us for w13, 57 vs
 * 108 us for w2; 64 experts of 2048 x 2048: 41 vs 416 us).  epilogue->activation =
 * PETIT_ACT_SILU_MUL works in this form too (C_g is [m_g, n / 2]): an MoE MLP is two launches.
 * Otherwise, and with a bias, the groups are issued back to back on the stream (each the stream-K
 * kernel, chained by programmatic dependent launch); it returns the first non-zero status.
 * PETIT_GROUPED_SINGLE=0 forces the second form. */
typedef struct PetitGroupedProblem {
    void *c;
    const void *a;
    const void *b;
    const void *scales;
    const float *global_scale_dev;
    unsigned m;
} PetitGroupedProblem;
int petit_gemm_fp4_a16_grouped(const PetitGroupedProblem *problems, unsigned num_groups, unsigned n,
                               unsigned k, const PetitSolutionHints *hints, uint64_t solution_id,
                               const PetitEpilogue *epilogue, petit_stream_t stream);

size_t petit_fused_allreduce_recv_bytes(unsigned n);
size_t petit_fused_allreduce_state_bytes(void);
int petit_fused_allreduce_status(const void *state, petit_stream_t stream);

/* Stream-K workspace (library-owned, one per (device, stream), ~25 MB, created on the first
 * GEMM of a stream, at most 16 alive).  GEMMs that cut output tiles between CTAs let one CTA
 * wait for the partial sums of CTAs with higher block ids, which publish as soon as they are
 * resident; that needs the grid (<= one CTA per SM) to become co-resident.  GEMMs issued on
 * ONE stream, or on several streams of EQUAL priority, always get there (CTAs are dispatched
 * grid after grid).  Two such GEMMs interleaved by streams of DIFFERENT priority can starve
 * each other: then the waiting CTA gives up after PETIT_WATCHDOG_MS (default 2000) and
 * petit_workspace_status reports it.
 *   petit_workspace_status: synchronises `stream`; *status = 0 if no reducer of a GEMM on this
 *     stream ever timed out, else 1 + the output tile that did (that GEMM's output is wrong;
 *     release the workspace before the next call).
 *   petit_release_workspace: synchronises `stream` and frees its workspace (a later GEMM on
 *     the stream creates a fresh one).  Not allowed while the stream is being captured. */
int petit_workspace_status(petit_stream_t stream, int *status);
int petit_release_workspace(petit_stream_t stream);

/* Version of the packed layouts produced by the repack functions. */
int petit_packed_layout_version(void);
/* Human-readable name of a solution id ("" if unknown); pointer is static. */
const char *petit_solution_name(uint64_t solution_id);

#ifdef __cplusplus
} /* extern "C" */
#endif

#endif /* CAUSALFLOW_PETIT_PETIT_H_ */
