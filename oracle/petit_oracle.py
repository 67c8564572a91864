"""CPU oracle for the FP4-weight x 16-bit-activation GEMM path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is imported by the
product (``petit_kernel`` / ``libpetit_b200.so``).  Only ``tests/``,
``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference``
legs of ``bench.py`` may import this module, and only as the checker / the
timed CPU baseline.

What it restates (all citations into /root/reference):

* NVFP4 dequantise + GEMM reference: ``tests/ops/test_fp4_gemm_quark.py:9-24``
  (``_dequant_nvfp4``: LUT order, low nibble = even k, group 16 along K,
  ``scales.float()``; ``_gemm_ref``: fp32 matmul then cast) and ``:51-54``
  (global scale folded into the fp32 weights before the matmul).
* MXFP4 dequantise: the reference test delegates to AMD Quark ``dq_mxfp4``
  (``tests/ops/test_fp4_gemm_quark.py:66-69,83``; dependency ``amd-quark``,
  unpinned in ``pyproject.toml:33-36``, NOT installed here and not vendored).
  We restate the algorithm the reference's own kernels implement:
  ``DequantTraitMxFp4::GetScale`` (``quantization_utils.cu:405-432``) and
  ``DequantizerForE8M0Scale`` e8m0 -> bf16 as ``(s & 0xff) << 7``
  (``dequant.cuh:197-203``), i.e. ``w = LUT[e2m1] * 2**(s-127)`` with group 32
  along K, and ``c = (a @ w.T) * global_scale`` (``test_fp4_gemm_quark.py:87``).
  Tested domain is s in [1, 237] (``quantization_utils_fp4_test.cc:266-278``).
* e4m3 decode used by the exhaustive dequant test:
  ``lib/tests/floating_points.h:21-75`` (fp8_e4m3_t::to_fp32).
* Dense dequant hooks (``DequantizeFp4Kernel``, ``quantization_utils.cu:542-612``):
  16-bit weight times ``Element(global_scale)`` with a 16-bit multiply.
* Synthetic input recipes: ``tests/ops/test_fp4_gemm_quark.py:41-46,71-76`` and
  ``lib/tests/quantization.cc:77-143`` (value ranges; mt19937(42)).
* The C++ GEMM matcher ``IsNearBf16/IsNearFp16``
  (``gemm_fp4_fp16_rocm_test.cc:31-67``).

Pinning status: the NVFP4 functions are checked bit-for-bit against the
reference's own Python oracle executed in the build container
(``tests/golden/make_golden.py`` imports it from /root/reference and commits
the vectors).  The MXFP4 functions are pinned to implementations this repository
did not write: AMD Quark itself is absent from the image, so
``tests/golden/make_golden_mx.py`` builds the expectations of the reference test's
recipe (``test_fp4_gemm_quark.py:71-87``) from torch's own OCP e8m0 dtype
(``uint8.view(torch.float8_e8m0fnu)``) and compressed-tensors' e2m1 decoder
(``unpack_fp4_from_uint8``), cross-checked against compressed-tensors'
``decompress_mx_scale``; ``tests/test_oracle.py`` requires this module to reproduce
``tests/golden/mxfp4_independent.npz`` bit for bit (dequantised weights incl. the
exhaustive 16 x 237 table and the reference's scale-mixing pattern) and the GEMM
vectors within one bf16 ulp.  What stays unpinned is only Quark's own code path.
"""
from __future__ import annotations

import numpy as np
import torch

# tests/ops/test_fp4_gemm_quark.py:10-14 and quantization_utils_fp4_test.cc:259-262
E2M1_VALUES = np.array(
    [0.0, 0.5, 1.0, 1.5, 2.0, 3.0, 4.0, 6.0,
     -0.0, -0.5, -1.0, -1.5, -2.0, -3.0, -4.0, -6.0],
    dtype=np.float32,
)

NVFP4_GROUP = 16
MXFP4_GROUP = 32


# --------------------------------------------------------------------------
# scalar format decoders
# --------------------------------------------------------------------------
def e4m3_to_f32(bits: np.ndarray) -> np.ndarray:
    """OCP e4m3fn byte -> float32 (lib/tests/floating_points.h:21-75).

    sign(1) exp(4, bias 7) mant(3); exp==0 is subnormal (mant/8 * 2**-6);
    0x7f/0xff are NaN; there is no infinity.
    """
    bits = np.asarray(bits, dtype=np.uint8).astype(np.int32)
    sign = np.where(bits & 0x80, -1.0, 1.0).astype(np.float32)
    exp = (bits >> 3) & 0xF
    man = bits & 0x7
    normal = np.ldexp((8 + man).astype(np.float32), exp - 7 - 3)
    sub = np.ldexp(man.astype(np.float32), -6 - 3)
    out = np.where(exp == 0, sub, normal).astype(np.float32)
    out = np.where((exp == 0xF) & (man == 0x7), np.float32(np.nan), out)
    return (sign * out).astype(np.float32)


def e8m0_to_f32(bits: np.ndarray) -> np.ndarray:
    """e8m0 byte -> float32 the way the reference decodes it:
    bf16 bit pattern ``(s & 0xff) << 7`` (dequant.cuh:197-203).

    Consequences outside the tested domain [1, 237]: s == 0 gives 0.0 (OCP says
    2**-127) and s == 255 gives +inf (OCP says NaN).
    """
    bits = np.asarray(bits, dtype=np.uint8).astype(np.uint32)
    as_f32 = (bits << np.uint32(7 + 16)).astype(np.uint32)
    return as_f32.view(np.float32)


def unpack_e2m1(q_u8: np.ndarray) -> np.ndarray:
    """[N, K/2] bytes -> [N, K] float32; low nibble is the even k
    (tests/ops/test_fp4_gemm_quark.py:15-19)."""
    q_u8 = np.asarray(q_u8, dtype=np.uint8)
    n, kh = q_u8.shape
    out = np.empty((n, kh * 2), dtype=np.float32)
    out[:, 0::2] = E2M1_VALUES[q_u8 & 0x0F]
    out[:, 1::2] = E2M1_VALUES[q_u8 >> 4]
    return out


# --------------------------------------------------------------------------
# dequantise
# --------------------------------------------------------------------------
def dequant_nvfp4(q_u8: np.ndarray, scales_e4m3: np.ndarray) -> np.ndarray:
    """[N,K/2] u8 + [N,K/16] e4m3 bytes -> [N,K] float32
    (tests/ops/test_fp4_gemm_quark.py:9-20)."""
    w = unpack_e2m1(q_u8)
    n, k = w.shape
    s = e4m3_to_f32(scales_e4m3).reshape(n, k // NVFP4_GROUP, 1)
    return (w.reshape(n, -1, NVFP4_GROUP) * s).reshape(n, k).astype(np.float32)


def dequant_mxfp4(q_u8: np.ndarray, scales_e8m0: np.ndarray) -> np.ndarray:
    """[N,K/2] u8 + [N,K/32] e8m0 bytes -> [N,K] float32 =
    LUT * 2**(s-127) (quantization_utils.cu:405-432, dequant.cuh:197-203)."""
    w = unpack_e2m1(q_u8)
    n, k = w.shape
    s = e8m0_to_f32(scales_e8m0).reshape(n, k // MXFP4_GROUP, 1)
    with np.errstate(invalid="ignore", over="ignore"):
        return (w.reshape(n, -1, MXFP4_GROUP) * s).reshape(n, k).astype(np.float32)


def _torch_dtype(name_or_dtype) -> torch.dtype:
    if isinstance(name_or_dtype, torch.dtype):
        return name_or_dtype
    return {"bf16": torch.bfloat16, "bfloat16": torch.bfloat16,
            "fp16": torch.float16, "float16": torch.float16}[name_or_dtype]


def dense16(w_f32: np.ndarray, global_scale: float, dtype) -> torch.Tensor:
    """What the reference's dense dequant hooks return
    (DequantizeFp4Kernel, quantization_utils.cu:563-585): the exact 16-bit
    weight multiplied by ``Element(global_scale)`` with a 16-bit multiply."""
    dt = _torch_dtype(dtype)
    w16 = torch.from_numpy(np.ascontiguousarray(w_f32)).to(dt)
    gs16 = torch.tensor(global_scale, dtype=torch.float32).to(dt)
    return (w16.float() * gs16.float()).to(dt)


# --------------------------------------------------------------------------
# GEMM references
# --------------------------------------------------------------------------
def gemm_ref(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """tests/ops/test_fp4_gemm_quark.py:23-24."""
    return (a.float() @ b.t().float()).to(a.dtype)


def nvfp4_gemm_ref(a: torch.Tensor, q_u8: torch.Tensor, scales_e4m3: torch.Tensor,
                   global_scale: torch.Tensor) -> torch.Tensor:
    """tests/ops/test_fp4_gemm_quark.py:51-53: global scale is folded into the
    fp32 weights, then fp32 matmul, then cast to a.dtype."""
    w = dequant_nvfp4(q_u8.cpu().numpy(), scales_e4m3.cpu().view(torch.uint8).numpy())
    b_ref = torch.from_numpy(w) * float(global_scale.item())
    return gemm_ref(a.cpu(), b_ref)


def nvfp4_gemm_ref_torch(a: torch.Tensor, q_u8: torch.Tensor, scales_e4m3: torch.Tensor,
                         global_scale: torch.Tensor) -> torch.Tensor:
    """Same computation as nvfp4_gemm_ref with torch ops only (multi-threaded on the
    host), statement for statement what tests/ops/test_fp4_gemm_quark.py:9-24,51-53
    does; used as the timed CPU baseline."""
    lut = torch.from_numpy(E2M1_VALUES)
    q_u8 = q_u8.cpu()
    lo = q_u8 & 0x0F
    hi = q_u8 >> 4
    deq = torch.empty((q_u8.size(0), q_u8.size(1) * 2), dtype=torch.float32)
    deq[:, 0::2] = lut[lo.long()]
    deq[:, 1::2] = lut[hi.long()]
    w = (deq.view(q_u8.size(0), -1, NVFP4_GROUP) * scales_e4m3.cpu().float().unsqueeze(-1)
         ).view(q_u8.size(0), -1)
    b_ref = w * float(global_scale.item())
    return gemm_ref(a.cpu(), b_ref)


def mxfp4_gemm_ref(a: torch.Tensor, q_u8: torch.Tensor, scales_e8m0: torch.Tensor,
                   global_scale: torch.Tensor) -> torch.Tensor:
    """tests/ops/test_fp4_gemm_quark.py:83-87: dequantise to bf16, fp32 matmul,
    multiply by global_scale, cast."""
    w = dequant_mxfp4(q_u8.cpu().numpy(), scales_e8m0.cpu().numpy())
    b = torch.from_numpy(w).to(torch.bfloat16)
    a = a.cpu()
    return ((a.float() @ b.t().float()) * float(global_scale.item())).to(a.dtype)


# --------------------------------------------------------------------------
# matchers
# --------------------------------------------------------------------------
def is_near_cpp(out: torch.Tensor, ref: torch.Tensor) -> torch.Tensor:
    """Element-wise IsNearBf16 / IsNearFp16
    (gemm_fp4_fp16_rocm_test.cc:31-67): |a-b| < max(1e-2, 0.01*|b|)."""
    a, b = out.float().cpu(), ref.float().cpu()
    return (a - b).abs() < torch.clamp(b.abs() * 0.01, min=1e-2)


def max_rel_err(out: torch.Tensor, ref_f32: torch.Tensor) -> float:
    """north_star tolerance: max |c - ref| / max |ref| against the fp32
    accumulation of the dequantised weights."""
    a, b = out.float().cpu(), ref_f32.float().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def bits_equal_pm0(x: torch.Tensor, y: torch.Tensor) -> bool:
    """Bit-exact comparison that treats +0 and -0 as equal and NaN as unequal
    (lib/tests/floating_points.h:184-202)."""
    assert x.dtype == y.dtype and x.shape == y.shape
    xi = x.cpu().contiguous().view(torch.int16)
    yi = y.cpu().contiguous().view(torch.int16)
    same = xi == yi
    both_zero = ((xi & 0x7FFF) == 0) & ((yi & 0x7FFF) == 0)
    nan = torch.isnan(x.cpu().float()) | torch.isnan(y.cpu().float())
    return bool(((same | both_zero) & ~nan).all())


# --------------------------------------------------------------------------
# synthetic inputs
# --------------------------------------------------------------------------
def make_nvfp4_case(m: int, n: int, k: int, seed: int, dtype=torch.bfloat16):
    """Recipe of tests/ops/test_fp4_gemm_quark.py:41-46, generated with the CPU
    generator so that the same tensors exist on every machine (the reference
    draws them with the device generator, whose stream is backend-specific)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    a = torch.randn((m, k), generator=g, dtype=torch.float32).to(dtype)
    q = torch.randint(0, 256, (n, k // 2), generator=g, dtype=torch.uint8)
    s = (torch.rand((n, k // NVFP4_GROUP), generator=g) * 3.5 + 0.25).to(torch.float8_e4m3fn)
    gs = torch.rand((1,), generator=g, dtype=torch.float32) * 1.5 + 0.5
    return a, q, s, gs


def make_mxfp4_case(m: int, n: int, k: int, seed: int, dtype=torch.bfloat16):
    """Recipe of tests/ops/test_fp4_gemm_quark.py:71-76 (scales in [1, 237])."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    a = torch.randn((m, k), generator=g, dtype=torch.float32).to(dtype)
    q = torch.randint(0, 256, (n, k // 2), generator=g, dtype=torch.uint8)
    s = torch.randint(1, 238, (n, k // MXFP4_GROUP), generator=g, dtype=torch.uint8)
    gs = torch.rand((1,), generator=g, dtype=torch.float32) * 1.5 + 0.5
    return a, q, s, gs


def make_gtest_style_case(m: int, n: int, k: int, fmt: str = "nvfp4",
                          dtype=torch.bfloat16, seed: int = 42):
    """Distributions of lib/tests/quantization.cc:77-143 (mt19937(seed)):
    A ~ U(-2,2) truncated to bf16 (U(-1,1) for fp16), every u32 of weights
    uniformly random, NV scales uniform over the positive e4m3 bit patterns
    0x01..0x7E, MX scales uniform in [1, 237], global_scale = 1.
    (The C++ stream itself is libstdc++-specific and is not reproduced.)"""
    rs = np.random.RandomState(seed)
    if dtype == torch.bfloat16:
        af = rs.uniform(-2.0, 2.0, size=(m, k)).astype(np.float32)
        a = torch.from_numpy((af.view(np.uint32) >> 16).astype(np.uint16).view(np.int16)
                             ).view(torch.bfloat16)
    else:
        a = torch.from_numpy(rs.uniform(-1.0, 1.0, size=(m, k)).astype(np.float32)).to(dtype)
    q = torch.from_numpy(rs.randint(0, 2 ** 32, size=(n, k // 8), dtype=np.uint32
                                    ).view(np.uint8).reshape(n, k // 2).copy())
    if fmt == "nvfp4":
        s = torch.from_numpy(rs.randint(0x01, 0x7F, size=(n, k // NVFP4_GROUP)
                                        ).astype(np.uint8)).view(torch.float8_e4m3fn)
    else:
        s = torch.from_numpy(rs.randint(1, 238, size=(n, k // MXFP4_GROUP)).astype(np.uint8))
    gs = torch.ones((1,), dtype=torch.float32)
    return a, q, s, gs


# --------------------------------------------------------------------------
# exactly representable GEMMs
# --------------------------------------------------------------------------
# Every dequantised weight is exact in 16 bits (csrc/dequant.cuh) and the kernel's A operand is
# that weight times a power of two.  With activations in {+-1/2, +-1, +-2} and scales from a
# narrow set, every product is a multiple of a quantum q; if for every output the sum of the
# magnitudes of its products, T = (|a| @ |w|^T)[m, n], is at most 2^22 q, every partial sum of
# every subset of the products is a multiple of q below 2^22 q, i.e. exact in fp32 whatever the
# order and grouping (tcgen05 accumulation, accumulator chains, stream-K partials, reducer).
# The output is then RN16(RN32(S * gs)) bit for bit, S the exact sum.
EXACT_ACTS = np.array([-2.0, -1.0, -0.5, 0.5, 1.0, 2.0], dtype=np.float32)
EXACT_BOUND_LOG2 = 22


def _nv_scale_options(k: int):
    """e4m3 bytes, widest set first.  Several mantissas per binade so that a scale read from the
    neighbouring group changes the value."""
    wide = [e * 8 + m for e in (7, 8, 9) for m in (0, 1, 2, 4, 6, 7)]     # 1 .. 3.75 x 2^2
    mid = [e * 8 + m for e in (7, 8) for m in (0, 1, 2, 4, 6, 7)]         # 1 .. 3.75
    narrow = [7 * 8 + m for m in (0, 2, 4, 6)]                           # 1, 1.25, 1.5, 1.75
    opts = [wide, mid, narrow]
    return opts if k <= 4096 else opts[1:] if k <= 12288 else opts[2:]


def _mx_scale_options(k: int):
    """e8m0 bytes straddling 125 / 126 (the kernel's two-step threshold), widest first."""
    opts = [list(range(122, 130)), list(range(123, 129)), list(range(124, 128))]
    return opts if k <= 4096 else opts[1:] if k <= 12288 else opts[2:]


def exact_quantum(fmt: str, scale_bytes) -> float:
    """q: every |act| * |e2m1| * scale is a multiple of it (act and e2m1 lsb are both 1/2)."""
    if fmt == "nvfp4":
        lsb = min(float(2.0 ** ((b >> 3) - 7 - 3)) if b >> 3 else 2.0 ** -9 for b in scale_bytes)
    else:
        lsb = 2.0 ** (min(scale_bytes) - 127)
    return 0.25 * lsb


def exact_magnitude_bound(a: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """T = |a| @ |w|^T in float64 (on a's device)."""
    return a.double().abs() @ w.to(a.device).double().abs().t()


def make_exact_case(fmt: str, dtype, m: int, n: int, k: int, seed: int, gs: float = 0.7):
    """Random e2m1 codes (all 16, -0 included), activations from EXACT_ACTS, scales from the
    widest set of _nv/_mx_scale_options whose T stays <= 2^22 q (asserted), global scale gs (a
    non-power of two, so that RN32(S * gs) rounds).  Returns a, q, s, gs (tensors like
    make_nvfp4_case), the dequantised weights w [n, k] float32 and the quantum q."""
    dt = _torch_dtype(dtype)
    rs = np.random.RandomState(seed)
    a_np = EXACT_ACTS[rs.randint(0, len(EXACT_ACTS), size=(m, k))]
    q = rs.randint(0, 256, size=(n, k // 2)).astype(np.uint8)
    opts = _nv_scale_options(k) if fmt == "nvfp4" else _mx_scale_options(k)
    group = NVFP4_GROUP if fmt == "nvfp4" else MXFP4_GROUP
    a = torch.from_numpy(a_np)
    for i, choice in enumerate(opts):
        sb = np.asarray(choice, dtype=np.uint8)[rs.randint(0, len(choice), size=(n, k // group))]
        w = dequant_nvfp4(q, sb) if fmt == "nvfp4" else dequant_mxfp4(q, sb)
        quantum = exact_quantum(fmt, choice)
        t_max = float(exact_magnitude_bound(a, torch.from_numpy(w)).max())
        if t_max <= 2.0 ** EXACT_BOUND_LOG2 * quantum or i == len(opts) - 1:
            break
    assert t_max <= 2.0 ** EXACT_BOUND_LOG2 * quantum, (fmt, m, n, k, t_max / quantum)
    s = torch.from_numpy(sb.copy())
    if fmt == "nvfp4":
        s = s.view(torch.float8_e4m3fn)
    return (a.to(dt), torch.from_numpy(q), s, torch.tensor([gs], dtype=torch.float32),
            w, quantum)


def rn16(x_f32: np.ndarray, dtype) -> torch.Tensor:
    """Round-to-nearest-even float32 -> bf16 / fp16 (subnormals and overflow to inf included)."""
    return torch.from_numpy(np.ascontiguousarray(x_f32, dtype=np.float32)).to(_torch_dtype(dtype))


def exact_epilogue(s_f64: np.ndarray, gs: float, dtype, bias=None, residual=None) -> torch.Tensor:
    """The kernel's epilogue (csrc/fp4_gemm.cu, 'Fused epilogue terms') on the exact sum S:
    RN32(S * gs), + bias[n], + residual[m, n], each addition rounded to fp32, then RN16.  The
    kernel multiplies by gs * epilogue_factor (a power of two) -- the same real product as long
    as that factor does not underflow or overflow gs, which the callers keep true."""
    s32 = np.asarray(s_f64, dtype=np.float32)
    assert np.array_equal(s32.astype(np.float64), np.asarray(s_f64), equal_nan=True), \
        "S is not exact in fp32: the case does not meet the exactness precondition"
    with np.errstate(over="ignore", invalid="ignore"):
        v = s32 * np.float32(gs)
        if bias is not None:
            v = v + bias.float().cpu().numpy().astype(np.float32)[None, :]
        if residual is not None:
            v = v + residual.float().cpu().numpy().astype(np.float32)
    return rn16(v, dtype)


def exact_ref(a: torch.Tensor, w: np.ndarray, gs: float, dtype, bias=None, residual=None) -> torch.Tensor:
    """Bit-exact expected output of the GEMM on an exact case: S = a @ w^T in float64 from the
    oracle's dequantised weights (never the kernel's dequant_dense hook), on a's device, then
    exact_epilogue on the host."""
    wt = torch.from_numpy(np.ascontiguousarray(w)).to(a.device).double()
    s = (a.double() @ wt.t()).cpu().numpy()
    return exact_epilogue(s, gs, dtype, bias, residual)


def ulp16(x: torch.Tensor, dtype) -> torch.Tensor:
    """Spacing of the 16-bit format at |x| (float64; the subnormal spacing below the normals)."""
    dt = _torch_dtype(dtype)
    p, emin = (8, -126) if dt == torch.bfloat16 else (11, -14)
    ax = x.double().abs()
    _, e = torch.frexp(torch.where(ax > 0, ax, torch.ones_like(ax)))
    e = torch.where(ax > 0, e - 1, torch.full_like(e, emin))
    return torch.exp2((torch.clamp(e, min=emin) - (p - 1)).double())


def accumulation_gamma(k: int) -> float:
    """Relative error bound factor of the kernel's fp32 accumulation, derived from its depth:
    every output is a sum of k products (exact: 16-bit x 16-bit fits fp32) added in
    k / 16 MMA steps along one accumulator chain, then the chains (<= 8) are added, then the
    stream-K partials (at most one per CTA, <= 160), then one multiply by the global scale.
    Each of these additions rounds once with a relative error below 2^-23 (2^-23 rather than
    2^-24 so that truncating adders are covered too), so |err| <= gamma * sum|terms| with
    gamma = (k / 16 + 8 + 160 + 1) * 2^-23."""
    return (k / 16 + 8 + 160 + 1) * 2.0 ** -23


def elementwise_ok(c: torch.Tensor, a: torch.Tensor, w, gs: float, dtype, bias=None, residual=None,
                   return_excess: bool = False):
    """Per-element check for general (non-exact) data:
        |c - ref| <= 1/2 ulp16(|ref| + E) + E,   E = gamma(k) |gs| (|a| @ |w|^T) + 3 * 2^-24 (|ref| + E')
    ref = (a @ w^T) gs (+ bias + residual) in float64; the first term is the final rounding to
    16 bits, gamma the accumulation (accumulation_gamma), the last term the fp32 rounding of the
    scale multiply and the bias / residual additions.  Computed on a's device; w is the oracle's
    dequantised [n, k] weight (numpy or tensor).  Returns a bool (or the largest
    |c - ref| / bound with return_excess)."""
    dev = a.device
    wt = (torch.from_numpy(np.ascontiguousarray(w)) if isinstance(w, np.ndarray) else w).to(dev).double()
    ad = a.double()
    ref = (ad @ wt.t()) * float(gs)
    extra = torch.zeros_like(ref)
    if bias is not None:
        ref = ref + bias.to(dev).double()[None, :]
        extra = extra + bias.to(dev).double().abs()[None, :]
    if residual is not None:
        ref = ref + residual.to(dev).double()
        extra = extra + residual.to(dev).double().abs()
    acc = accumulation_gamma(a.shape[1]) * abs(float(gs)) * (ad.abs() @ wt.abs().t())
    e = acc + 3 * 2.0 ** -24 * (ref.abs() + acc + extra)
    bound = 0.5 * ulp16(ref.abs() + e, dtype) + e
    diff = (c.to(dev).double() - ref).abs()
    if return_excess:
        return float((diff / bound).max())
    return bool((diff <= bound).all())


# --------------------------------------------------------------------------
# stream-K plan (restates launch_variant / launch_mode / Cfg of csrc/fp4_gemm.cu)
# --------------------------------------------------------------------------
TILE_N, TILE_K, MAX_GRID = 128, 256, 160
MAX_GROUP_TILES = 96  # kMaxGroupTiles (csrc/fp4_gemm.h)
MODES = ("nv_bf16", "nv_f16", "nv_f16n", "mx_bf16")


def stage_k(ntok: int) -> int:
    return 256 if ntok <= 64 else (128 if ntok == 128 else 64)


def ring_fit(mode: str, ntok: int) -> int:
    """kRingFit = kStages * kStageBytes / (NTOK * 128 * 4): contributor partials the reducer can
    pull into its drained stage ring (Cfg in csrc/fp4_gemm.cu)."""
    ks = stage_k(ntok)
    subs, chunks = ks // 64, ks // 32
    sc_per_sub = 2 if mode == "mx_bf16" else 4
    stage = (subs * ntok * 128 + chunks * 128 * 16 + subs * 128 * sc_per_sub + 1023) // 1024 * 1024
    teams = 3 if ntok >= 256 else 1
    bufs = 2 if (teams > 1 or ntok <= 64) else 3
    budget = 227 * 1024 - 1024 - teams * bufs * 16 * 128 * 2 - 16 * 128 * 4 - 1024
    raw = min(16, budget // stage)
    stages = 6 if (ntok <= 64 and 6 <= raw < 12) else raw
    return stages * stage // (ntok * TILE_N * 4)


def stream_k_plan(m: int, n: int, k: int, ntok: int, num_sms: int, pdl: bool, cluster: bool,
                  cuts_fn, mode: str = "nv_bf16", whole_tiles_rule: bool = True,
                  tilt_units: int = -1, tilt_late: int = -1, all_reduce: bool = False,
                  tile_rows=None, tile_groups=None):
    """Grid, range cuts and per-tile reducer facts of one launch.

    cuts_fn(units, k_tiles, grid, lat, late) -> grid + 1 cuts: the library's
    petit_debug_stream_k_cuts (lat = late = 0 gives the equal split).  `cluster` is the
    PETIT_CLUSTER setting, `whole_tiles_rule` PETIT_WHOLE_TILES, tilt_units / tilt_late
    PETIT_TILT_UNITS / PETIT_TILT_LATE (-1: unset).  Each tile entry: contributors (CTAs other
    than the reducer that add a partial; 0 = unsplit), m_valid, n_partial, and the reducer path
    of its first 16 tokens ('reg' <= 3 contributors, 'ring' up to ring_fit, else 'reg' over all
    of them) and whether tokens 16.. reach the L2 tail loop.

    all_reduce: the GEMM fused with its all-reduce (launch_mode with ar_world > 1, i.e.
    launch_variant<..., CL = false, AR = true>): decode tiles only (ntok 16 / 32 / 64, m <= 64),
    never a cluster, and no arrival term in the cut tilt (late = 0).

    tile_rows: the grouped launch (launch_variant<..., GR = true>, decode tiles only): token tile
    t covers tile_rows[t] rows (the `rows` of group_table's entry t) instead of the rows of a
    plain [m, k] tensor, and m_tiles = len(tile_rows).  tile_groups[t] is entry t's expert; it
    only feeds the grouped coverage labels of plan_paths."""
    if all_reduce:
        assert ntok in (16, 32, 64) and 1 <= m <= 64, (ntok, m)
        cluster = False
    if tile_rows is not None:
        assert ntok in (16, 32, 64) and 1 <= len(tile_rows) <= MAX_GROUP_TILES, (ntok, len(tile_rows))
        assert all(1 <= r <= ntok for r in tile_rows) and len(tile_groups) == len(tile_rows)
    num_sms = min(num_sms, MAX_GRID)
    n_tiles = (n + TILE_N - 1) // TILE_N
    m_tiles = (m + ntok - 1) // ntok if tile_rows is None else len(tile_rows)
    k_tiles = k // TILE_K
    cl = ntok >= 128 and cluster and n_tiles % 2 == 0 and n % TILE_N == 0
    units = (n_tiles // 2 if cl else n_tiles) * m_tiles * k_tiles
    grid = min(units, num_sms)
    whole = False
    tiles = n_tiles * m_tiles
    if not cl and ntok <= 64 and whole_tiles_rule:
        if tiles <= num_sms and tiles * 3 >= num_sms and k_tiles <= 6:
            grid, whole = tiles, True
    sched_grid = grid
    if cl:
        sched_grid = min(units, num_sms // 2)
        grid = 2 * sched_grid
    tilt = (not cl) and ntok <= 64 and grid > 1 and not whole and units >= 8 * grid
    lat = late = 0
    if tilt:
        lat = tilt_units if tilt_units >= 0 else (5 if ntok <= 32 else 3)
        late = 0 if (not pdl or all_reduce) else (tilt_late if tilt_late >= 0 else (4 if ntok <= 32 else 3))
    cuts = list(cuts_fn(units, k_tiles, sched_grid, lat, late))
    assert cuts[0] == 0 and cuts[-1] == units and len(cuts) == sched_grid + 1

    def owner(u):
        lo, hi = 0, sched_grid - 1
        while lo < hi:  # last b with cuts[b] <= u
            mid = (lo + hi + 1) // 2
            if cuts[mid] <= u:
                lo = mid
            else:
                hi = mid - 1
        return lo

    fit = ring_fit(mode, ntok)
    out = []
    for t in range(units // k_tiles):
        b_first, b_last = owner(t * k_tiles), owner(t * k_tiles + k_tiles - 1)
        c = b_last - b_first
        m_tile = t % m_tiles
        m_valid = min(ntok, m - m_tile * ntok) if tile_rows is None else tile_rows[m_tile]
        n_tile = (2 if cl else 1) * (t // m_tiles)
        rows = [min(TILE_N, n - nt * TILE_N) for nt in ((n_tile, n_tile + 1) if cl else (n_tile,))]
        path = None if c == 0 else ("ring" if 3 < c <= fit else "reg")
        out.append(dict(tile=t, m_tile=m_tile, contributors=c, m_valid=m_valid, n_partial=min(rows) < TILE_N,
                        path=path, l2_tail=c > 0 and path == "reg" and m_valid > 16 and c > fit))
    # experts whose units each CTA's range holds (grouped launch)
    cta_groups = None if tile_groups is None else [
        {tile_groups[t % m_tiles] for t in range(cuts[b] // k_tiles, (cuts[b + 1] - 1) // k_tiles + 1)}
        for b in range(sched_grid)]
    return dict(ntok=ntok, grid=grid, sched_grid=sched_grid, cluster=cl, whole_tiles=whole, tilt=tilt, lat=lat,
                late=late, units=units, k_tiles=k_tiles, m_tiles=m_tiles, ring_fit=fit, cuts=cuts, tiles=out,
                tile_groups=tile_groups, cta_groups=cta_groups)


def plan_paths(plan) -> set:
    """Coverage labels of one launch (see stream_k_plan).  A grouped launch adds:
      group_switch      a CTA's range holds units of two or more experts (weights, scales and gs
                        change inside one CTA's k-range);
      split_group_tail  a split tile with fewer than ntok rows that is not the last token tile
                        (the rows its token tile loads after its last row are the next expert's);
      direct_store      a tile whose rows are not a multiple of 16 (its last 16-token group is
                        written with 16-byte stores instead of a TMA box);
      multi_tile_group  an expert with more than one token tile;
      table_full        a table of exactly MAX_GROUP_TILES entries."""
    got = set()
    if plan["tile_groups"] is not None:
        if any(len(g) >= 2 for g in plan["cta_groups"]):
            got.add("group_switch")
        for t in plan["tiles"]:
            if t["contributors"] and t["m_valid"] < plan["ntok"] and t["m_tile"] != plan["m_tiles"] - 1:
                got.add("split_group_tail")
            if t["m_valid"] % 16:
                got.add("direct_store")
        if len(set(plan["tile_groups"])) < plan["m_tiles"]:
            got.add("multi_tile_group")
        if plan["m_tiles"] == MAX_GROUP_TILES:
            got.add("table_full")
    if plan["whole_tiles"]:
        got.add("whole_tiles")
    if plan["ntok"] >= 128:
        got.add("cluster" if plan["cluster"] else "cluster_fallback")
    if plan["tilt"]:
        got.add("tilt")
    for t in plan["tiles"]:
        c = t["contributors"]
        if c == 0:
            got.add("unsplit")
            continue
        got.add("reg_1_3" if c <= 3 else ("ring" if t["path"] == "ring" else "many_reg"))
        if c > plan["ring_fit"] and c > 3:
            got.add("many_m_le16" if t["m_valid"] <= 16 else "many_m_gt16")
        if t["l2_tail"]:
            got.add("l2_tail")
        if t["n_partial"]:
            got.add("split_partial_n")
        if t["m_valid"] < plan["ntok"]:
            got.add("split_partial_m")
    return got


# --------------------------------------------------------------------------
# grouped (MoE) launch (restates petit_gemm_fp4_a16_grouped of csrc/capi.cu)
# --------------------------------------------------------------------------
def group_table(counts, ntok: int):
    """[(group, row0, rows)]: the token tiles of the single grouped launch.  Expert g owns rows
    [sum(counts[:g]), sum(counts[:g + 1])) of the concatenated activations / output; each of its
    ntok-row blocks is one entry, the last one holding the remainder; empty experts have none."""
    out, row = [], 0
    for g, c in enumerate(counts):
        for r in range(0, c, ntok):
            out.append((g, row + r, min(ntok, c - r)))
        row += c
    return out


def grouped_launch(counts, n: int, k: int, sid: int, dtype, contiguous: bool = True, bias: bool = False,
                   single_env: bool = True):
    """How petit_gemm_fp4_a16_grouped issues a call: ("single", ntok, group_table(counts, ntok))
    or ("one_by_one", None, [(group, m)] of the live groups in order).  One launch needs all of:
    PETIT_GROUPED_SINGLE not 0 (single_env), no bias, n and k non-zero, the live groups'
    activations and outputs consecutive row blocks of one tensor (contiguous), at least two live
    groups, a decode tile (sid -1: 16 / 32 / 64 tokens by the largest group; an explicit id must
    name a tile of <= 64 tokens) and a table of at most MAX_GROUP_TILES entries.  dtype is the
    activation type (bf16 or fp16: both have the single form)."""
    assert _torch_dtype(dtype) in (torch.bfloat16, torch.float16)
    live = [(g, c) for g, c in enumerate(counts) if c]
    ntok = 0
    if single_env and not bias and n and k and contiguous and len(live) >= 2:
        if sid == -1:
            top = max(c for _, c in live)
            ntok = 16 if top <= 16 else (32 if top <= 32 else 64)
        elif (sid & 0xFF) * 16 <= 64:
            ntok = (sid & 0xFF) * 16
    if ntok:
        table = group_table(counts, ntok)
        if len(table) <= MAX_GROUP_TILES:
            return "single", ntok, table
    return "one_by_one", None, live


def rank_order_sum(partials, dtype) -> torch.Tensor:
    """What the fused all-reduce computes from the ranks' 16-bit partial outputs (one-shot and
    two-shot alike): an fp32 sum that starts from +0.0f and adds ranks 0 .. world - 1 in that
    order, each addition rounded to fp32, then one RN16.  partials: 16-bit tensors of one
    shape, rank 0 first."""
    dt = _torch_dtype(dtype)
    acc = np.zeros(tuple(partials[0].shape), dtype=np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        for p in partials:
            assert p.dtype == dt, (p.dtype, dt)
            acc = (acc + p.detach().cpu().float().numpy()).astype(np.float32)
    return rn16(acc, dt)
