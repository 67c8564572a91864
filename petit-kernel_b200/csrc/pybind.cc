// PyTorch extension module `petit_kernel.ops`.
//
// Mirrors the reference's binding layer lib/pybind/{pybind.cc,fp4.cc}: same
// function names, argument order, checks and error messages
// (fp4.cc:38-283), re-targeted at the C ABI of libpetit_b200.so and
// ATen/cuda.  Additions over the reference (SURVEY Appendix C): a CUDA device
// guard, shape/device checks on B and s in mul_nvfp4_a16, the DataType enum, the
// Python-level get_fp4_solutions signature, and the unpack / dense-dequant test
// hooks.  There is no CPU path: every op requires CUDA tensors.
#include "causalflow/petit/petit.h"

#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include <vector>

namespace py = pybind11;

namespace {

constexpr int64_t kLayoutM = 128; // fp4.cc:17 (k divisibility checked at repack)
constexpr int64_t kLayoutN = 16;  // fp4.cc:18
constexpr int64_t kPackFactor = 8;
constexpr int64_t kKTile = 256;   // k granularity of the packed layout

petit_stream_t stream_of(const torch::Tensor &t) {
    return reinterpret_cast<petit_stream_t>(
        at::cuda::getCurrentCUDAStream(t.get_device()).stream());
}

void check_status(int err, int64_t m, int64_t n, int64_t k, int64_t solution_id) {
    // fp4.cc:201-206
    if (err == PETIT_ERROR_PROBLEM_SHAPE) {
        AT_ERROR("Incompatible problem shape (m=", m, ", n=", n, ", k=", k, ")");
    } else if (err == PETIT_ERROR_KERNEL_SHAPE) {
        AT_ERROR("No kernel implementation for solution_id=", solution_id, ".");
    } else if (err != PETIT_OK) {
        AT_ERROR("petit CUDA failure (code ", err, "): ",
                 cudaGetErrorString(cudaGetLastError()));
    }
}

PetitDataType dtype_of(const torch::Tensor &A) {
    if (A.dtype() != torch::kBFloat16 && A.dtype() != torch::kFloat16) {
        AT_ERROR("A must be bfloat16 or float16.");
    }
    return A.dtype() == torch::kBFloat16 ? PETIT_DTYPE_BF16 : PETIT_DTYPE_FP16;
}

// The packed weight tensor carries its layout in its shape (the tensor is opaque to callers and
// keeps the reference's dtype and byte count either way): [N/16, 2K] = default layout
// (fp4.cc:62-63), [N/32, 4K] = fp16-native layout (petit.h, PETIT_WEIGHT_LAYOUT_F16_NATIVE).
int weight_layout_of(const torch::Tensor &B, int64_t size_n, int64_t size_k) {
    if (B.dim() == 2 && size_n % 32 == 0 && B.size(0) == size_n / 32 && B.size(1) == 4 * size_k)
        return PETIT_WEIGHT_LAYOUT_F16_NATIVE;
    return PETIT_WEIGHT_LAYOUT_DEFAULT;
}

// ---- fp4.cc:38-78 ------------------------------------------------------------
torch::Tensor RepackNvFp4Layout(torch::Tensor &b_q_weight, int64_t size_n, int64_t size_k,
                                const py::object &a_dtype);
torch::Tensor RepackNvFp4(torch::Tensor &b_q_weight, int64_t size_n, int64_t size_k) {
    return RepackNvFp4Layout(b_q_weight, size_n, size_k, py::none());
}
torch::Tensor RepackNvFp4Layout(torch::Tensor &b_q_weight, int64_t size_n, int64_t size_k,
                                const py::object &a_dtype) {
    TORCH_CHECK(size_k % kLayoutM == 0, "size_k = ", size_k,
                " is not divisible by tile_k_size = ", kLayoutM);
    TORCH_CHECK(size_n % kLayoutN == 0, "size_n = ", size_n,
                " is not divisible by tile_n_size = ", kLayoutN);
    TORCH_CHECK((size_k / kPackFactor) == b_q_weight.size(1),
                "Shape mismatch: b_q_weight.size(1) = ", b_q_weight.size(1),
                ", size_k = ", size_k, ", pack_factor = ", kPackFactor);
    TORCH_CHECK(b_q_weight.size(0) == size_n, "b_q_weight.size(0) = ", b_q_weight.size(0),
                " is not size_n = ", size_n);
    TORCH_CHECK(b_q_weight.device().is_cuda(), "b_q_weight is not on GPU");
    TORCH_CHECK(b_q_weight.is_contiguous(), "b_q_weight is not contiguous");
    TORCH_CHECK(b_q_weight.dtype() == at::kInt, "b_q_weight type is not kInt");
    // the reference's kernel grid needs k % 256 (quantization_utils.cu:733-735)
    TORCH_CHECK(size_k % kKTile == 0, "size_k = ", size_k,
                " is not divisible by tile_k_size = ", kKTile);

    // a_dtype = torch.float16: the weights will only ever meet fp16 activations -> fp16-native
    // layout (needs N % 32 for its shape tag; otherwise, and by default, the layout every
    // activation type can use)
    int layout = PETIT_WEIGHT_LAYOUT_DEFAULT;
    if (!a_dtype.is_none() &&
        torch::python::detail::py_object_to_dtype(a_dtype) == torch::kFloat16 && size_n % 32 == 0)
        layout = PETIT_WEIGHT_LAYOUT_F16_NATIVE;
    c10::cuda::CUDAGuard guard(b_q_weight.device());
    auto options = torch::TensorOptions().dtype(b_q_weight.dtype()).device(b_q_weight.device());
    torch::Tensor out =
        layout == PETIT_WEIGHT_LAYOUT_F16_NATIVE
            ? torch::empty({size_n / 32, size_k * 32 / kPackFactor}, options)
            : torch::empty({size_n / kLayoutN, size_k * kLayoutN / kPackFactor}, options);
    int err = petit_repack_fp4_weights_layout(
        reinterpret_cast<uint32_t *>(out.data_ptr()),
        reinterpret_cast<const uint32_t *>(b_q_weight.data_ptr()), size_k, size_n, layout,
        stream_of(b_q_weight));
    check_status(err, 0, size_n, size_k, -1);
    return out;
}

torch::Tensor UnpackFp4(torch::Tensor &packed, int64_t size_n, int64_t size_k) {
    TORCH_CHECK(packed.device().is_cuda() && packed.is_contiguous() && packed.dtype() == at::kInt,
                "packed weights must be a contiguous CUDA int32 tensor");
    TORCH_CHECK(packed.numel() == size_n * size_k / kPackFactor, "packed size mismatch");
    c10::cuda::CUDAGuard guard(packed.device());
    torch::Tensor out = torch::empty({size_n, size_k / kPackFactor}, packed.options());
    int err = petit_unpack_fp4_weights_layout(
        reinterpret_cast<uint32_t *>(out.data_ptr()),
        reinterpret_cast<const uint32_t *>(packed.data_ptr()), size_k, size_n,
        weight_layout_of(packed, size_n, size_k), stream_of(packed));
    check_status(err, 0, size_n, size_k, -1);
    return out;
}

// ---- fp4.cc:80-121 -----------------------------------------------------------
torch::Tensor ProcessNvFp4Scales(torch::Tensor &scales, int64_t size_n, int64_t size_k) {
    constexpr int64_t kGroupM = 2 * kLayoutM;
    TORCH_CHECK(size_k % kGroupM == 0, "size_k = ", size_k,
                " is not divisible by tile_k_size = ", kGroupM);
    TORCH_CHECK(size_n % kLayoutN == 0, "size_n = ", size_n,
                " is not divisible by tile_n_size = ", kLayoutN);
    int64_t group_size = size_k / scales.size(1);
    if (group_size != 16) {
        AT_ERROR("Only groupsize = 16 is supported.");
    }
    TORCH_CHECK(scales.size(0) == size_n, "scales.size(0) = ", scales.size(0),
                " is not size_n = ", size_n);
    TORCH_CHECK(scales.device().is_cuda(), "scales is not on GPU");
    TORCH_CHECK(scales.is_contiguous(), "scales is not contiguous");
    TORCH_CHECK(scales.dtype() == at::kFloat8_e4m3fn, "scales type is not float8_e4m3fn");

    c10::cuda::CUDAGuard guard(scales.device());
    auto options = torch::TensorOptions().dtype(scales.dtype()).device(scales.device());
    torch::Tensor out = torch::empty({scales.size(0), scales.size(1)}, options);
    int err = petit_repack_nvfp4_scales(out.data_ptr(), scales.data_ptr(), size_k, size_n,
                                        stream_of(scales));
    check_status(err, 0, size_n, size_k, -1);
    return out;
}

// ---- fp4.cc:123-161 ----------------------------------------------------------
torch::Tensor ProcessMxFp4Scales(torch::Tensor &scales, int64_t size_n, int64_t size_k) {
    constexpr int64_t kScaleLayoutN = 32, kMxRowGroupSize = 32;
    constexpr int64_t kGroupM = 2 * kLayoutM;
    TORCH_CHECK(size_k % kGroupM == 0, "size_k = ", size_k,
                " is not divisible by tile_k_size = ", kGroupM);
    TORCH_CHECK(size_n % kLayoutN == 0, "size_n = ", size_n,
                " is not divisible by tile_n_size = ", kLayoutN);
    int64_t group_size = size_k / scales.size(1);
    if (group_size != 32) {
        AT_ERROR("Only groupsize = 32 is supported.");
    }
    TORCH_CHECK(scales.size(0) == size_n, "scales.size(0) = ", scales.size(0),
                " is not size_n = ", size_n);
    TORCH_CHECK(scales.device().is_cuda(), "scales is not on GPU");
    TORCH_CHECK(scales.is_contiguous(), "scales is not contiguous");
    TORCH_CHECK(scales.dtype() == at::kByte, "scales type is not uint8");
    // the reference output shape [N/32, K] needs N % 32 (fp4.cc:146-148)
    TORCH_CHECK(size_n % kScaleLayoutN == 0, "size_n = ", size_n,
                " is not divisible by scale tile_n_size = ", kScaleLayoutN);

    c10::cuda::CUDAGuard guard(scales.device());
    auto options = torch::TensorOptions().dtype(scales.dtype()).device(scales.device());
    torch::Tensor out = torch::empty(
        {size_n / kScaleLayoutN, size_k * kScaleLayoutN / kMxRowGroupSize}, options);
    int err = petit_repack_mxfp4_scales(out.data_ptr(), scales.data_ptr(), size_k, size_n,
                                        stream_of(scales));
    check_status(err, 0, size_n, size_k, -1);
    return out;
}

void check_gemm_operands(const torch::Tensor &A, const torch::Tensor &B, const torch::Tensor &s,
                         const torch::Tensor &global_scale, int64_t size_m, int64_t size_n,
                         int64_t size_k, int64_t scale_bytes) {
    TORCH_CHECK(A.device().is_cuda(), "A is not on GPU");
    TORCH_CHECK(B.device() == A.device() && s.device() == A.device() &&
                    global_scale.device() == A.device(),
                "A, B, s and global_scale must be on the same CUDA device");
    TORCH_CHECK(A.is_contiguous(), "A is not contiguous");
    TORCH_CHECK(B.is_contiguous(), "B is not contiguous");
    TORCH_CHECK(s.is_contiguous(), "s is not contiguous");
    TORCH_CHECK(A.dim() == 2 && A.size(0) == size_m && A.size(1) == size_k,
                "A must have shape [size_m, size_k]");
    TORCH_CHECK(B.numel() * B.element_size() == size_n * size_k / 2,
                "B does not hold size_n * size_k packed fp4 values");
    TORCH_CHECK(s.numel() * s.element_size() == scale_bytes,
                "s does not hold the processed scales of a [size_n, size_k] weight");
    TORCH_CHECK(global_scale.dtype() == torch::kFloat32 && global_scale.numel() >= 1,
                "global_scale must be a float32 tensor");
}

// ---- fp4.cc:163-209 ----------------------------------------------------------
torch::Tensor alloc_or_check_out(const c10::optional<torch::Tensor> &out, const torch::Tensor &A,
                                 int64_t size_m, int64_t size_n) {
    if (!out.has_value()) {
        auto options = torch::TensorOptions().dtype(A.dtype()).device(A.device());
        return torch::empty({size_m, size_n}, options);
    }
    const torch::Tensor &c = *out;
    TORCH_CHECK(c.device() == A.device() && c.dtype() == A.dtype() && c.is_contiguous() &&
                    c.dim() == 2 && c.size(0) == size_m && c.size(1) == size_n,
                "out must be a contiguous [size_m, size_n] tensor of A's dtype on A's device");
    return c;
}

torch::Tensor MulNvFp4A16Impl(const torch::Tensor &A, const torch::Tensor &B, const torch::Tensor &s,
                              const torch::Tensor &global_scale, int64_t size_m, int64_t size_n,
                              int64_t size_k, int64_t solution_id,
                              const c10::optional<torch::Tensor> &out) {
    int64_t groupsize = s.size(1) ? size_k / s.size(1) : 0;
    if (groupsize != 16) {
        AT_ERROR("Only groupsize = 16 is supported. size_k = ", size_k,
                 ", s.size(1) = ", s.size(1));
    }
    PetitDataType a_type = dtype_of(A);
    check_gemm_operands(A, B, s, global_scale, size_m, size_n, size_k, size_n * size_k / 16);

    c10::cuda::CUDAGuard guard(A.device());
    torch::Tensor c = alloc_or_check_out(out, A, size_m, size_n);

    PetitSolutionHints hints;
    hints.a_type = a_type;
    hints.b_type = PETIT_DTYPE_FP4_E2M1;
    hints.c_type = a_type;
    hints.require_high_precision = 0; // gfx90a workaround (fp4.cc:24-34): n/a on B200

    PetitEpilogue epi = {nullptr, nullptr, PETIT_ACT_NONE, weight_layout_of(B, size_n, size_k)};
    TORCH_CHECK(epi.weight_layout == PETIT_WEIGHT_LAYOUT_DEFAULT || a_type == PETIT_DTYPE_FP16,
                "B was repacked for float16 activations (repack_nvfp4(..., a_dtype=torch.float16)); "
                "A is bfloat16");
    int err = petit_gemm_nvfp4_a16_ex(c.data_ptr(), A.data_ptr(), B.data_ptr(), s.data_ptr(),
                                      global_scale.data_ptr<float>(), size_m, size_n, size_k, &hints,
                                      static_cast<uint64_t>(solution_id), &epi, nullptr,
                                      stream_of(A));
    check_status(err, size_m, size_n, size_k, solution_id);
    return c;
}

torch::Tensor MulNvFp4A16(const torch::Tensor &A, const torch::Tensor &B, const torch::Tensor &s,
                          const torch::Tensor &global_scale, int64_t size_m, int64_t size_n,
                          int64_t size_k, int64_t solution_id) {
    return MulNvFp4A16Impl(A, B, s, global_scale, size_m, size_n, size_k, solution_id, c10::nullopt);
}

// ---- fp4.cc:211-260 ----------------------------------------------------------
torch::Tensor MulMxFp4A16Impl(const torch::Tensor &A, const torch::Tensor &B, const torch::Tensor &s,
                              const torch::Tensor &global_scale, int64_t size_m, int64_t size_n,
                              int64_t size_k, int64_t solution_id,
                              const c10::optional<torch::Tensor> &out) {
    TORCH_CHECK(B.size(0) == size_n / kLayoutN, "B.size(0) = ", B.size(0),
                " is not size_n / 16 = ", size_n / kLayoutN);
    TORCH_CHECK(B.size(1) == size_k * kLayoutN / kPackFactor, "B.size(1) = ", B.size(1),
                " is not packed size = ", size_k * kLayoutN / kPackFactor);
    TORCH_CHECK(s.size(0) == size_n / 32, "s.size(0) = ", s.size(0),
                " is not size_n / 32 = ", size_n / 32);
    TORCH_CHECK(s.size(1) == size_k, "s.size(1) = ", s.size(1), " is not size_k = ", size_k);
    PetitDataType a_type = dtype_of(A);
    check_gemm_operands(A, B, s, global_scale, size_m, size_n, size_k, size_n * size_k / 32);

    c10::cuda::CUDAGuard guard(A.device());
    torch::Tensor c = alloc_or_check_out(out, A, size_m, size_n);

    PetitSolutionHints hints;
    hints.a_type = a_type;
    hints.b_type = PETIT_DTYPE_MXFP4_E2M1;
    hints.c_type = a_type;
    hints.require_high_precision = 0;

    int err = petit_gemm_mxfp4_a16(c.data_ptr(), A.data_ptr(), B.data_ptr(), s.data_ptr(),
                                   global_scale.data_ptr<float>(), size_m, size_n, size_k, &hints,
                                   static_cast<uint64_t>(solution_id), stream_of(A));
    check_status(err, size_m, size_n, size_k, solution_id);
    return c;
}

torch::Tensor MulMxFp4A16(const torch::Tensor &A, const torch::Tensor &B, const torch::Tensor &s,
                          const torch::Tensor &global_scale, int64_t size_m, int64_t size_n,
                          int64_t size_k, int64_t solution_id) {
    return MulMxFp4A16Impl(A, B, s, global_scale, size_m, size_n, size_k, solution_id, c10::nullopt);
}

// ---- fp4.cc:262-283 ----------------------------------------------------------
py::list GetNvFp4Solutions(const PetitSolutionHints &hints, int64_t size_m, int64_t size_n,
                           int64_t size_k) {
    unsigned n_solutions = 0;
    int err = petit_get_solutions(&hints, size_m, size_n, size_k, nullptr, &n_solutions);
    if (err != 0) {
        AT_ERROR("Failed to get solutions: ", err);
    }
    std::vector<uint64_t> solutions(n_solutions);
    err = petit_get_solutions(&hints, size_m, size_n, size_k, solutions.data(), &n_solutions);
    if (err != 0) {
        AT_ERROR("Failed to get solutions: ", err);
    }
    py::list ret;
    for (unsigned i = 0; i < n_solutions; ++i) ret.append(solutions[i]);
    return ret;
}

int dtype_code(py::object dt) {
    auto t = torch::python::detail::py_object_to_dtype(dt);
    if (t == torch::kBFloat16) return PETIT_DTYPE_BF16;
    if (t == torch::kFloat16) return PETIT_DTYPE_FP16;
    AT_ERROR("a_type / c_type must be torch.bfloat16 or torch.float16");
}

// Accepts both the reference's bound form (hints, m, n, k) (pybind.cc:14-17) and the
// form its Python wrapper actually passes (m, n, k, a_type, c_type)
// (petit_kernel/__init__.py:63-66); the latter raises TypeError in the reference.
py::list GetFp4Solutions(py::args args, py::kwargs kwargs) {
    if (args.size() >= 1 && py::isinstance<PetitSolutionHints>(args[0])) {
        TORCH_CHECK(args.size() == 4, "get_fp4_solutions(hints, size_m, size_n, size_k)");
        return GetNvFp4Solutions(args[0].cast<PetitSolutionHints>(), args[1].cast<int64_t>(),
                                 args[2].cast<int64_t>(), args[3].cast<int64_t>());
    }
    TORCH_CHECK(args.size() == 5,
                "get_fp4_solutions(size_m, size_n, size_k, a_type, c_type[, b_type=])");
    PetitSolutionHints hints;
    hints.a_type = dtype_code(args[3]);
    hints.c_type = dtype_code(args[4]);
    hints.b_type = PETIT_DTYPE_FP4_E2M1;
    if (kwargs.contains("b_type")) hints.b_type = kwargs["b_type"].cast<int>();
    hints.require_high_precision = 0;
    return GetNvFp4Solutions(hints, args[0].cast<int64_t>(), args[1].cast<int64_t>(),
                             args[2].cast<int64_t>());
}

// Dense dequant hooks (fp4/gemm_fp4.h:11-21, quantization_utils.cu:614-727).
torch::Tensor DequantDense(const torch::Tensor &w, const torch::Tensor &scales, double global_scale,
                           py::object out_dtype, int64_t size_n, int64_t size_k, bool mx,
                           bool packed) {
    TORCH_CHECK(w.device().is_cuda() && scales.device().is_cuda(), "tensors must be on GPU");
    TORCH_CHECK(w.is_contiguous() && scales.is_contiguous(), "tensors must be contiguous");
    c10::cuda::CUDAGuard guard(w.device());
    auto dt = torch::python::detail::py_object_to_dtype(out_dtype);
    int code = dt == torch::kBFloat16 ? PETIT_DTYPE_BF16
                                      : (dt == torch::kFloat16 ? PETIT_DTYPE_FP16 : -1);
    torch::Tensor out =
        torch::empty({size_n, size_k}, torch::TensorOptions().dtype(dt).device(w.device()));
    int err;
    auto st = stream_of(w);
    if (mx)
        err = packed ? petit_dequant_packed_mxfp4(out.data_ptr(), w.data_ptr(), scales.data_ptr(),
                                                  global_scale, code, size_k, size_n, st)
                     : petit_dequant_mxfp4(out.data_ptr(), w.data_ptr(), scales.data_ptr(),
                                           global_scale, code, size_k, size_n, st);
    else
        err = packed ? petit_dequant_packed_nvfp4_layout(out.data_ptr(), w.data_ptr(),
                                                         scales.data_ptr(), global_scale, code, size_k,
                                                         size_n, weight_layout_of(w, size_n, size_k), st)
                     : petit_dequant_nvfp4(out.data_ptr(), w.data_ptr(), scales.data_ptr(),
                                           global_scale, code, size_k, size_n, st);
    TORCH_CHECK(err == 0, "dequant hook failed with code ", err,
                " (bad shape or unsupported output type)");
    return out;
}

} // namespace

PYBIND11_MODULE(ops, m) {
    // pybind.cc:9-25 of the reference
    m.def("repack_nvfp4", &RepackNvFp4Layout, "Repack NVFP4 to Petit FP4", py::arg("qw"),
          py::arg("size_n"), py::arg("size_k"), py::arg("a_dtype") = py::none());
    m.def("process_nvfp4_scales", &ProcessNvFp4Scales, "Process NVFP4 scales", py::arg("scales"),
          py::arg("size_n"), py::arg("size_k"));
    m.def("process_mxfp4_scales", &ProcessMxFp4Scales, "Process MXFP4 scales", py::arg("scales"),
          py::arg("size_n"), py::arg("size_k"));
    m.def("mul_nvfp4_a16", &MulNvFp4A16, "Multiply NVFP4 FP16", py::arg("a"), py::arg("b"),
          py::arg("s"), py::arg("global_scale"), py::arg("size_m"), py::arg("size_n"),
          py::arg("size_k"), py::arg("solution_id") = -1);
    m.def("mul_mxfp4_a16", &MulMxFp4A16, "Multiply MXFP4 FP16", py::arg("a"), py::arg("b"),
          py::arg("s"), py::arg("global_scale"), py::arg("size_m"), py::arg("size_n"),
          py::arg("size_k"), py::arg("solution_id") = -1);
    m.def("get_nvfp4_solutions", &GetNvFp4Solutions, "Get possible fp4 solutions");
    m.def("get_fp4_solutions", &GetFp4Solutions, "Get possible fp4 solutions");

    py::class_<PetitSolutionHints>(m, "PetitSolutionHints")
        .def(py::init([]() {
            PetitSolutionHints h;
            h.a_type = PETIT_DTYPE_BF16;
            h.b_type = PETIT_DTYPE_FP4_E2M1;
            h.c_type = PETIT_DTYPE_BF16;
            h.require_high_precision = 0;
            return h;
        }))
        .def_readwrite("a_type", &PetitSolutionHints::a_type)
        .def_readwrite("b_type", &PetitSolutionHints::b_type)
        .def_readwrite("c_type", &PetitSolutionHints::c_type)
        .def_property(
            "require_high_precision",
            [](const PetitSolutionHints &h) { return h.require_high_precision != 0; },
            [](PetitSolutionHints &h, bool v) { h.require_high_precision = v ? 1 : 0; });

    // the C++ DataType values (types.h:4-13), not registered in the reference
    py::enum_<PetitDataType>(m, "CDataType")
        .value("kDataTypeInt4", PETIT_DTYPE_INT4)
        .value("kDataTypeFp8e4m3", PETIT_DTYPE_FP8_E4M3)
        .value("kDataTypeFp8e8m0", PETIT_DTYPE_FP8_E8M0)
        .value("kDataTypeFp4e2m1", PETIT_DTYPE_FP4_E2M1)
        .value("kDataTypeFp16", PETIT_DTYPE_FP16)
        .value("kDataTypeBf16", PETIT_DTYPE_BF16)
        .value("kDataTypeFp8e5m2Fnuz", PETIT_DTYPE_FP8_E5M2_FNUZ)
        .value("kDataTypeMxFp4e2m1", PETIT_DTYPE_MXFP4_E2M1)
        .export_values();

    // extras: write into a caller-provided output (e.g. a symmetric-memory buffer that a
    // one-shot all-reduce of a row-parallel layer reads in place)
    m.def("mul_nvfp4_a16_out",
          [](const torch::Tensor &out, const torch::Tensor &a, const torch::Tensor &b,
             const torch::Tensor &s, const torch::Tensor &gs, int64_t sm, int64_t sn, int64_t sk,
             int64_t sol) { return MulNvFp4A16Impl(a, b, s, gs, sm, sn, sk, sol, out); },
          py::arg("out"), py::arg("a"), py::arg("b"), py::arg("s"), py::arg("global_scale"),
          py::arg("size_m"), py::arg("size_n"), py::arg("size_k"), py::arg("solution_id") = -1);
    m.def("mul_mxfp4_a16_out",
          [](const torch::Tensor &out, const torch::Tensor &a, const torch::Tensor &b,
             const torch::Tensor &s, const torch::Tensor &gs, int64_t sm, int64_t sn, int64_t sk,
             int64_t sol) { return MulMxFp4A16Impl(a, b, s, gs, sm, sn, sk, sol, out); },
          py::arg("out"), py::arg("a"), py::arg("b"), py::arg("s"), py::arg("global_scale"),
          py::arg("size_m"), py::arg("size_n"), py::arg("size_k"), py::arg("solution_id") = -1);

    // extras: GEMM with the fused epilogue (bias / residual added in fp32 before the rounding)
    m.def(
        "mul_fp4_a16_ex_out",
        [](const c10::optional<torch::Tensor> &out, const torch::Tensor &a, const torch::Tensor &b,
           const torch::Tensor &s, const torch::Tensor &gs, int64_t sm, int64_t sn, int64_t sk,
           int64_t sol, bool mx, const c10::optional<torch::Tensor> &bias,
           const c10::optional<torch::Tensor> &residual, bool silu_mul) {
            PetitDataType a_type = dtype_of(a);
            check_gemm_operands(a, b, s, gs, sm, sn, sk, sn * sk / (mx ? 32 : 16));
            c10::cuda::CUDAGuard guard(a.device());
            TORCH_CHECK(!silu_mul || sn % 128 == 0, "silu_mul needs size_n % 128 == 0");
            torch::Tensor c = alloc_or_check_out(out, a, sm, silu_mul ? sn / 2 : sn);
            PetitEpilogue epi = {nullptr, nullptr, silu_mul ? PETIT_ACT_SILU_MUL : PETIT_ACT_NONE,
                                 mx ? PETIT_WEIGHT_LAYOUT_DEFAULT : weight_layout_of(b, sn, sk)};
            TORCH_CHECK(epi.weight_layout == PETIT_WEIGHT_LAYOUT_DEFAULT || a_type == PETIT_DTYPE_FP16,
                        "b was repacked for float16 activations; a is bfloat16");
            if (bias.has_value()) {
                TORCH_CHECK(bias->is_cuda() && bias->is_contiguous() && bias->numel() == sn &&
                                bias->scalar_type() == a.scalar_type(),
                            "bias must be a contiguous CUDA tensor of size_n elements in a's dtype");
                epi.bias = bias->data_ptr();
            }
            if (residual.has_value()) {
                TORCH_CHECK(residual->is_cuda() && residual->is_contiguous() &&
                                residual->numel() == sm * sn && residual->scalar_type() == a.scalar_type(),
                            "residual must be a contiguous CUDA [size_m, size_n] tensor in a's dtype");
                epi.residual = residual->data_ptr();
            }
            PetitSolutionHints hints;
            hints.a_type = a_type;
            hints.b_type = mx ? PETIT_DTYPE_MXFP4_E2M1 : PETIT_DTYPE_FP4_E2M1;
            hints.c_type = a_type;
            hints.require_high_precision = 0;
            auto fn = mx ? petit_gemm_mxfp4_a16_ex : petit_gemm_nvfp4_a16_ex;
            int err = fn(c.data_ptr(), a.data_ptr(), b.data_ptr(), s.data_ptr(), gs.data_ptr<float>(),
                         sm, sn, sk, &hints, static_cast<uint64_t>(sol), &epi, nullptr, stream_of(a));
            check_status(err, sm, sn, sk, sol);
            return c;
        },
        py::arg("out"), py::arg("a"), py::arg("b"), py::arg("s"), py::arg("global_scale"),
        py::arg("size_m"), py::arg("size_n"), py::arg("size_k"), py::arg("solution_id") = -1,
        py::arg("mx") = false, py::arg("bias") = py::none(), py::arg("residual") = py::none(),
        py::arg("silu_mul") = false);

    // extras: grouped (MoE) GEMM -- tokens sorted by expert, expert g owns rows
    // [offsets[g], offsets[g + 1]) of a / out; b and s are [E, ...] stacks of repacked experts
    m.def(
        "mul_fp4_a16_grouped_out",
        [](const torch::Tensor &out, const torch::Tensor &a, const torch::Tensor &b,
           const torch::Tensor &s, const torch::Tensor &gs, const std::vector<int64_t> &offsets,
           int64_t sn, int64_t sk, int64_t sol, bool mx, bool silu_mul) {
            const int64_t e = (int64_t)offsets.size() - 1;
            TORCH_CHECK(e >= 1 && b.dim() == 3 && s.dim() == 3 && b.size(0) == e && s.size(0) == e,
                        "b and s must be [num_experts, ...] stacks matching offsets");
            TORCH_CHECK(a.is_cuda() && a.is_contiguous() && a.dim() == 2 && a.size(1) == sk &&
                            a.size(0) == offsets.back() && offsets.front() == 0,
                        "a must be contiguous [total_tokens, size_k] with offsets[-1] rows");
            TORCH_CHECK(!silu_mul || sn % 128 == 0, "silu_mul needs size_n % 128 == 0");
            const int64_t out_n = silu_mul ? sn / 2 : sn;
            TORCH_CHECK(out.is_cuda() && out.is_contiguous() && out.dim() == 2 &&
                            out.size(0) == a.size(0) && out.size(1) == out_n && out.dtype() == a.dtype(),
                        "out must be contiguous [total_tokens, size_n (/ 2 with silu_mul)] in a's dtype");
            TORCH_CHECK(b.is_cuda() && b.is_contiguous() && s.is_cuda() && s.is_contiguous() &&
                            b[0].numel() * 4 == sn * sk / 2 && s[0].numel() == sn * sk / (mx ? 32 : 16),
                        "per-expert packed weight / scale size mismatch");
            TORCH_CHECK(gs.is_cuda() && gs.scalar_type() == torch::kFloat && gs.numel() == e,
                        "global_scale must be a float32 CUDA tensor with one entry per expert");
            PetitDataType a_type = dtype_of(a);
            c10::cuda::CUDAGuard guard(a.device());
            std::vector<PetitGroupedProblem> probs((size_t)e);
            const int64_t esz = a.element_size();
            for (int64_t g = 0; g < e; ++g) {
                TORCH_CHECK(offsets[g + 1] >= offsets[g], "offsets must be non-decreasing");
                probs[g].c = static_cast<char *>(out.data_ptr()) + offsets[g] * out_n * esz;
                probs[g].a = static_cast<const char *>(a.data_ptr()) + offsets[g] * sk * esz;
                probs[g].b = b[g].data_ptr();
                probs[g].scales = s[g].data_ptr();
                probs[g].global_scale_dev = gs.data_ptr<float>() + g;
                probs[g].m = (unsigned)(offsets[g + 1] - offsets[g]);
            }
            PetitSolutionHints hints;
            hints.a_type = a_type;
            hints.b_type = mx ? PETIT_DTYPE_MXFP4_E2M1 : PETIT_DTYPE_FP4_E2M1;
            hints.c_type = a_type;
            hints.require_high_precision = 0;
            PetitEpilogue epi = {nullptr, nullptr, silu_mul ? PETIT_ACT_SILU_MUL : PETIT_ACT_NONE,
                                 mx ? PETIT_WEIGHT_LAYOUT_DEFAULT : weight_layout_of(b[0], sn, sk)};
            int err = petit_gemm_fp4_a16_grouped(probs.data(), (unsigned)e, sn, sk, &hints,
                                                 static_cast<uint64_t>(sol), &epi, stream_of(a));
            check_status(err, a.size(0), sn, sk, sol);
            return out;
        },
        py::arg("out"), py::arg("a"), py::arg("b"), py::arg("s"), py::arg("global_scale"),
        py::arg("offsets"), py::arg("size_n"), py::arg("size_k"), py::arg("solution_id") = -1,
        py::arg("mx") = false, py::arg("silu_mul") = false);

    // extras: row-parallel GEMM fused with the all-reduce of its output (petit_tp.FusedAllReduce)
    m.def(
        "mul_fp4_a16_allreduce_out",
        [](const torch::Tensor &out, const torch::Tensor &a, const torch::Tensor &b,
           const torch::Tensor &s, const torch::Tensor &gs, int64_t sm, int64_t sn, int64_t sk,
           int64_t sol, bool mx, const std::vector<int64_t> &recv_ptrs, const torch::Tensor &state,
           int64_t rank) {
            TORCH_CHECK(recv_ptrs.size() >= 2 && recv_ptrs.size() <= 8, "world must be 2..8");
            TORCH_CHECK(state.is_cuda() && state.nbytes() >= petit_fused_allreduce_state_bytes(),
                        "state buffer too small");
            PetitDataType a_type = dtype_of(a);
            check_gemm_operands(a, b, s, gs, sm, sn, sk, sn * sk / (mx ? 32 : 16));
            c10::cuda::CUDAGuard guard(a.device());
            torch::Tensor c = alloc_or_check_out(out, a, sm, sn);
            PetitSolutionHints hints;
            hints.a_type = a_type;
            hints.b_type = mx ? PETIT_DTYPE_MXFP4_E2M1 : PETIT_DTYPE_FP4_E2M1;
            hints.c_type = a_type;
            hints.require_high_precision = 0;
            PetitEpilogue epi = {nullptr, nullptr, PETIT_ACT_NONE,
                                 mx ? PETIT_WEIGHT_LAYOUT_DEFAULT : weight_layout_of(b, sn, sk)};
            TORCH_CHECK(epi.weight_layout == PETIT_WEIGHT_LAYOUT_DEFAULT || a_type == PETIT_DTYPE_FP16,
                        "b was repacked for float16 activations; a is bfloat16");
            PetitFusedAllReduce ar;
            ar.world = (int32_t)recv_ptrs.size();
            ar.rank = (int32_t)rank;
            for (int r = 0; r < 8; ++r)
                ar.recv[r] = r < ar.world ? reinterpret_cast<void *>(recv_ptrs[r]) : nullptr;
            ar.state = state.data_ptr();
            auto fn = mx ? petit_gemm_mxfp4_a16_ex : petit_gemm_nvfp4_a16_ex;
            int err = fn(c.data_ptr(), a.data_ptr(), b.data_ptr(), s.data_ptr(), gs.data_ptr<float>(),
                         sm, sn, sk, &hints, static_cast<uint64_t>(sol), &epi, &ar, stream_of(a));
            check_status(err, sm, sn, sk, sol);
            return c;
        },
        py::arg("out"), py::arg("a"), py::arg("b"), py::arg("s"), py::arg("global_scale"),
        py::arg("size_m"), py::arg("size_n"), py::arg("size_k"), py::arg("solution_id"),
        py::arg("mx"), py::arg("recv_ptrs"), py::arg("state"), py::arg("rank"));
    m.def("fused_allreduce_recv_bytes",
          [](int64_t n) { return (int64_t)petit_fused_allreduce_recv_bytes((unsigned)n); });
    m.def("fused_allreduce_state_bytes", []() { return (int64_t)petit_fused_allreduce_state_bytes(); });
    m.def("fused_allreduce_status", [](const torch::Tensor &state) {
        c10::cuda::CUDAGuard guard(state.device());
        return (int64_t)petit_fused_allreduce_status(
            state.data_ptr(), at::cuda::getCurrentCUDAStream(state.device().index()).stream());
    });

    // extras: tensor-parallel one-shot all-reduce over peer-mapped memory (petit_tp)
    m.def(
        "allreduce_oneshot",
        [](const torch::Tensor &out, const std::vector<int64_t> &buf_ptrs,
           const std::vector<int64_t> &pad_ptrs, const torch::Tensor &epoch, int64_t rank,
           int64_t numel, bool end_barrier, bool fenced) {
            TORCH_CHECK(out.is_cuda() && out.is_contiguous(), "out must be a contiguous CUDA tensor");
            TORCH_CHECK(out.scalar_type() == torch::kBFloat16 || out.scalar_type() == torch::kHalf,
                        "out must be bf16 or fp16");
            TORCH_CHECK(buf_ptrs.size() == pad_ptrs.size() && !buf_ptrs.empty() && buf_ptrs.size() <= 8,
                        "need one buffer and one pad pointer per rank (world <= 8)");
            TORCH_CHECK(numel <= out.numel(), "out is smaller than numel");
            TORCH_CHECK(epoch.is_cuda() && epoch.nbytes() >= petit_allreduce_epoch_bytes(),
                        "epoch buffer too small");
            const void *bufs[8];
            void *pads[8];
            for (size_t r = 0; r < buf_ptrs.size(); ++r) {
                bufs[r] = reinterpret_cast<const void *>(buf_ptrs[r]);
                pads[r] = reinterpret_cast<void *>(pad_ptrs[r]);
            }
            c10::cuda::CUDAGuard guard(out.device());
            int rc = petit_allreduce_oneshot(
                out.data_ptr(), bufs, pads, epoch.data_ptr(), (int)rank, (int)buf_ptrs.size(),
                (size_t)numel,
                out.scalar_type() == torch::kBFloat16 ? PETIT_DTYPE_BF16 : PETIT_DTYPE_FP16,
                (end_barrier ? PETIT_ALLREDUCE_END_BARRIER : 0) | (fenced ? PETIT_ALLREDUCE_FENCED : 0),
                at::cuda::getCurrentCUDAStream(out.device().index()).stream());
            TORCH_CHECK(rc == 0, "petit_allreduce_oneshot failed with code ", rc);
            return out;
        },
        py::arg("out"), py::arg("buf_ptrs"), py::arg("pad_ptrs"), py::arg("epoch"), py::arg("rank"),
        py::arg("numel"), py::arg("end_barrier") = true, py::arg("fenced") = false);
    m.def("allreduce_status", [](const torch::Tensor &epoch) {
        c10::cuda::CUDAGuard guard(epoch.device());
        return (int64_t)petit_allreduce_status(
            epoch.data_ptr(), at::cuda::getCurrentCUDAStream(epoch.device().index()).stream());
    });
    m.def("allreduce_pad_bytes", []() { return (int64_t)petit_allreduce_pad_bytes(); });
    m.def("allreduce_epoch_bytes", []() { return (int64_t)petit_allreduce_epoch_bytes(); });

    // extras: round-trip / bit-exactness hooks and introspection
    m.def("unpack_fp4", &UnpackFp4, "Inverse of repack_nvfp4 (test hook)");
    m.def("dequant_dense", &DequantDense, "Dense dequantisation hook", py::arg("w"),
          py::arg("scales"), py::arg("global_scale"), py::arg("out_dtype"), py::arg("size_n"),
          py::arg("size_k"), py::arg("mx"), py::arg("packed"));
    // extras: the default chooser and its tuned-solution table (petit.h: petit_tune_table_*)
    m.def(
        "get_default_solution",
        [](int64_t size_m, int64_t size_n, int64_t size_k, py::object a_type, bool mx) {
            PetitSolutionHints hints;
            hints.a_type = hints.c_type = dtype_code(a_type);
            hints.b_type = mx ? PETIT_DTYPE_MXFP4_E2M1 : PETIT_DTYPE_FP4_E2M1;
            hints.require_high_precision = 0;
            uint64_t id = 0;
            int rc = petit_get_default_solution(&hints, size_m, size_n, size_k, &id);
            TORCH_CHECK(rc == 0, "no kernel for this problem (code ", rc, ")");
            return id;
        },
        py::arg("size_m"), py::arg("size_n"), py::arg("size_k"), py::arg("a_type"),
        py::arg("mx") = false);
    m.def(
        "tune_table_set",
        [](int64_t size_m, int64_t size_n, int64_t size_k, py::object a_type, bool mx,
           int64_t solution_id) {
            PetitSolutionHints hints;
            hints.a_type = hints.c_type = dtype_code(a_type);
            hints.b_type = mx ? PETIT_DTYPE_MXFP4_E2M1 : PETIT_DTYPE_FP4_E2M1;
            hints.require_high_precision = 0;
            int rc = petit_tune_table_set(&hints, size_m, size_n, size_k, (uint64_t)solution_id);
            TORCH_CHECK(rc == 0, "solution id does not belong to these types (code ", rc, ")");
        },
        py::arg("size_m"), py::arg("size_n"), py::arg("size_k"), py::arg("a_type"), py::arg("mx"),
        py::arg("solution_id"));
    m.def("tune_table_load", [](const std::string &path) {
        int n = petit_tune_table_load(path.c_str());
        TORCH_CHECK(n >= 0, "cannot read tune table ", path);
        return n;
    });
    m.def("tune_table_clear", []() { petit_tune_table_clear(); });
    m.def("solution_name", [](uint64_t id) { return std::string(petit_solution_name(id)); });
    m.def("packed_layout_version", []() { return petit_packed_layout_version(); });
    // stream-K workspace of the current stream: watchdog status and explicit release
    m.def("workspace_status", []() {
        int st = 0;
        int rc = petit_workspace_status(at::cuda::getCurrentCUDAStream().stream(), &st);
        TORCH_CHECK(rc == 0, "petit_workspace_status failed with code ", rc);
        return (int64_t)st;
    });
    m.def("release_workspace", []() {
        int rc = petit_release_workspace(at::cuda::getCurrentCUDAStream().stream());
        TORCH_CHECK(rc == 0, "petit_release_workspace failed with code ", rc);
    });
}
