// quant_cuda -- the torch extension over the C ABI of libfpq_b200.so (include/fpq_b200.h).
//
// It carries the name and the entry point of the reference's extension (quant/quant.cpp:27-29:
// `m.def("quant", &quant, ...)`, called as `quant_array, _ = quant_cuda.quant(quant_array, quant_grid)` at 91 sites of
// models_fp_quant*/quant_utils.py), so putting fpqvar_b200/dropin on sys.path ahead of the reference's quant/ build directory
// replaces the reference's kernel with fpq_quant_grid and nothing else changes.  Next to it are the fused operators
// fpqvar_b200/ops.py calls: argument checks, output allocation and the launch on torch's current stream in C++, a few
// microseconds of host time per call instead of the ~10 us of a ctypes round trip with Python-side checks (the early scales
// of a VAR pass are host-bound).  No arithmetic happens here and there is no fallback: every operator ends in one C-ABI call.
#include <torch/extension.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>

#include "../../include/fpq_b200.h"

namespace {

void check_rc(int rc, const char* what) {
    if (rc == FPQ_OK) return;
    if (rc == FPQ_ERR_CUDA) throw std::runtime_error(std::string(what) + ": CUDA error: " + fpq_last_cuda_error());
    throw std::runtime_error(std::string(what) + (rc == FPQ_ERR_ARG ? ": invalid argument" : rc == FPQ_ERR_UNSUPPORTED ? ": unsupported configuration" : ": error"));
}

void require_cuda(const at::Tensor& t, const char* what) {
    if (!t.is_cuda()) throw std::runtime_error(std::string(what) + ": expected a CUDA tensor (fpqvar_b200 has no CPU fallback); got " + t.device().str());
}

int dtype_code(const at::Tensor& t, const char* what) {
    if (t.scalar_type() == at::kFloat) return FPQ_F32;
    if (t.scalar_type() == at::kHalf) return FPQ_F16;
    throw std::runtime_error(std::string(what) + ": dtype " + std::string(c10::toString(t.scalar_type())) + " is not supported (float16 / float32 only)");
}

void* stream_of(const at::Tensor& t) { return at::cuda::getCurrentCUDAStream(t.get_device()).stream(); }

// rows that share a scale: row_len <= 0 means "the last dimension"
std::pair<size_t, size_t> rows_of(const at::Tensor& x, int64_t row_len) {
    if (row_len <= 0) row_len = x.dim() > 0 ? x.size(-1) : 1;
    const int64_t n = x.numel();
    if (row_len <= 0 || n % row_len != 0) throw std::runtime_error("numel " + std::to_string(n) + " is not a multiple of the group/row length " + std::to_string(row_len));
    return {size_t(n / row_len), size_t(row_len)};
}

// ---- the reference's entry point (quant/quant.cpp:17-29) -----------------------------------------------------------------
std::vector<at::Tensor> quant(at::Tensor x, at::Tensor y) {
    require_cuda(x, "quant_cuda.quant");
    require_cuda(y, "quant_cuda.quant(grid)");
    if (x.scalar_type() != at::kFloat) throw std::runtime_error("quant_cuda.quant: x must be float32 (the reference reads every input as float, quant_kernel.cu:28)");
    c10::cuda::CUDAGuard guard(x.device());
    x = x.contiguous();
    at::Tensor grid = y.to(at::kFloat).contiguous();
    at::Tensor z = at::empty_like(x);
    check_rc(fpq_quant_grid(x.data_ptr<float>(), grid.data_ptr<float>(), int(grid.numel()), size_t(x.numel()), z.data_ptr<float>(), FPQ_TIE_KERNEL,
                            stream_of(x)),
             "fpq_quant_grid");
    // the reference's second output is a zero tensor it never writes (quant_kernel.cu:49,58); a zero-stride view costs nothing
    at::Tensor idx = at::zeros({}, x.options()).expand(x.sizes());
    return {z, idx};
}

// ---- fused operators (fpqvar_b200/ops.py) ----------------------------------------------------------------------------------
at::Tensor fake_quant(at::Tensor x, int64_t format, int64_t row_len, int64_t tie, int64_t flags, int64_t out_dtype) {
    require_cuda(x, "fake_quant");
    const int din = dtype_code(x, "fake_quant");
    c10::cuda::CUDAGuard guard(x.device());
    x = x.contiguous();
    const int dout = out_dtype < 0 ? (tie == FPQ_TIE_KERNEL ? din : FPQ_F32) : int(out_dtype);
    at::Tensor out = at::empty(x.sizes(), x.options().dtype(dout == FPQ_F32 ? at::kFloat : at::kHalf));
    const auto r = rows_of(x, row_len);
    check_rc(fpq_fake_quant(x.data_ptr(), out.data_ptr(), r.first, r.second, din, dout, int(format), int(tie), unsigned(flags), stream_of(x)), "fpq_fake_quant");
    return out;
}

at::Tensor fake_quant_signsplit(at::Tensor x, int64_t split, int64_t row_len, int64_t tie, int64_t flags, c10::optional<at::Tensor> workspace,
                                int64_t out_dtype) {
    require_cuda(x, "fake_quant_signsplit");
    const int din = dtype_code(x, "signsplit");
    c10::cuda::CUDAGuard guard(x.device());
    x = x.contiguous();
    const int dout = out_dtype < 0 ? (tie == FPQ_TIE_KERNEL ? din : FPQ_F32) : int(out_dtype);
    at::Tensor out = at::empty(x.sizes(), x.options().dtype(dout == FPQ_F32 ? at::kFloat : at::kHalf));
    const auto r = rows_of(x, row_len);
    void* ws = nullptr;
    if (workspace.has_value()) {
        const at::Tensor& w = *workspace;
        if (!w.is_cuda() || w.get_device() != x.get_device() || w.scalar_type() != at::kInt || w.numel() < 2 || !w.is_contiguous())
            throw std::runtime_error("fake_quant_signsplit: the workspace must be 2 contiguous int32 on the input's device");
        ws = w.data_ptr();
    }
    check_rc(fpq_fake_quant_signsplit(x.data_ptr(), out.data_ptr(), r.first, r.second, din, dout, int(split), int(tie), unsigned(flags), ws, stream_of(x)),
             "fpq_fake_quant_signsplit");
    return out;
}

const float* smooth_ptr(c10::optional<at::Tensor>& smooth, const at::Tensor& x, int64_t n_cols, const char* what) {
    if (!smooth.has_value()) return nullptr;
    at::Tensor s = smooth->detach();
    require_cuda(s, what);
    if (s.numel() != n_cols) throw std::runtime_error(std::string(what) + ": smooth has " + std::to_string(s.numel()) + " entries, expected " + std::to_string(n_cols));
    if (s.get_device() != x.get_device()) throw std::runtime_error(std::string(what) + ": smooth lives on another device");
    if (s.scalar_type() != at::kFloat || !s.is_contiguous()) s = s.to(at::kFloat).contiguous();       // ordered like any producer: the kernels read it after their dependency wait
    smooth = s;
    return s.data_ptr<float>();
}

// Arguments of the rotate operators, checked and converted in one place for both outputs (fp16 and codes).  `scale` / `shift`
// present: the adaLN-modulated entry, x = [B, ..., C] with [B, 1, C] operands.  The device guard lives as long as the call.
struct RotateCall {
    c10::cuda::OptionalCUDAGuard guard;
    at::Tensor x;
    at::Tensor mods[2];                 // fp32 gain or scale, fp32 shift (modulated entry only)
    const float* sp = nullptr;          // smooth
    uint32_t bits[4] = {0, 0, 0, 0};
    size_t rows = 0, cols = 0, rows_per_batch = 0;
    int flags = 0;

    RotateCall(at::Tensor x_, const at::Tensor* scale, const at::Tensor* shift, c10::optional<at::Tensor>& smooth, const std::vector<int64_t>& sign_bits,
               const std::string& what) {
        const bool mod = scale != nullptr;
        require_cuda(x_, what.c_str());
        if (!mod && x_.scalar_type() != at::kFloat) throw std::runtime_error(what + ": x must be float32 (the adaLN-modulated LayerNorm output)");
        if (mod && (x_.scalar_type() != at::kFloat || x_.dim() < 2)) throw std::runtime_error(what + ": x must be float32 [B, ..., C]");
        if (sign_bits.size() != 4) throw std::runtime_error(what + ": sign_bits must hold 4 words");
        guard.set_device(x_.device());
        x = x_.contiguous();
        const int64_t c = x.dim() > 0 ? x.size(-1) : 0;
        cols = size_t(c);
        rows = c ? size_t(x.numel() / c) : 0;
        if (mod) {
            const int64_t b = x.size(0);
            const int64_t rpb = (b * c) ? x.numel() / (b * c) : 0;
            mods[0] = scale->detach();
            mods[1] = shift->detach();
            const char* names[2] = {"scale", "shift"};
            for (int i = 0; i < 2; ++i) {
                const at::Tensor& t = mods[i];
                require_cuda(t, (what + "(scale/shift)").c_str());
                if (t.numel() != b * c || t.dim() < 1 || t.size(0) != b || t.size(-1) != c)
                    throw std::runtime_error(std::string(names[i]) + " must be [B, 1, C] = [" + std::to_string(b) + ", 1, " + std::to_string(c) + "]");
                if (t.scalar_type() != at::kFloat && t.scalar_type() != at::kHalf) throw std::runtime_error(std::string(names[i]) + " must be float32 or float16");
            }
            // fp16 adaLN tensors (the reference's fp16 autocast): `scale.add(1)` is an fp16 add there; do it with the same ATen op on
            // the tiny [B, 1, C] tensor and hand the rounded result to the kernel as a gain
            if (mods[0].scalar_type() == at::kHalf) { mods[0] = mods[0].add(1); flags = FPQ_MOD_GAIN; }
            for (auto& t : mods) t = t.to(at::kFloat).contiguous();
            rows_per_batch = size_t(rpb);
            rows = size_t(b * rpb);
        }
        sp = smooth_ptr(smooth, x, c, (what + "(smooth)").c_str());
        for (int i = 0; i < 4; ++i) bits[i] = uint32_t(sign_bits[i]);
    }
    const float* scale_ptr() const { return mods[0].data_ptr<float>(); }
    const float* shift_ptr() const { return mods[1].data_ptr<float>(); }
};

std::vector<at::Tensor> transform_rotate_quant(at::Tensor x, c10::optional<at::Tensor> smooth, std::vector<int64_t> sign_bits, int64_t format, bool want_rotated) {
    RotateCall r(x, nullptr, nullptr, smooth, sign_bits, "transform_rotate_quant");
    at::Tensor out = at::empty(r.x.sizes(), r.x.options().dtype(at::kHalf));
    at::Tensor rot;
    if (want_rotated) rot = at::empty_like(out);
    check_rc(fpq_transform_rotate_quant(r.x.data_ptr<float>(), r.sp, r.bits, out.data_ptr(), want_rotated ? rot.data_ptr() : nullptr, r.rows, r.cols,
                                        int(format), stream_of(r.x)),
             "fpq_transform_rotate_quant");
    if (want_rotated) return {out, rot};
    return {out};
}

std::vector<at::Tensor> modulate_transform_rotate_quant(at::Tensor x, at::Tensor scale, at::Tensor shift, c10::optional<at::Tensor> smooth,
                                                        std::vector<int64_t> sign_bits, int64_t format, bool want_rotated) {
    RotateCall r(x, &scale, &shift, smooth, sign_bits, "modulate_transform_rotate_quant");
    at::Tensor out = at::empty(r.x.sizes(), r.x.options().dtype(at::kHalf));
    at::Tensor rot;
    if (want_rotated) rot = at::empty_like(out);
    check_rc(fpq_modulate_transform_rotate_quant(r.x.data_ptr<float>(), r.scale_ptr(), r.shift_ptr(), r.rows_per_batch, r.sp, r.bits, out.data_ptr(),
                                                 want_rotated ? rot.data_ptr() : nullptr, r.rows, r.cols, int(format), r.flags, stream_of(r.x)),
             "fpq_modulate_transform_rotate_quant");
    if (want_rotated) return {out, rot};
    return {out};
}

// codes output: (codes uint8 [rows_pad * C], scales fp32 [C / 128, rows_pad]), the operand layout of fpq_gemm_codes
std::vector<at::Tensor> codes_buffers(const RotateCall& r) {
    const size_t rows_pad = fpq_codes_rows_padded(r.rows);
    at::Tensor codes = at::empty({int64_t(rows_pad * r.cols)}, r.x.options().dtype(at::kByte));
    at::Tensor scales = at::empty({int64_t(r.cols / 128), int64_t(rows_pad)}, r.x.options().dtype(at::kFloat));
    return {codes, scales};
}

std::vector<at::Tensor> transform_rotate_pack_codes(at::Tensor x, c10::optional<at::Tensor> smooth, std::vector<int64_t> sign_bits, int64_t format) {
    RotateCall r(x, nullptr, nullptr, smooth, sign_bits, "transform_rotate_pack_codes");
    std::vector<at::Tensor> o = codes_buffers(r);
    check_rc(fpq_transform_rotate_pack_codes(r.x.data_ptr<float>(), r.sp, r.bits, o[0].data_ptr<uint8_t>(), o[1].data_ptr<float>(), r.rows, r.cols,
                                             int(format), stream_of(r.x)),
             "fpq_transform_rotate_pack_codes");
    return o;
}

std::vector<at::Tensor> modulate_transform_rotate_pack_codes(at::Tensor x, at::Tensor scale, at::Tensor shift, c10::optional<at::Tensor> smooth,
                                                             std::vector<int64_t> sign_bits, int64_t format) {
    RotateCall r(x, &scale, &shift, smooth, sign_bits, "modulate_transform_rotate_pack_codes");
    std::vector<at::Tensor> o = codes_buffers(r);
    check_rc(fpq_modulate_transform_rotate_pack_codes(r.x.data_ptr<float>(), r.scale_ptr(), r.shift_ptr(), r.rows_per_batch, r.sp, r.bits,
                                                      o[0].data_ptr<uint8_t>(), o[1].data_ptr<float>(), r.rows, r.cols, int(format), r.flags,
                                                      stream_of(r.x)),
             "fpq_modulate_transform_rotate_pack_codes");
    return o;
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
    m.doc() = "fpq_b200 torch extension over the C ABI of libfpq_b200.so; `quant` is the reference's quant_cuda.quant";
    m.def("quant", &quant, py::arg("x"), py::arg("y"), "quant(x, y) -> (z, idx): nearest entry of the grid y, the reference's scan semantics (quant/quant.cpp:27-29)");
    m.def("fake_quant", &fake_quant);
    m.def("fake_quant_signsplit", &fake_quant_signsplit);
    m.def("transform_rotate_quant", &transform_rotate_quant);
    m.def("modulate_transform_rotate_quant", &modulate_transform_rotate_quant);
    m.def("transform_rotate_pack_codes", &transform_rotate_pack_codes);
    m.def("modulate_transform_rotate_pack_codes", &modulate_transform_rotate_pack_codes);
    m.def("launch_count", []() { return fpq_launch_count(); });
    m.def("version", []() { return std::string(fpq_version()); });
}
