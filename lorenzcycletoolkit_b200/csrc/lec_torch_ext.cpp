// The thin PyTorch C++ extension over the C ABI (BASELINE.json north_star: "hands contiguous ... fields to
// hand-written sm_100a CUDA kernels through a thin PyTorch C++/CUDA extension (C-ABI)").
//
// Two operators, `torch.ops.lec_b200.run_device` (fp fields) and `run_device_packed` (int16 fields): five CUDA tensors
// [slot][level][lat][lon] in, the per-step results written into caller-provided CUDA tensors, asynchronous on torch's
// CURRENT stream of the fields' device.
// It adds nothing to the engine: argument checks, the current stream, and one call of `lec_run_device`
// (include/lec_b200.h), which replaces the arithmetic of the reference's BoxData + four term classes
// (src/utils/box_data.py:157-295, src/analysis/*.py) for a batch of time steps.  There are no torch types in
// liblec_b200.so itself; this file is the only place where the two meet.
//
// Built in-tree by __graft_entry__.build() into lorenzcycletoolkit_b200/_lib/lec_torch_ext.so (g++, no nvcc:
// there is no device code here) and loaded with torch.ops.load_library by lorenzcycletoolkit_b200/engine.py.
#include <cstring>

#include <ATen/ATen.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/library.h>

#include "../../include/lec_b200.h"

namespace {

// handle: the lec_handle* of lec_create as an integer; steps: CPU uint8 tensor holding nsteps lec_step records
// returns the C ABI's status code (LEC_OK = 0): the Python wrapper maps it to the same exceptions as the ctypes route
int64_t run_device(int64_t handle, at::TensorList fields, const at::Tensor& steps, at::Tensor terms,
                const c10::optional<at::Tensor>& levels, const c10::optional<at::Tensor>& flags) {
  TORCH_CHECK(handle != 0, "lec_b200::run_device: null engine handle");
  TORCH_CHECK(fields.size() == 5, "lec_b200::run_device: five fields (T, u, v, omega, Phi), got ", fields.size());
  const at::Tensor& f0 = fields[0];
  TORCH_CHECK(f0.is_cuda() && f0.dim() == 4, "fields must be CUDA tensors [slot][level][lat][lon]");
  for (const at::Tensor& f : fields) {
    TORCH_CHECK(f.is_cuda() && f.is_contiguous() && f.device() == f0.device() && f.scalar_type() == f0.scalar_type() &&
                    f.sizes() == f0.sizes(),
                "fields must be contiguous CUDA tensors of one shape, dtype and device");
  }
  TORCH_CHECK(f0.scalar_type() == at::kFloat || f0.scalar_type() == at::kDouble, "fields must be float32 or float64");
  TORCH_CHECK(steps.device().is_cpu() && steps.scalar_type() == at::kByte && steps.is_contiguous() &&
                  steps.numel() % (int64_t)sizeof(lec_step) == 0,
              "steps must be a contiguous CPU uint8 tensor of lec_step records");
  const int64_t nsteps = steps.numel() / (int64_t)sizeof(lec_step);
  const int64_t nlev = f0.size(1);
  TORCH_CHECK(terms.is_cuda() && terms.device() == f0.device() && terms.scalar_type() == at::kDouble &&
                  terms.is_contiguous() && terms.numel() == nsteps * LEC_NTERMS,
              "terms must be a contiguous CUDA float64 tensor [nsteps][16] on the fields' device");
  double* lv = nullptr;
  if (levels.has_value() && levels->defined()) {
    TORCH_CHECK(levels->is_cuda() && levels->device() == f0.device() && levels->scalar_type() == at::kDouble &&
                    levels->is_contiguous() && levels->numel() == nsteps * LEC_NLEVEL_TERMS * nlev,
                "levels must be a contiguous CUDA float64 tensor [nsteps][19][nlev]");
    lv = levels->data_ptr<double>();
  }
  int32_t* fl = nullptr;
  if (flags.has_value() && flags->defined()) {
    TORCH_CHECK(flags->is_cuda() && flags->device() == f0.device() && flags->scalar_type() == at::kInt &&
                    flags->is_contiguous() && flags->numel() == nsteps,
                "flags must be a contiguous CUDA int32 tensor [nsteps]");
    fl = flags->data_ptr<int32_t>();
  }
  const c10::cuda::CUDAGuard guard(f0.device());
  const c10::cuda::CUDAStream stream = c10::cuda::getCurrentCUDAStream(f0.device().index());
  const void* ptrs[5];
  for (int i = 0; i < 5; ++i) ptrs[i] = fields[i].data_ptr();
  lec_handle* h = reinterpret_cast<lec_handle*>(static_cast<intptr_t>(handle));
  const int rc = lec_run_device(h, ptrs, static_cast<int32_t>(f0.size(0)), reinterpret_cast<const lec_step*>(steps.data_ptr()),
                                static_cast<int32_t>(nsteps), terms.data_ptr<double>(), lv, fl,
                                static_cast<void*>(stream.stream()));
  return rc;
}

// lec_run_device_packed: five int16 CUDA tensors [slot][level][lat][n] whose rows are contiguous and `pitch` =
// stride(2) elements apart (n <= pitch: a [.., :nlon] view of padded rows, or the padded rows themselves);
// decode: CPU uint8 tensor holding one lec_packed_desc (its pitch is taken from the tensors)
int64_t run_device_packed(int64_t handle, at::TensorList fields, const at::Tensor& decode, const at::Tensor& steps,
                          at::Tensor terms, const c10::optional<at::Tensor>& levels, const c10::optional<at::Tensor>& flags) {
  TORCH_CHECK(handle != 0, "lec_b200::run_device_packed: null engine handle");
  TORCH_CHECK(fields.size() == 5, "lec_b200::run_device_packed: five fields (T, u, v, omega, Phi), got ", fields.size());
  const at::Tensor& f0 = fields[0];
  TORCH_CHECK(f0.is_cuda() && f0.dim() == 4 && f0.scalar_type() == at::kShort,
              "packed fields must be int16 CUDA tensors [slot][level][lat][lon]");
  const int64_t pitch = f0.stride(2);
  TORCH_CHECK(f0.stride(3) == 1 && pitch >= f0.size(3) && pitch % 8 == 0 && f0.stride(1) == f0.size(2) * pitch &&
                  f0.stride(0) == f0.size(1) * f0.stride(1),
              "packed fields must have contiguous rows with a pitch (row stride) that is a multiple of 8 elements");
  for (const at::Tensor& f : fields) {
    TORCH_CHECK(f.is_cuda() && f.scalar_type() == at::kShort && f.device() == f0.device() && f.sizes() == f0.sizes() &&
                    f.strides() == f0.strides(),
                "packed fields must be int16 CUDA tensors of one shape, layout and device");
  }
  TORCH_CHECK(decode.device().is_cpu() && decode.scalar_type() == at::kByte && decode.is_contiguous() &&
                  decode.numel() == (int64_t)sizeof(lec_packed_desc),
              "decode must be a contiguous CPU uint8 tensor holding one lec_packed_desc");
  lec_packed_desc pd;
  std::memcpy(&pd, decode.data_ptr(), sizeof pd);
  pd.pitch = static_cast<int32_t>(pitch);
  TORCH_CHECK(steps.device().is_cpu() && steps.scalar_type() == at::kByte && steps.is_contiguous() &&
                  steps.numel() % (int64_t)sizeof(lec_step) == 0,
              "steps must be a contiguous CPU uint8 tensor of lec_step records");
  const int64_t nsteps = steps.numel() / (int64_t)sizeof(lec_step);
  const int64_t nlev = f0.size(1);
  TORCH_CHECK(terms.is_cuda() && terms.device() == f0.device() && terms.scalar_type() == at::kDouble &&
                  terms.is_contiguous() && terms.numel() == nsteps * LEC_NTERMS,
              "terms must be a contiguous CUDA float64 tensor [nsteps][16] on the fields' device");
  double* lv = nullptr;
  if (levels.has_value() && levels->defined()) {
    TORCH_CHECK(levels->is_cuda() && levels->device() == f0.device() && levels->scalar_type() == at::kDouble &&
                    levels->is_contiguous() && levels->numel() == nsteps * LEC_NLEVEL_TERMS * nlev,
                "levels must be a contiguous CUDA float64 tensor [nsteps][19][nlev]");
    lv = levels->data_ptr<double>();
  }
  int32_t* fl = nullptr;
  if (flags.has_value() && flags->defined()) {
    TORCH_CHECK(flags->is_cuda() && flags->device() == f0.device() && flags->scalar_type() == at::kInt &&
                    flags->is_contiguous() && flags->numel() == nsteps,
                "flags must be a contiguous CUDA int32 tensor [nsteps]");
    fl = flags->data_ptr<int32_t>();
  }
  const c10::cuda::CUDAGuard guard(f0.device());
  const c10::cuda::CUDAStream stream = c10::cuda::getCurrentCUDAStream(f0.device().index());
  const int16_t* ptrs[5];
  for (int i = 0; i < 5; ++i) ptrs[i] = static_cast<const int16_t*>(fields[i].data_ptr());
  lec_handle* h = reinterpret_cast<lec_handle*>(static_cast<intptr_t>(handle));
  return lec_run_device_packed(h, &pd, ptrs, static_cast<int32_t>(f0.size(0)), reinterpret_cast<const lec_step*>(steps.data_ptr()),
                               static_cast<int32_t>(nsteps), terms.data_ptr<double>(), lv, fl, static_cast<void*>(stream.stream()));
}

}  // namespace

TORCH_LIBRARY(lec_b200, m) {
  m.def("run_device(int handle, Tensor[] fields, Tensor steps, Tensor(a!) terms, Tensor(b!)? levels, Tensor(c!)? flags) -> int");
  m.def("run_device_packed(int handle, Tensor[] fields, Tensor decode, Tensor steps, Tensor(a!) terms, Tensor(b!)? levels, "
        "Tensor(c!)? flags) -> int");
}

TORCH_LIBRARY_IMPL(lec_b200, CUDA, m) {
  m.impl("run_device", &run_device);
  m.impl("run_device_packed", &run_device_packed);
}
