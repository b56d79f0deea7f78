// b3d — shared helpers for the sm_100a kernels and the C-ABI layer.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/b3d_dlpack.h"

#define B3D_OK 0
#define B3D_ERR_ARG (-1)
#define B3D_ERR_DEVICE (-2)
#define B3D_ERR_DTYPE (-3)
#define B3D_ERR_LAYOUT (-4)
#define B3D_ERR_SHAPE (-5)
#define B3D_ERR_CUDA (-6)
#define B3D_ERR_UNSUPPORTED (-7)

namespace b3d {

void set_error(const char* fmt, ...);

// ---- DLPack validation ---------------------------------------------------------------------
struct TView {
  void* p = nullptr;
  int ndim = 0;
  int64_t shape[6] = {0, 0, 0, 0, 0, 0};
  int64_t pitch = 0;  // elements between consecutive "rows" of the last dim (== shape[last] if compact)
  int64_t numel = 0;
  int device = 0;
};

// dtype codes
enum { DT_F32 = 0, DT_F64 = 1, DT_I64 = 2, DT_BF16 = 3, DT_F16 = 4, DT_U8 = 5 };

// Validates: CUDA device, dtype, ndim, and compact row-major strides; if allow_pitch, the last
// dim may be a channel slice of a wider NDHWC buffer (stride[last]==1, outer strides compact
// w.r.t. a pitch >= shape[last]).
int view(const DLTensor* t, int dtype, int ndim, bool allow_pitch, const char* name, TView* out);

// "P16" operand twin of an activation / gradient tensor (DESIGN.md section 3): 16-bit [B, D, H, C/8, W, 8] — channel
// octets as planes inside every (d, h) row, so that a halo row of one plane is W*16 contiguous bytes (wide TMA rows)
// and a voxel's 8 channels are one 16-byte UMMA cell.  fp16 for forward activations, bf16 for gradients.
struct P16View {
  void* p = nullptr;
  int B = 0, D = 0, H = 0, W = 0, C8 = 0;   // C = 8 * C8 channels
  int bf16 = 0;                            // 1 = bf16, 0 = fp16
};
int view_p16(const DLTensor* t, const char* name, P16View* out);

inline int cuda_ok(cudaError_t e, const char* what) {
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return B3D_ERR_CUDA;
  }
  return B3D_OK;
}

#define B3D_TRY(expr)            \
  do {                           \
    int _rc = (expr);            \
    if (_rc != B3D_OK) return _rc; \
  } while (0)

#define B3D_LAUNCH_CHECK(name) B3D_TRY(b3d::cuda_ok(cudaGetLastError(), name))

#define B3D_REQUIRE(cond, code, ...) \
  do {                               \
    if (!(cond)) {                   \
      b3d::set_error(__VA_ARGS__);   \
      return code;                   \
    }                                \
  } while (0)

int sm_count();

// ---- device helpers -------------------------------------------------------------------------
// Programmatic dependent launch: a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may start
// its CTAs (prologue: barrier init, TMEM allocation) while the previous kernel in the stream drains; pdl_wait() blocks
// until that kernel has completed and its writes are visible.  pdl_trigger() in the previous kernel allows the start.
// Both are no-ops in launches without the attribute / without a dependent.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// <<<grid, block, smem, s>>> with the programmatic-serialization attribute.  Only for kernels that read nothing the
// previous kernel writes before their pdl_wait().
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                              Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of NV values per thread; result valid in thread 0.  smem: NV*32 floats.
template <int NV, typename T>
__device__ __forceinline__ void block_sum(T (&v)[NV], T* smem) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) smem[i * 32 + wid] = v[i];
  }
  __syncthreads();
  if (wid == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      T t = lane < nw ? smem[i * 32 + lane] : T(0);
      v[i] = warp_sum(t);
    }
  }
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }

// streaming 128-bit accesses (read-once / write-once tensors)
__device__ __forceinline__ float4 ld_stream(const float4* p) {
  float4 r;
  asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream(float4* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w));
}

// 8 consecutive floats of a read-once / write-once tensor.  Stores: ONE 256-bit access when 32-byte aligned (sm_100
// STG.256: a lane owns a whole 32-byte sector, where a pair of 128-bit stores makes every warp instruction write 32
// sectors half), else the pair.
__device__ __forceinline__ void ld8(const float* p, float (&v)[8]) {
  // loads stay a pair of 128-bit accesses: measured on B200 (tools/hbm_bench.py) the 256-bit form is no faster for the
  // apply kernels and SLOWER for the reducing ones (gn_bwd_reduce 67 -> 58 % of the HBM peak)
  const float4 a = ld_stream(reinterpret_cast<const float4*>(p));
  const float4 c = ld_stream(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
}
__device__ __forceinline__ void st8(float* p, const float (&v)[8]) {
  if ((reinterpret_cast<unsigned long long>(p) & 31ull) == 0) {
    asm volatile("st.global.L1::no_allocate.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]),
                 "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]));
  } else {
    st_stream(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
    st_stream(reinterpret_cast<float4*>(p) + 1, make_float4(v[4], v[5], v[6], v[7]));
  }
}

}  // namespace b3d
