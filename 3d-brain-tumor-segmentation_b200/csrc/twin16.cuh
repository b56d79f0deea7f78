// b3d — the store side of a P16 operand twin ([B, D, H, C/8, W, 8], common.cuh) for kernels that stream a fp32 NDHWC
// tensor one 16-byte CELL (8 consecutive channels of a voxel) per thread and step: the twin position of a thread's
// first cell, its advance by a loop stride without a division, the 16-bit packing and the store.  Shared by the
// GroupNorm apply kernels of both semantics (norm.cu, norm_channel.cu).
#pragma once
#include "common.cuh"

namespace b3d {

struct Twin16 {
  uint4* p;         // first twin (type `bf16`), nullptr: none
  uint4* p2;        // optional second twin, always bf16
  unsigned W, C8;   // voxels per row, channel octets
  unsigned rows;    // D*H rows per sample
  int bf16;
};
struct CellPos {
  unsigned long long rowbase;   // (b * rows + row) * C8 + c8
  unsigned w;                   // voxel inside the row
  unsigned dr1, dw1;            // small step (to the thread's next cell of a pass: one block of cells on) as rows / voxels
  unsigned dr2, dw2;            // big step (from the last cell of a pass to the first of the next)
};
// elem: index of the thread's first element inside sample b; cells1 / cells2: the two strides in cells (multiples of C8)
__device__ __forceinline__ CellPos cell_pos(const Twin16& o, unsigned b, unsigned long long elem, unsigned cells1,
                                            unsigned long long cells2) {
  const unsigned cell = (unsigned)(elem >> 3);
  const unsigned vox = cell / o.C8, c8 = cell - vox * o.C8;
  const unsigned row = vox / o.W;
  CellPos k;
  k.rowbase = ((unsigned long long)b * o.rows + row) * o.C8 + c8;
  k.w = vox - row * o.W;
  const unsigned v1 = cells1 / o.C8;
  const unsigned long long v2 = cells2 / o.C8;
  k.dr1 = v1 / o.W; k.dw1 = v1 - k.dr1 * o.W;
  k.dr2 = (unsigned)(v2 / o.W); k.dw2 = (unsigned)(v2 - (unsigned long long)k.dr2 * o.W);
  return k;
}
__device__ __forceinline__ void cell_step(const Twin16& o, CellPos& k, unsigned dr, unsigned dw) {
  k.w += dw;
  unsigned r = dr;
  if (k.w >= o.W) { k.w -= o.W; ++r; }
  k.rowbase += (unsigned long long)r * o.C8;
}
__device__ __forceinline__ uint32_t pk16(float lo, float hi, int bf16) {
  uint32_t r;
  if (bf16) asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  else asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ void cell_store(const Twin16& o, const CellPos& k, const float (&v)[8]) {
  const unsigned long long idx = k.rowbase * o.W + k.w;
  o.p[idx] = make_uint4(pk16(v[0], v[1], o.bf16), pk16(v[2], v[3], o.bf16), pk16(v[4], v[5], o.bf16),
                        pk16(v[6], v[7], o.bf16));
  if (o.p2 != nullptr)
    o.p2[idx] = make_uint4(pk16(v[0], v[1], 1), pk16(v[2], v[3], 1), pk16(v[4], v[5], 1), pk16(v[6], v[7], 1));
}

// Twin16 of the twin tensor(s) t1_ (and the optional bf16 t2_) of the fp32 NDHWC tensor x
inline int twin_view(const DLTensor* t1_, const DLTensor* t2_, const TView& x, Twin16* tw) {
  tw->p = nullptr; tw->p2 = nullptr;
  P16View v;
  B3D_TRY(view_p16(t1_, "twin", &v));
  B3D_REQUIRE(x.ndim == 5 && v.B == x.shape[0] && v.D == x.shape[1] && v.H == x.shape[2] && v.W == x.shape[3] &&
                  8 * v.C8 == x.shape[4], B3D_ERR_SHAPE, "twin: must be the [B, D, H, C/8, W, 8] form of the fp32 tensor");
  tw->p = (uint4*)v.p; tw->W = (unsigned)v.W; tw->C8 = (unsigned)v.C8; tw->rows = (unsigned)(v.D * v.H); tw->bf16 = v.bf16;
  if (t2_ != nullptr) {
    P16View v2;
    B3D_TRY(view_p16(t2_, "twin (bf16)", &v2));
    B3D_REQUIRE(v2.bf16 && v2.B == v.B && v2.D == v.D && v2.H == v.H && v2.W == v.W && v2.C8 == v.C8, B3D_ERR_SHAPE,
                "second twin: bf16, same shape");
    tw->p2 = (uint4*)v2.p;
  }
  return B3D_OK;
}

}  // namespace b3d
