// Corner points of one stixel on the device, shared by the export (export.cu) and the bird's-eye-view grid (bev.cu).
#pragma once
#include "kernels.h"

namespace isx {

// Stixels::Get3DVertices for one Section, in the header's operation order (xl = i * step, xr = xl + step,
// yt = rows - vT - 1, yb = rows - vB; z = bf / disparity for objects, bf / (alpha_ground * (vhor - v)) for ground,
// 0 for sky; then per corner -z / f * (c - x), -z / f * (c - y), z), with every operation rounded on its own.
// Args: ExportArgs, ObjectArgs or BevArgs (column_step, rows, bf, focal, camera_center_x/y).
template <class Args>
__device__ __forceinline__ void stixel_vertices(const isx_section &s, int col, const Args &a, float alpha, int vhor,
                                                float *v) {
  const float xl = (float)(col * a.column_step), xr = __fadd_rn(xl, (float)a.column_step);
  const float yt = (float)(a.rows - s.vT - 1), yb = (float)(a.rows - s.vB);
  float zt = 0.0f, zb = 0.0f;
  if (s.type == OBJECT) {
    zt = zb = __fdiv_rn(a.bf, s.disparity);
  } else if (s.type == GROUND) {
    zt = __fdiv_rn(a.bf, __fmul_rn(alpha, (float)(vhor - s.vT)));
    zb = __fdiv_rn(a.bf, __fmul_rn(alpha, (float)(vhor - s.vB)));
  }
  const float cx[4] = {xl, xr, xr, xl}, cy[4] = {yt, yt, yb, yb}, cz[4] = {zt, zt, zb, zb};
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const float q = __fdiv_rn(-cz[k], a.focal);
    v[3 * k + 0] = __fmul_rn(q, __fsub_rn(a.camera_center_x, cx[k]));
    v[3 * k + 1] = __fmul_rn(q, __fsub_rn(a.camera_center_y, cy[k]));
    v[3 * k + 2] = cz[k];
  }
}

}  // namespace isx
