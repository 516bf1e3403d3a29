// 8-bit frame codes (include/ltxcuda.h, LTX_FRAMES_*): the arithmetic shared by the fused conv_out store (conv3d.cu, epilogue
// modes 5 / 6) and the streaming converter (vae.cu), so that both produce the same bytes from the same fp32 values.
// Every operation is an explicit round-to-nearest intrinsic: nothing may be contracted into an FMA differently in the two
// callers, and tests/frames_u8_ref.py restates each step in numpy float32.
#pragma once

#include <cstdint>

namespace ltx {

// RGB8: q = (uint8_t)(v * 255.0f) -- one fp32 multiply, then truncation (v already clipped to [0, 1])
__device__ __forceinline__ uint32_t rgb8_code(float v) { return __float2uint_rz(__fmul_rn(v, 255.0f)); }

__device__ __forceinline__ float bt709_luma(float r, float g, float b) {
  return __fadd_rn(__fadd_rn(__fmul_rn(0.2126f, r), __fmul_rn(0.7152f, g)), __fmul_rn(0.0722f, b));
}

__device__ __forceinline__ uint32_t code_u8(float x) {   // rint (ties to even), clamped to a byte
  return static_cast<uint32_t>(min(max(__float2int_rn(x), 0), 255));
}

// I420 (BT.709, limited range) of one 2x2 chroma cell: p[i] = (R, G, B) of pixel i = 2 * row + col, clipped to [0, 1].
//   y[i] = rint(16 + 219 Y'(p[i]))
//   cb   = rint(128 + 224 (B_m - Y'(m)) / 1.8556),  cr = rint(128 + 224 (R_m - Y'(m)) / 1.5748)
// m = the cell's mean colour, each component summed as ((p0 + p1) + p2) + p3, then * 0.25.
__device__ __forceinline__ void i420_cell(const float (&p)[4][3], uint32_t (&y)[4], uint32_t& cb, uint32_t& cr) {
#pragma unroll
  for (int i = 0; i < 4; ++i) y[i] = code_u8(__fadd_rn(16.0f, __fmul_rn(219.0f, bt709_luma(p[i][0], p[i][1], p[i][2]))));
  float m[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) m[c] = __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(p[0][c], p[1][c]), p[2][c]), p[3][c]), 0.25f);
  const float ym = bt709_luma(m[0], m[1], m[2]);
  cb = code_u8(__fadd_rn(128.0f, __fdiv_rn(__fmul_rn(224.0f, __fsub_rn(m[2], ym)), 1.8556f)));
  cr = code_u8(__fadd_rn(128.0f, __fdiv_rn(__fmul_rn(224.0f, __fsub_rn(m[0], ym)), 1.5748f)));
}

}  // namespace ltx
