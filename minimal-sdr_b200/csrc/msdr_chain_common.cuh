// msdr_chain_common.cuh — device code shared by the fused receive-chain kernels:
// demodulation kind of a mode, biquad cascade helpers (biquad warps).
#pragma once
#include "msdr_device.cuh"
#include "msdr_internal.h"

namespace msdr {

__device__ __forceinline__ int demod_kind_of(int mode, uint32_t am_q31)
{
  // Minimal-SDR.ino:589-628: LSB, USB; AM/CW (+SYNCAM on Teensy 3.2) envelope
  if (mode == 2) return 0;
  if (mode == 3) return 1;
  if (mode == 0) return 3;
  return am_q31 ? 3 : 2;
}

// two samples (one packed word) through NS fused stages — integer (IMAD.HI) representation, values carried as v << 16
template <int NS>
__device__ __forceinline__ uint32_t bq_word(BqStage (&st)[NS], uint32_t w)
{
  int xe = (int)(w << 16), xo = (int)(w & 0xFFFF0000u);
#pragma unroll
  for (int k = 0; k < NS; ++k) xe = bq_step(st[k], xe);
#pragma unroll
  for (int k = 0; k < NS; ++k) xo = bq_step(st[k], xo);
  return __byte_perm((uint32_t)xe, (uint32_t)xo, 0x7632);
}
template <int NS>
__device__ __forceinline__ uint32_t bq_word(BqStageW (&st)[NS], uint32_t w)
{
  int xe, xo = (int)(w & 0xFFFF0000u);
  asm("prmt.b32 %0, %1, 0, 0x1044;" : "=r"(xe) : "r"(w)); // w << 16 on the ALU pipe (ptxas turns a shift into IMAD.U32 x 0x10000: multiplier pipe)
#pragma unroll
  for (int k = 0; k < NS; ++k) xe = bq_step(st[k], xe);
#pragma unroll
  for (int k = 0; k < NS; ++k) xo = bq_step(st[k], xo);
  return __byte_perm((uint32_t)xe, (uint32_t)xo, 0x7632);
}
template <int NS>
__device__ __forceinline__ uint32_t bq_word(BqStageWS (&st)[NS], uint32_t w)
{
  int xe, xo = (int)(w & 0xFFFF0000u);
  asm("prmt.b32 %0, %1, 0, 0x1044;" : "=r"(xe) : "r"(w));
#pragma unroll
  for (int k = 0; k < NS; ++k) xe = bq_step(st[k], xe);
#pragma unroll
  for (int k = 0; k < NS; ++k) xo = bq_step(st[k], xo);
  return __byte_perm((uint32_t)xe, (uint32_t)xo, 0x7632);
}
template <int NS>
__device__ __forceinline__ uint32_t bq_word(BqStageHS (&st)[NS], uint32_t w)
{
  int xe = (int)(w << 16), xo = (int)(w & 0xFFFF0000u);
#pragma unroll
  for (int k = 0; k < NS; ++k) xe = bq_step(st[k], xe);
#pragma unroll
  for (int k = 0; k < NS; ++k) xo = bq_step(st[k], xo);
  return __byte_perm((uint32_t)xe, (uint32_t)xo, 0x7632);
}
// hybrid stage (feed-forward on the FP64 pipe): inputs sign-extended with one PRMT each, outputs arrive as y << 16
template <int NS>
__device__ __forceinline__ uint32_t bq_word(BqStageH (&st)[NS], uint32_t w)
{
  int xe, xo; // prmt selector bit 3 replicates the sign of the selected byte: one instruction per sign extension
  asm("prmt.b32 %0, %1, 0, 0x9910;" : "=r"(xe) : "r"(w));
  asm("prmt.b32 %0, %1, 0, 0xBB32;" : "=r"(xo) : "r"(w));
  int ye = bq_step(st[0], xe);
#pragma unroll
  for (int k = 1; k < NS; ++k) ye = bq_step(st[k], ye >> 16); // stages take the int16 value, hand on y << 16
  int yo = bq_step(st[0], xo);
#pragma unroll
  for (int k = 1; k < NS; ++k) yo = bq_step(st[k], yo >> 16);
  return __byte_perm((uint32_t)ye, (uint32_t)yo, 0x7632);
}

template <int NS>
__device__ __forceinline__ uint32_t bq_word(BqStageC (&st)[NS], uint32_t w)
{
  int xe, xo; // prmt selector bit 3 replicates the sign of the selected byte: one instruction per sign extension
  asm("prmt.b32 %0, %1, 0, 0x9910;" : "=r"(xe) : "r"(w));
  asm("prmt.b32 %0, %1, 0, 0xBB32;" : "=r"(xo) : "r"(w));
  int ye = bq_step(st[0], xe);
#pragma unroll
  for (int k = 1; k < NS; ++k) ye = bq_step(st[k], ye >> 16); // stages take the int16 value, hand on y << 16
  int yo = bq_step(st[0], xo);
#pragma unroll
  for (int k = 1; k < NS; ++k) yo = bq_step(st[k], yo >> 16);
  return __byte_perm((uint32_t)ye, (uint32_t)yo, 0x7632);
}
__device__ __forceinline__ void bq_load_stage(BqStageC &s, uint32_t &flag, const int32_t *__restrict__ bq, uint32_t Cpad, int obj, int stage, uint32_t ch)
{
  const int32_t *b = bq + (size_t)((obj * 4 + stage) * 8) * Cpad + ch;
  bq_set_coefs(s, __ldcg(b + 0 * (size_t)Cpad), __ldcg(b + 1 * (size_t)Cpad), __ldcg(b + 2 * (size_t)Cpad), __ldcg(b + 3 * (size_t)Cpad),
               __ldcg(b + 4 * (size_t)Cpad));
  const uint32_t w5 = (uint32_t)__ldcg(b + 5 * (size_t)Cpad);
  s.x1 = bq_d_from_int((int)w5 >> 16); s.x2 = bq_d_from_int((int)(short)(w5 & 0xFFFFu));
  bq_unpack_hist((uint32_t)__ldcg(b + 6 * (size_t)Cpad), s.y1, s.y2);
  const uint32_t w7 = (uint32_t)__ldcg(b + 7 * (size_t)Cpad);
  s.res = (int)(w7 & 0x3FFFu);
  flag = w7 & 0x80000000u;
}
__device__ __forceinline__ void bq_store_stage(const BqStageC &s, uint32_t flag, int32_t *__restrict__ bq, uint32_t Cpad, int obj, int stage, uint32_t ch)
{
  int32_t *b = bq + (size_t)((obj * 4 + stage) * 8) * Cpad + ch;
  b[5 * (size_t)Cpad] = (int32_t)(((uint32_t)bq_int_from_d(s.x1) << 16) | ((uint32_t)bq_int_from_d(s.x2) & 0xFFFFu));
  b[6 * (size_t)Cpad] = (int32_t)bq_pack_hist(s.y1, s.y2);
  b[7 * (size_t)Cpad] = (int32_t)((uint32_t)s.res | flag);
}

template <int NS>
__device__ __forceinline__ uint32_t bq_word(BqStageE (&st)[NS], uint32_t w)
{
  int xe, xo;
  asm("prmt.b32 %0, %1, 0, 0x9910;" : "=r"(xe) : "r"(w));
  asm("prmt.b32 %0, %1, 0, 0xBB32;" : "=r"(xo) : "r"(w));
#pragma unroll
  for (int k = 0; k < NS; ++k) xe = bq_step(st[k], xe);
#pragma unroll
  for (int k = 0; k < NS; ++k) xo = bq_step(st[k], xo);
  return __byte_perm((uint32_t)xe, (uint32_t)xo, 0x5410);
}
__device__ __forceinline__ void bq_load_stage(BqStageE &s, uint32_t &flag, const int32_t *__restrict__ bq, uint32_t Cpad, int obj, int stage, uint32_t ch)
{
  const int32_t *b = bq + (size_t)((obj * 4 + stage) * 8) * Cpad + ch;
  bq_set_coefs(s, __ldcg(b + 0 * (size_t)Cpad), __ldcg(b + 1 * (size_t)Cpad), __ldcg(b + 2 * (size_t)Cpad), __ldcg(b + 3 * (size_t)Cpad),
               __ldcg(b + 4 * (size_t)Cpad));
  const uint32_t w5 = (uint32_t)__ldcg(b + 5 * (size_t)Cpad), w6 = (uint32_t)__ldcg(b + 6 * (size_t)Cpad);
  s.x1 = bq_d_from_int((int)w5 >> 16); s.x2 = bq_d_from_int((int)(short)(w5 & 0xFFFFu));
  s.y1 = bq_d_from_int((int)w6 >> 16); s.y2 = bq_d_from_int((int)(short)(w6 & 0xFFFFu));
  const uint32_t w7 = (uint32_t)__ldcg(b + 7 * (size_t)Cpad);
  s.res = (int)(w7 & 0x3FFFu);
  flag = w7 & 0x80000000u;
}
__device__ __forceinline__ void bq_store_stage(const BqStageE &s, uint32_t flag, int32_t *__restrict__ bq, uint32_t Cpad, int obj, int stage, uint32_t ch)
{
  int32_t *b = bq + (size_t)((obj * 4 + stage) * 8) * Cpad + ch;
  b[5 * (size_t)Cpad] = (int32_t)(((uint32_t)bq_int_from_d(s.x1) << 16) | ((uint32_t)bq_int_from_d(s.x2) & 0xFFFFu));
  b[6 * (size_t)Cpad] = (int32_t)(((uint32_t)bq_int_from_d(s.y1) << 16) | ((uint32_t)bq_int_from_d(s.y2) & 0xFFFFu));
  b[7 * (size_t)Cpad] = (int32_t)((uint32_t)s.res | flag);
}

template <int NS>
__device__ __forceinline__ uint32_t bq_word(BqStageS (&st)[NS], uint32_t w)
{
  static_assert(NS == 1, "the split stage takes plain values in and hands y << 16 out: single stages only");
  int xe, xo;
  asm("prmt.b32 %0, %1, 0, 0x9910;" : "=r"(xe) : "r"(w));
  asm("prmt.b32 %0, %1, 0, 0xBB32;" : "=r"(xo) : "r"(w));
  xe = bq_step(st[0], xe);
  xo = bq_step(st[0], xo);
  return __byte_perm((uint32_t)xe, (uint32_t)xo, 0x7632);
}
__device__ __forceinline__ void bq_load_stage(BqStageS &s, uint32_t &flag, const int32_t *__restrict__ bq, uint32_t Cpad, int obj, int stage, uint32_t ch)
{
  const int32_t *b = bq + (size_t)((obj * 4 + stage) * 8) * Cpad + ch;
  bq_set_coefs(s, __ldcg(b + 0 * (size_t)Cpad), __ldcg(b + 1 * (size_t)Cpad), __ldcg(b + 2 * (size_t)Cpad), __ldcg(b + 3 * (size_t)Cpad),
               __ldcg(b + 4 * (size_t)Cpad));
  const uint32_t w5 = (uint32_t)__ldcg(b + 5 * (size_t)Cpad), w6 = (uint32_t)__ldcg(b + 6 * (size_t)Cpad);
  s.x1 = (int)w5 >> 16; s.x2 = (int)(short)(w5 & 0xFFFFu);
  s.y1s = (int)(w6 & 0xFFFF0000u); s.y2 = (int)(short)(w6 & 0xFFFFu);
  const uint32_t w7 = (uint32_t)__ldcg(b + 7 * (size_t)Cpad);
  s.res = (int)(w7 & 0x3FFFu);
  flag = w7 & 0x80000000u;
}
__device__ __forceinline__ void bq_store_stage(const BqStageS &s, uint32_t flag, int32_t *__restrict__ bq, uint32_t Cpad, int obj, int stage, uint32_t ch)
{
  int32_t *b = bq + (size_t)((obj * 4 + stage) * 8) * Cpad + ch;
  b[5 * (size_t)Cpad] = (int32_t)(((uint32_t)s.x1 << 16) | ((uint32_t)s.x2 & 0xFFFFu));
  b[6 * (size_t)Cpad] = (int32_t)(((uint32_t)s.y1s & 0xFFFF0000u) | ((uint32_t)s.y2 & 0xFFFFu));
  b[7 * (size_t)Cpad] = (int32_t)((uint32_t)s.res | flag);
}
__device__ __forceinline__ void bq_load_stage(BqStage &s, uint32_t &flag, const int32_t *__restrict__ bq, uint32_t Cpad, int obj, int stage, uint32_t ch)
{
  const int32_t *b = bq + (size_t)((obj * 4 + stage) * 8) * Cpad + ch;
  s.b0 = __ldcg(b + 0 * (size_t)Cpad);
  s.b1 = __ldcg(b + 1 * (size_t)Cpad);
  s.b2 = __ldcg(b + 2 * (size_t)Cpad);
  s.a1 = __ldcg(b + 3 * (size_t)Cpad);
  s.a2 = __ldcg(b + 4 * (size_t)Cpad);
  bq_unpack_hist((uint32_t)__ldcg(b + 5 * (size_t)Cpad), s.x1, s.x2);
  bq_unpack_hist((uint32_t)__ldcg(b + 6 * (size_t)Cpad), s.y1, s.y2);
  const uint32_t w7 = (uint32_t)__ldcg(b + 7 * (size_t)Cpad);
  s.res = (int)(w7 & 0x3FFFu); // filter_biquad.cpp:52
  flag = w7 & 0x80000000u;
}
__device__ __forceinline__ void bq_store_stage(const BqStage &s, uint32_t flag, int32_t *__restrict__ bq, uint32_t Cpad, int obj, int stage, uint32_t ch)
{
  int32_t *b = bq + (size_t)((obj * 4 + stage) * 8) * Cpad + ch;
  b[5 * (size_t)Cpad] = (int32_t)bq_pack_hist(s.x1, s.x2);
  b[6 * (size_t)Cpad] = (int32_t)bq_pack_hist(s.y1, s.y2);
  b[7 * (size_t)Cpad] = (int32_t)((uint32_t)s.res | flag); // filter_biquad.cpp:75-78
}
__device__ __forceinline__ void bq_load_stage(BqStageH &s, uint32_t &flag, const int32_t *__restrict__ bq, uint32_t Cpad, int obj, int stage, uint32_t ch)
{
  const int32_t *b = bq + (size_t)((obj * 4 + stage) * 8) * Cpad + ch;
  bq_set_coefs(s, __ldcg(b + 0 * (size_t)Cpad), __ldcg(b + 1 * (size_t)Cpad), __ldcg(b + 2 * (size_t)Cpad), __ldcg(b + 3 * (size_t)Cpad),
               __ldcg(b + 4 * (size_t)Cpad));
  const uint32_t w5 = (uint32_t)__ldcg(b + 5 * (size_t)Cpad);
  s.x1 = bq_d_from_int((int)w5 >> 16); s.x2 = bq_d_from_int((int)(short)(w5 & 0xFFFFu));
  bq_unpack_hist((uint32_t)__ldcg(b + 6 * (size_t)Cpad), s.y1, s.y2);
  const uint32_t w7 = (uint32_t)__ldcg(b + 7 * (size_t)Cpad);
  s.res = (int)(w7 & 0x3FFFu);
  flag = w7 & 0x80000000u;
}
__device__ __forceinline__ void bq_store_stage(const BqStageH &s, uint32_t flag, int32_t *__restrict__ bq, uint32_t Cpad, int obj, int stage, uint32_t ch)
{
  int32_t *b = bq + (size_t)((obj * 4 + stage) * 8) * Cpad + ch;
  b[5 * (size_t)Cpad] = (int32_t)(((uint32_t)bq_int_from_d(s.x1) << 16) | ((uint32_t)bq_int_from_d(s.x2) & 0xFFFFu));
  b[6 * (size_t)Cpad] = (int32_t)bq_pack_hist(s.y1, s.y2);
  b[7 * (size_t)Cpad] = (int32_t)((uint32_t)s.res | flag);
}


// ---- one stage split in two (chain kernel v4, FF shape) ---------------------------------------------------------------
// filter_biquad.cpp:56-63 per sample:  sum = res + b0 x[n] + b1 x[n-1] + b2 x[n-2] + a1 y[n-1] + a2 y[n-2]  (SMLAW products,
// adds wrap mod 2^32, so the order is free).  The three input-side products depend on the input only: a helper warp forms
//   e[n] = hi(b0 x[n]) + hi(b1 x[n-1]) + hi(b2 x[n-2])
// for a whole sub-tile, and the chain warp is left with the recurrence  sum = e[n] + res + hi(a2 y[n-2]) + hi(a1 y[n-1]).
// The helper warps form e[n] on the FP64 pipe (exact DFMA.RM form of msdr_device.cuh): the integer-multiply pipe of their
// sub-partition stays free for the tensor-core epilogue and the converters that live there.
struct BqFF {
  double b0, b1, b2; // coefficient * 2^-16
  double m0, m1, m2; // 1.5 * 2^52 - 17 * coefficient: the low word of fma_rd(b', D, m) is the SMLAW product itself (msdr_device.cuh)
  double x1, x2;     // D-form input history
};
struct BqRec {
  int a1, a2; // already negated as stored by setCoefficients (filter_biquad.cpp:93-94)
  int y1, y2; // << 16
  int res;
};
// x: the int16 input value, sign-extended
__device__ __forceinline__ int ff_step(BqFF &f, int x)
{
  const double xD = bq_d_from_int(x);
  const int e = __double2loint(__fma_rd(f.b0, xD, f.m0)) + __double2loint(__fma_rd(f.b1, f.x1, f.m1)) +
                __double2loint(__fma_rd(f.b2, f.x2, f.m2));
  f.x2 = f.x1; f.x1 = xD;
  return e;
}
// returns y << 16
__device__ __forceinline__ int rec_step(BqRec &r, int e)
{
  int t, pre;
  asm("mad.hi.s32 %0, %1, %2, %3;" : "=r"(t) : "r"(r.a2), "r"(r.y2), "r"(e));
  asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(pre) : "r"(r.res), "r"(kBqOne), "r"(t)); // keeps res off the IMAD.HI chain (kBqOne)
  const int sum = smlaw_s(pre, r.a1, r.y1);
  int ys;
  asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(ys) : "r"(sum >> 14), "r"(0)); // ssat #16, asr #14, << 16
  r.res = sum & 0x3FFF;
  r.y2 = r.y1; r.y1 = ys;
  return ys;
}
__device__ __forceinline__ void bq_load_ff(BqFF &f, const int32_t *__restrict__ bq, uint32_t Cpad, int obj, uint32_t ch)
{
  const int32_t *b = bq + (size_t)(obj * 4 * 8) * Cpad + ch;
  const int b0 = __ldcg(b + 0 * (size_t)Cpad), b1 = __ldcg(b + 1 * (size_t)Cpad), b2 = __ldcg(b + 2 * (size_t)Cpad);
  const double k = 1.0 / 65536.0;
  f.b0 = (double)b0 * k; f.b1 = (double)b1 * k; f.b2 = (double)b2 * k;
  f.m0 = kBqM - 17.0 * (double)b0; f.m1 = kBqM - 17.0 * (double)b1; f.m2 = kBqM - 17.0 * (double)b2;
  const uint32_t w5 = (uint32_t)__ldcg(b + 5 * (size_t)Cpad); // (x[n-1] << 16) | (x[n-2] & 0xffff), filter_biquad.cpp:66-69
  f.x1 = bq_d_from_int((int)w5 >> 16);
  f.x2 = bq_d_from_int((int)(short)(w5 & 0xFFFFu));
}
__device__ __forceinline__ void bq_store_ff(const BqFF &f, int32_t *__restrict__ bq, uint32_t Cpad, int obj, uint32_t ch)
{
  bq[(size_t)(obj * 4 * 8 + 5) * Cpad + ch] = (int32_t)(((uint32_t)bq_int_from_d(f.x1) << 16) | ((uint32_t)bq_int_from_d(f.x2) & 0xFFFFu));
}
__device__ __forceinline__ void bq_load_rec(BqRec &r, uint32_t &flag, const int32_t *__restrict__ bq, uint32_t Cpad, int obj, uint32_t ch)
{
  const int32_t *b = bq + (size_t)(obj * 4 * 8) * Cpad + ch;
  r.a1 = __ldcg(b + 3 * (size_t)Cpad);
  r.a2 = __ldcg(b + 4 * (size_t)Cpad);
  bq_unpack_hist((uint32_t)__ldcg(b + 6 * (size_t)Cpad), r.y1, r.y2);
  const uint32_t w7 = (uint32_t)__ldcg(b + 7 * (size_t)Cpad);
  r.res = (int)(w7 & 0x3FFFu);
  flag = w7 & 0x80000000u;
}
__device__ __forceinline__ void bq_store_rec(const BqRec &r, uint32_t flag, int32_t *__restrict__ bq, uint32_t Cpad, int obj, uint32_t ch)
{
  int32_t *b = bq + (size_t)(obj * 4 * 8) * Cpad + ch;
  b[6 * (size_t)Cpad] = (int32_t)bq_pack_hist(r.y1, r.y2);
  b[7 * (size_t)Cpad] = (int32_t)((uint32_t)r.res | flag);
}

} // namespace msdr
