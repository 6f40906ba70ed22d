// msdr_frontend.cuh — the front-end arithmetic (SURVEY 8f rank 1), shared by K4 (msdr_frontend.cu) and the ADC-code instantiations of
// the row-block chain kernel (msdr_chain_v5.cu, both forms):
//   raw unsigned ADC codes -> 1-pole DC-blocking high-pass in S1.30 (AudioInputAnalog::update, input_adc.cpp:198-212)
//   -> AudioAmplifier gain with SSAT16 (mixer.cpp:34-47,134-159, mixer.h:75-79) -> int16 IF samples,
//   and per 128-sample block the AGC of the sketch (Minimal-SDR.ino:445-515): block maximum of |x| through the halfword SIMD
//   idiom, 25-block history, float gain law, new amplifier multiplier for the blocks that follow.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace msdr {
namespace fe {

constexpr int kBlock = 128;                    // AUDIO_BLOCK_SAMPLES
constexpr int kAgcBuf = 25;                    // .ino:445
constexpr int kCoefHpf = 1048300 << 10;        // input_adc.cpp:32, S1.30

struct State { // one channel
  int32_t hpf_x1, hpf_y1; // input_adc.cpp:37-38
  int32_t mult;           // AudioAmplifier::multiplier
  int32_t agc_idx;        // .ino:451
  float agc_val;          // AGC_val
  int16_t agc_buf[kAgcBuf];
  int16_t pad;
};
static_assert(sizeof(State) == 72, "State layout is mirrored by msdr_frontend_state");

__host__ __device__ inline int32_t amp_multiplier(float n) // AudioAmplifier::gain, mixer.h:75-79
{
  if (n > 32767.0f) n = 32767.0f;
  else if (n < -32767.0f) n = -32767.0f;
#ifdef __CUDA_ARCH__
  return __float2int_rz(__fmul_rn(n, 65536.0f));
#else
  return (int32_t)(n * 65536.0f);
#endif
}

// a channel before its first block: high-pass at rest, empty AGC history, gain agc_start
inline State initial_state(float agc_start)
{
  State s{};
  s.agc_idx = kAgcBuf;                // .ino:451
  s.agc_val = agc_start;              // .ino:104
  s.mult = amp_multiplier(agc_start); // .ino:385
  return s;
}

// ARMv7E-M SSUB16 (sets APSR.GE[1:0] / [3:2] when the low / high halfword difference is >= 0) and SEL (bytes of `a` where GE is set)
__device__ __forceinline__ uint32_t ssub16(int a, int b, uint32_t &ge)
{
  const int lo = (int)(short)(a & 0xFFFF) - (int)(short)(b & 0xFFFF), hi = (a >> 16) - (b >> 16);
  ge = (lo >= 0 ? 3u : 0u) | (hi >= 0 ? 12u : 0u);
  return ((uint32_t)hi << 16) | ((uint32_t)lo & 0xFFFFu);
}
__device__ __forceinline__ uint32_t sel(uint32_t a, uint32_t b, uint32_t ge)
{
  const uint32_t m = ((ge & 1u) ? 0x000000FFu : 0u) | ((ge & 2u) ? 0x0000FF00u : 0u) | ((ge & 4u) ? 0x00FF0000u : 0u) | ((ge & 8u) ? 0xFF000000u : 0u);
  return (a & m) | (b & ~m);
}

// running per-halfword maximum / minimum of a block start here (.ino:457-458, as packed halfword pairs)
constexpr uint32_t kMaxInit = (uint32_t)(-32767), kMinInit = 32767u;

// Two codes of a word (low half = earlier sample) through the high-pass, the gain and SSAT16, in time order; the packed result also
// enters the block's running maximum / minimum.  x1, y1: the recurrence state; mult: AudioAmplifier::multiplier.
__device__ __forceinline__ uint32_t condition2(uint32_t w, int &x1, int &y1, int mult, uint32_t &maxv, uint32_t &minv)
{
  int o[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    // the ALU pipe (shifts, min/max, logic) is K4's busiest unit: the code word is widened on the multiplier,
    // both clamps are cvt.pack.sat (one I2IP each instead of a min/max pair), the gain product is one IMAD.HI
    const uint32_t code = k ? __byte_perm(w, 0u, 0x4432) : __byte_perm(w, 0u, 0x4410);
    const int tmp = (int)(code * 16384u);
    const int acc = (int)((uint32_t)y1 - (uint32_t)x1 + (uint32_t)tmp);
    // FRACMUL_SHL(acc, COEF, 1): bits [61:30] of the product.  4 * COEF = 2^32 - 69 * 2^14, so
    //   (acc * COEF) >> 30 = (acc * 4 COEF) >> 32 = acc + floor(-69 * 2^14 * acc / 2^32) = acc + mulhi(acc, -69 << 14)
    // exactly: one IMAD.HI and an add (13 cycles of dependent latency) instead of IMAD.WIDE and a 64-bit funnel shift (20) on the
    // per-sample recurrence.
    static_assert(4ll * kCoefHpf == (1ll << 32) - (69ll << 14), "the identity above is derived from this coefficient");
    y1 = acc + __mulhi(acc, -(69 << 14));
    x1 = tmp;
    int ss; // SSAT16(y1 >> 14) in the upper half (signed_saturate_rshift, input_adc.cpp:209)
    asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(ss) : "r"(y1 >> 14), "r"(0));
    // AudioAmplifier::update special-cases multiplier 0 (nothing transmitted -> zeros here) and 65536 (pass-through,
    // mixer.cpp:139-151); SSAT16((mult * s) >> 16) gives exactly those values for them, so no branch per sample.
    // hi32(mult * (s << 16)) == (mult * s) >> 16
    o[k] = __mulhi(mult, ss);
  }
  uint32_t r;
  asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(r) : "r"(o[1]), "r"(o[0])); // both SSAT16 and the packing
  maxv = __vmaxs2(maxv, r); // SSUB16 + SEL: per-halfword signed maximum / minimum
  minv = __vmins2(minv, r);
  return r;
}

// .ino:468-478, literally: the cross-halfword compares, abs() of the whole words, the final select -> the block's maximum of |x|
__device__ __forceinline__ uint32_t block_absmax(uint32_t maxv, uint32_t minv)
{
  int mx = (int)maxv, mn = (int)minv;
  uint32_t ge;
  (void)ssub16(mx, mx >> 16, ge); mx = (int)sel((uint32_t)mx, (uint32_t)(mx >> 16), ge); // max of the two halfwords -> low half
  (void)ssub16(mn >> 16, mn, ge); mn = (int)sel((uint32_t)mn, (uint32_t)(mn >> 16), ge); // min -> low half
  mn = (int)(mn < 0 ? 0u - (uint32_t)mn : (uint32_t)mn);                                   // abs() of the WHOLE words
  mx = (int)(mx < 0 ? 0u - (uint32_t)mx : (uint32_t)mx);
  (void)ssub16(mx, mn, ge);
  return sel((uint32_t)mx, (uint32_t)mn, ge) & 0xFFFFu;
}

// .ino:487-514: the gain law on m, the sum of the 25 stored block maxima; a change sets the amplifier multiplier
__device__ __forceinline__ void agc_law(float &agc_val, int32_t &mult, int m, float agc_max)
{
  const int d = m / kAgcBuf;
  const float f = __fdiv_rn(16000.0f, __int2float_rn(d));
  const float val = agc_val;
  const float vf = __fmul_rn(val, f);
  bool changed = false;
  if ((double)f > 1.3) {
    const float fagc = __fadd_rn(val, __fdiv_rn(vf, 1500.0f));
    if (fagc < agc_max) { agc_val = fagc; changed = true; }
  } else if ((double)val > 0.1) {
    if ((double)f < 0.6) { agc_val = __fsub_rn(val, __fdiv_rn(vf, 50.0f)); changed = true; }
    else if ((double)f < 0.7) { agc_val = __fsub_rn(val, __fdiv_rn(vf, 200.0f)); changed = true; }
    else if ((double)f < 0.8) { agc_val = __fsub_rn(val, __fdiv_rn(vf, 2000.0f)); changed = true; }
    else if ((double)f < 0.9) { agc_val = __fsub_rn(val, __fdiv_rn(vf, 4000.0f)); changed = true; }
  }
  if (changed) mult = amp_multiplier(agc_val);
}

// .ino:481-482 with the 26th-store defect resolved as in the oracle (value dropped): the history slot this block's maximum goes to,
// or -1 when it is dropped; agc_idx advances either way
__device__ __forceinline__ int agc_slot(int32_t &agc_idx)
{
  const int i = --agc_idx;
  if (i < 0) agc_idx = kAgcBuf;
  return i;
}

// the whole AGC step on a state held in one place (K4: registers / local memory)
__device__ __forceinline__ void agc_update(State &s, uint32_t absmax, float agc_max)
{
  const int i = agc_slot(s.agc_idx);
  if (i >= 0) s.agc_buf[i] = (int16_t)absmax;
  int m = 0;
#pragma unroll
  for (int k = 0; k < kAgcBuf; ++k) m += s.agc_buf[k];
  agc_law(s.agc_val, s.mult, m, agc_max);
}

} // namespace fe
} // namespace msdr
