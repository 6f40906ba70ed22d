// msdr_chain_v5_common.cuh — helpers of the row-block kernel (msdr_chain_v5.cu, whole- and half-tile forms): epilogue drain and
// demodulation on registers, the biquad tile loop, the developer profile, the front end of the ADC-code input.
#pragma once
#include "msdr_chain_common.cuh"
#include "msdr_frontend.cuh"
#include "msdr_tc_common.cuh"

namespace msdr {
namespace v5 {

using namespace tc;

constexpr uint32_t kPad = 0xFFFFFFFFu;

// chain channel of launch row `row` (never kPad): its entry of the channel list, or ch0 + row for a range; hist_ch as the 64-bit index
// of the history row (the range form keeps the index arithmetic the kernels had before lists)
template <bool kList>
__device__ __forceinline__ uint32_t chan_of(const ChainParams &p, uint32_t row)
{
  if constexpr (kList) return __ldg(p.chlist + row);
  else return p.ch0 + row;
}
template <bool kList>
__device__ __forceinline__ size_t hist_ch(const ChainParams &p, uint32_t row)
{
  if constexpr (kList) return __ldg(p.chlist + row);
  else return (size_t)p.ch0 + row;
}
// sleep between mbarrier probes per role (nanoseconds; msdr_device.cuh::mbar_wait).  The tensor-memory hand-off between the MMA warp
// and the epilogue is the kernel's tightest loop and probes often; everything that sits behind a ring of slots can afford to find
// out late that its barrier has flipped, and its probes otherwise delay the dependent instruction chains of the biquad warps.
#ifndef MSDR_V5_NS
#define MSDR_V5_NS 1
#endif
constexpr uint32_t kNsLoad = 256 * MSDR_V5_NS, kNsConv = 128 * MSDR_V5_NS, kNsSlot = 128 * MSDR_V5_NS, kNsBq = 128 * MSDR_V5_NS, kNsStore = 256 * MSDR_V5_NS;

// developer profile (MSDR_PROF=1): per-CTA cycle totals, slot = role * 4 + counter
struct Prof {
  long long *base;
  long long acc[4];
  long long t;
  __device__ __forceinline__ Prof(long long *b, int role) : base(b ? b + (size_t)blockIdx.x * 64 + role * 4 : nullptr), acc{0, 0, 0, 0}, t(0) {}
  __device__ __forceinline__ void start() { if (base) t = clock64(); }
  __device__ __forceinline__ void lap(int i) { if (base) { const long long n = clock64(); acc[i] += n - t; t = n; } }
  __device__ __forceinline__ void flush() { if (base && (threadIdx.x & 31) == 0) for (int i = 0; i < 4; ++i) base[i] = acc[i]; }
};

__device__ __forceinline__ uint4 lds128(uint32_t a)
{
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t a, const uint4 &v)
{
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// NQ * 8 samples of one row in place (NQ even): 128-bit words, two register sets alternating (the next eight samples are on their
// way while the recurrence runs)
template <class BQ, int NQ = N / 8>
__device__ __forceinline__ void bq_tile(BQ (&st)[1], uint32_t a)
{
  uint4 v0 = lds128(a), v1;
#pragma unroll 1
  for (int q = 0; q < NQ; q += 2) {
    v1 = lds128(a + 16u * (uint32_t)(q + 1));
    v0.x = bq_word<1>(st, v0.x);
    v0.y = bq_word<1>(st, v0.y);
    v0.z = bq_word<1>(st, v0.z);
    v0.w = bq_word<1>(st, v0.w);
    sts128(a + 16u * (uint32_t)q, v0);
    if (q + 2 < NQ) v0 = lds128(a + 16u * (uint32_t)(q + 2));
    v1.x = bq_word<1>(st, v1.x);
    v1.y = bq_word<1>(st, v1.y);
    v1.z = bq_word<1>(st, v1.z);
    v1.w = bq_word<1>(st, v1.w);
    sts128(a + 16u * (uint32_t)(q + 1), v1);
  }
}

// one branch of eight output columns: the three byte-plane accumulators -> the reference's accumulator mod 2^32
__device__ __forceinline__ void drain8(uint32_t taddr, uint32_t (&acc)[8])
{
  uint32_t a0[8], a1[8], a2[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(a0[0]), "=r"(a0[1]), "=r"(a0[2]), "=r"(a0[3]), "=r"(a0[4]), "=r"(a0[5]), "=r"(a0[6]), "=r"(a0[7]) : "r"(taddr));
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(a1[0]), "=r"(a1[1]), "=r"(a1[2]), "=r"(a1[3]), "=r"(a1[4]), "=r"(a1[5]), "=r"(a1[6]), "=r"(a1[7]) : "r"(taddr + (uint32_t)N));
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(a2[0]), "=r"(a2[1]), "=r"(a2[2]), "=r"(a2[3]), "=r"(a2[4]), "=r"(a2[5]), "=r"(a2[6]), "=r"(a2[7]) : "r"(taddr + 2u * (uint32_t)N));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = (a0[j] << 16) + (a1[j] << 8) + a2[j]; // mod 2^32, like the reference accumulator
}

// demodulation switch (Minimal-SDR.ino:589-628) over the 32 packed (I | Q << 16) words a thread holds -> 16 words of int16 pairs
// SSB kinds straight on the packed words p = I | Q << 16 (Minimal-SDR.ino:591-604: the int16 sum wraps, no saturation):
//   USB  I + Q = upper half of p * 65537;   LSB  I - Q = I + ~Q + 1 = upper half of (p ^ 0xFFFF0000) * 65537 + 0x10000
// one LOP3 and one IMAD per sample, one PRMT per pair.  xm / xc: the per-row XOR mask and addend (0 / 0 for USB).
__device__ __forceinline__ void demod_ssb_regs(const uint32_t (&iq)[32], uint32_t xm, uint32_t xc, uint32_t (&out)[16])
{
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const uint32_t t0 = (iq[2 * j] ^ xm) * 65537u + xc, t1 = (iq[2 * j + 1] ^ xm) * 65537u + xc;
    out[j] = __byte_perm(t0, t1, 0x7632);
  }
}

template <int KIND>
__device__ __forceinline__ void demod_regs(const uint32_t (&iq)[32], int sgn, uint32_t (&out)[16])
{
#pragma unroll
  for (int c0 = 0; c0 < 32; c0 += 8) { // eight samples in flight: the envelope kinds are a dependent-latency problem
    int y[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) y[j] = demod_inline<KIND>((int)(short)(iq[c0 + j] & 0xFFFFu), (int)iq[c0 + j] >> 16, sgn);
#pragma unroll
    for (int j = 0; j < 4; ++j) out[c0 / 2 + j] = ((uint32_t)y[2 * j] & 0xFFFFu) | ((uint32_t)y[2 * j + 1] << 16);
  }
}

// ADC-code input (p.fe != NULL): the converter thread of a row owns the row's front end (msdr_frontend.cuh) for the whole row block and
// runs it over the staged codes in time order, ahead of the fs/4 fold.  Per row: the recurrence and gain state in registers, the AGC's
// 25-entry history in the chain's state array in global memory (the long window leaves no shared memory for it), touched once per
// 128-sample block through an exact running sum of its entries; the slot a block overwrites is read when the block starts.
struct FeRow {
  fe::State *s;    // this row's state; NULL for a padded row
  int x1, y1, mult, idx, sum, old;
  float val;
  uint32_t maxv, minv;
};

__device__ __forceinline__ void fe_row_begin(FeRow &f, const ChainParams &p, uint32_t row)
{
  f.s = nullptr;
  if (row == kPad) return;
  const size_t ch = (size_t)p.ch0 + row;
  fe::State *s = p.fe + ch;
  f.s = s;
  f.x1 = s->hpf_x1; f.y1 = s->hpf_y1; f.mult = s->mult; f.idx = s->agc_idx; f.val = s->agc_val;
  f.sum = 0;
#pragma unroll 5
  for (int k = 0; k < fe::kAgcBuf; ++k) f.sum += s->agc_buf[k];
  f.old = 0;
  f.maxv = fe::kMaxInit; f.minv = fe::kMinInit;
}

// The history rows hold conditioned IF samples in both input formats; here the converter writes them as it produces them.  For an
// update shorter than the history (L < H) part of the old history survives and moves down first, in increasing order.  Call this only
// once the converter has consumed the row block's history stages (j < 0): from then on the loader reads no history of this row, so
// neither the move nor the new samples can race its copies.
__device__ __forceinline__ uint4 *fe_row_hist(const FeRow &f, const ChainParams &p)
{
  return reinterpret_cast<uint4 *>(p.hist + (size_t)(f.s - p.fe) * p.H);
}
__device__ __forceinline__ void fe_row_shift_hist(const FeRow &f, const ChainParams &p)
{
  if (!f.s || p.L >= p.H) return;
  uint4 *hrow = fe_row_hist(f, p);
  const uint32_t lq = p.L >> 3, keep = (p.H >> 3) - lq;
  for (uint32_t i = 0; i < keep; ++i) hrow[i] = __ldcg(hrow + i + lq);
}

// The 8 NQ staged codes of this thread's row at shared address `a`, samples t0 .. t0 + 8 NQ - 1 of the update (8 NQ divides 128), are
// conditioned in place, one 16-byte word at a time: the fs/4 fold then reads IF samples as in the int16 form, and the conversion's
// operands and the front end's state are never live together (the 736-thread CTA leaves 80 registers a thread).
template <int NQ>
__device__ __forceinline__ void fe_row_run(FeRow &f, const ChainParams &p, uint32_t a, uint32_t t0)
{
  if (!f.s) return;
  if ((t0 & (fe::kBlock - 1)) == 0 && p.agc_on) f.old = f.idx > 0 ? f.s->agc_buf[f.idx - 1] : 0; // the slot this block's maximum takes
  // the last H samples of hist || in become the history (sample t lands at t + H - L; L and H are multiples of 8)
  uint4 *hrow = fe_row_hist(f, p) + (((int)t0 + (int)p.H - (int)p.L) >> 3);
#pragma unroll 2
  for (int q = 0; q < NQ; ++q) {
    uint4 v = lds128(a + 16u * q);
    v.x = fe::condition2(v.x, f.x1, f.y1, f.mult, f.maxv, f.minv);
    v.y = fe::condition2(v.y, f.x1, f.y1, f.mult, f.maxv, f.minv);
    v.z = fe::condition2(v.z, f.x1, f.y1, f.mult, f.maxv, f.minv);
    v.w = fe::condition2(v.w, f.x1, f.y1, f.mult, f.maxv, f.minv);
    sts128(a + 16u * q, v);
    if ((int)(t0 + 8u * q) + (int)p.H >= (int)p.L) hrow[q] = v;
  }
  if (((t0 + 8u * NQ) & (fe::kBlock - 1)) == 0) { // an audio block is complete
    if (p.agc_on) {
      const int16_t m = (int16_t)fe::block_absmax(f.maxv, f.minv);
      const int i = fe::agc_slot(f.idx);
      if (i >= 0) { f.sum += (int)m - f.old; f.s->agc_buf[i] = m; }
      fe::agc_law(f.val, f.mult, f.sum, p.agc_max);
    }
    f.maxv = fe::kMaxInit; f.minv = fe::kMinInit;
  }
}

__device__ __forceinline__ void fe_row_end(const FeRow &f)
{
  if (!f.s) return;
  f.s->hpf_x1 = f.x1; f.s->hpf_y1 = f.y1; f.s->mult = f.mult; f.s->agc_idx = f.idx; f.s->agc_val = f.val;
}

} // namespace v5
} // namespace msdr
