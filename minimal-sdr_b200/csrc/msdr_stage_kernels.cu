// msdr_stage_kernels.cu — one kernel per reference primitive, on device buffers.
// These back the stage-level C-ABI operators (msdr_op_*) used by the AudioStream façade and the per-stage
// parity tests; the production path is the fused chain kernels in msdr_chain_v4.cu, v5.cu, v5l.cu and v6.cu.
#include "msdr_device.cuh"
#include "msdr_internal.h"
#include <algorithm>

namespace msdr {

// ---- fs/4 mix (Minimal-SDR.ino:546-558): one thread per 4 samples --------------------------------
__global__ void mix_fs4_kernel(const int16_t *__restrict__ in, int16_t *__restrict__ I, int16_t *__restrict__ Q, uint32_t rows, uint32_t n4,
                               size_t stride)
{
  const size_t total = (size_t)rows * n4;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t r = idx / n4, q = idx - r * n4;
    const size_t off = r * stride + q * 4;
    const uint2 v = *reinterpret_cast<const uint2 *>(in + off); // x0,x1 | x2,x3
    const uint32_t nv = neg16x2(v.y);
    // I = {x0, 0, -x2, 0}   Q = {0, x1, 0, -x3}
    *reinterpret_cast<uint2 *>(I + off) = make_uint2(v.x & 0xFFFFu, nv & 0xFFFFu);
    *reinterpret_cast<uint2 *>(Q + off) = make_uint2(v.x & 0xFFFF0000u, nv & 0xFFFF0000u);
  }
}

cudaError_t launch_mix_fs4(const int16_t *in, int16_t *I, int16_t *Q, uint32_t rows, uint32_t n, size_t stride, cudaStream_t s)
{
  const size_t total = (size_t)rows * (n / 4);
  if (total == 0) return cudaSuccess;
  const int block = 256;
  const int grid = (int)std::min<size_t>((total + block - 1) / block, 148 * 16);
  mix_fs4_kernel<<<grid, block, 0, s>>>(in, I, Q, rows, n / 4, stride);
  return cudaGetLastError();
}

// ---- arm_fir_fast_q15 (arm_fir_fast_q15.c:60-329), dense taps, any even T ----------------------------
// CTA = (row, 1024-sample span); the span plus its (T-1)-sample history is staged in shared memory together with
// the taps; each thread computes 4 consecutive outputs from a sliding register window.
constexpr int kFirSpan = 1024;

__global__ void __launch_bounds__(256) fir_fast_q15_kernel(uint32_t T, const int16_t *__restrict__ coef, const int16_t *__restrict__ hist_in,
                                                           const int16_t *__restrict__ in, int16_t *__restrict__ out, uint32_t n, size_t stride)
{
  extern __shared__ int32_t sm[];
  int32_t *s_c = sm;     // T taps, widened
  int32_t *s_x = sm + T; // (T-1) + span samples, widened
  const uint32_t row = blockIdx.y;
  const uint32_t t0 = blockIdx.x * kFirSpan;
  const uint32_t len = min((uint32_t)kFirSpan, n - t0);
  const uint32_t Hn = T - 1;
  for (uint32_t i = threadIdx.x; i < T; i += blockDim.x) s_c[i] = coef[i];
  for (uint32_t i = threadIdx.x; i < Hn + len; i += blockDim.x) {
    const long long g = (long long)t0 + i - Hn; // stream index
    int v;
    if (g >= 0) v = in[row * stride + (size_t)g];
    else v = hist_in ? hist_in[(size_t)row * Hn + (size_t)(g + Hn)] : 0;
    s_x[i] = v;
  }
  __syncthreads();
  const uint32_t o0 = threadIdx.x * 4;
  if (o0 >= len) return;
  uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  uint32_t w0 = (uint32_t)s_x[o0], w1 = (uint32_t)s_x[o0 + 1], w2 = (uint32_t)s_x[o0 + 2];
  for (uint32_t k = 0; k < T; ++k) {
    const uint32_t c = (uint32_t)s_c[k];
    const uint32_t w3 = (uint32_t)s_x[o0 + k + 3 < Hn + len ? o0 + k + 3 : Hn + len - 1];
    a0 += c * w0; a1 += c * w1; a2 += c * w2; a3 += c * w3;
    w0 = w1; w1 = w2; w2 = w3;
  }
  int16_t *o = out + row * stride + t0 + o0;
  const int y0 = ssat16((int)a0 >> 15), y1 = ssat16((int)a1 >> 15), y2 = ssat16((int)a2 >> 15), y3 = ssat16((int)a3 >> 15);
  if (o0 + 3 < len) {
    o[0] = (int16_t)y0; o[1] = (int16_t)y1; o[2] = (int16_t)y2; o[3] = (int16_t)y3;
  } else {
    o[0] = (int16_t)y0;
    if (o0 + 1 < len) o[1] = (int16_t)y1;
    if (o0 + 2 < len) o[2] = (int16_t)y2;
  }
}

// new history = last T-1 samples of (old history || in[0..n))
__global__ void fir_hist_kernel(uint32_t T, const int16_t *__restrict__ hist_in, int16_t *__restrict__ hist_out, const int16_t *__restrict__ in,
                                uint32_t rows, uint32_t n, size_t stride)
{
  const uint32_t Hn = T - 1;
  const size_t total = (size_t)rows * Hn;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t r = idx / Hn;
    const uint32_t i = (uint32_t)(idx - r * Hn);
    const long long g = (long long)n - Hn + i;
    hist_out[idx] = g >= 0 ? in[r * stride + (size_t)g] : (hist_in ? hist_in[r * Hn + (size_t)(g + Hn)] : (int16_t)0);
  }
}

cudaError_t launch_fir_fast_q15(uint32_t T, const int16_t *coef, const int16_t *hist_in, int16_t *hist_out, const int16_t *in, int16_t *out,
                                uint32_t rows, uint32_t n, size_t stride, cudaStream_t s)
{
  if (rows == 0 || n == 0) return cudaSuccess;
  const size_t smem = (size_t)(2 * T + kFirSpan + 8) * sizeof(int32_t);
  if (smem > 48 * 1024) {
    cudaError_t ea = cudaFuncSetAttribute(fir_fast_q15_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ea != cudaSuccess) return ea;
  }
  cudaError_t e = cudaSuccess;
  for (uint32_t r0 = 0; r0 < rows && e == cudaSuccess; r0 += 32768) { // gridDim.y limit
    const uint32_t nr = min(rows - r0, 32768u);
    dim3 grid((n + kFirSpan - 1) / kFirSpan, nr);
    fir_fast_q15_kernel<<<grid, 256, smem, s>>>(T, coef, hist_in ? hist_in + (size_t)r0 * (T - 1) : nullptr, in + (size_t)r0 * stride,
                                               out + (size_t)r0 * stride, n, stride);
    e = cudaGetLastError();
  }
  if (e != cudaSuccess || !hist_out) return e;
  const size_t total = (size_t)rows * (T - 1);
  const int g2 = (int)std::min<size_t>((total + 255) / 256, 148 * 8);
  fir_hist_kernel<<<g2, 256, 0, s>>>(T, hist_in, hist_out, in, rows, n, stride);
  return cudaGetLastError();
}

// ---- demodulation switch (Minimal-SDR.ino:589-628) -----------------------------------------------------
__global__ void demod_kernel(int kind, const int16_t *__restrict__ I, const int16_t *__restrict__ Q, int16_t *__restrict__ out, uint32_t rows,
                             uint32_t n, size_t stride)
{
  const size_t total = (size_t)rows * n;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t r = idx / n, i = idx - r * n;
    const size_t off = r * stride + i;
    out[off] = (int16_t)demod_sample(kind, I[off], Q[off]);
  }
}
cudaError_t launch_demod(int kind, const int16_t *I, const int16_t *Q, int16_t *out, uint32_t rows, uint32_t n, size_t stride, cudaStream_t s)
{
  const size_t total = (size_t)rows * n;
  if (total == 0) return cudaSuccess;
  const int grid = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
  demod_kernel<<<grid, 256, 0, s>>>(kind, I, Q, out, rows, n, stride);
  return cudaGetLastError();
}

// ---- AudioOutputAnalog ISR (output_dac.cpp:140-144): int16 audio -> 12-bit DAC codes, ((s) + 32768) >> 4 ---------------------------
__global__ void dac_codes_kernel(const int16_t *__restrict__ in, uint16_t *__restrict__ out, uint32_t rows, uint32_t n, size_t stride)
{
  const size_t total = (size_t)rows * n;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t r = i / n, off = r * stride + (i - r * n);
    out[off] = (uint16_t)(((int)in[off] + 32768) >> 4);
  }
}
cudaError_t launch_dac_codes(const int16_t *in, uint16_t *out, uint32_t rows, uint32_t n, size_t stride, cudaStream_t s)
{
  const size_t total = (size_t)rows * n;
  if (total == 0) return cudaSuccess;
  dac_codes_kernel<<<(int)std::min<size_t>((total + 255) / 256, 148 * 16), 256, 0, s>>>(in, out, rows, n, stride);
  return cudaGetLastError();
}

// ---- AudioAmplifier::update / applyGain (mixer.cpp:34-47,134-159): SSAT16((mult * x) >> 16), one multiplier per row --------
// (multiplier 65536 passes data through and 0 yields zeros: exactly what the formula gives; the reference transmits no block
// at all for 0, which a caller handles by not forwarding the block)
__global__ void amplifier_kernel(const int32_t *__restrict__ mult, int16_t *__restrict__ data, uint32_t rows, uint32_t n, size_t stride)
{
  const size_t total = (size_t)rows * n;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t r = i / n, off = r * stride + (i - r * n);
    data[off] = (int16_t)ssat16((int)(((long long)mult[r] * (long long)data[off]) >> 16));
  }
}
cudaError_t launch_amplifier(const int32_t *mult, int16_t *data, uint32_t rows, uint32_t n, size_t stride, cudaStream_t s)
{
  const size_t total = (size_t)rows * n;
  if (total == 0) return cudaSuccess;
  const int grid = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
  amplifier_kernel<<<grid, 256, 0, s>>>(mult, data, rows, n, stride);
  return cudaGetLastError();
}

// ---- AudioFilterBiquad::update (filter_biquad.cpp:33-82): one thread per stream, stage-major -----------
__global__ void biquad_kernel(int32_t *__restrict__ definition, int16_t *__restrict__ data, uint32_t rows, uint32_t n, size_t stride)
{
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  int32_t *def = definition + (size_t)r * 32;
  uint32_t *d = reinterpret_cast<uint32_t *>(data + (size_t)r * stride);
  // the reference runs every stage over one 128-sample block before the next block arrives; running each stage
  // over the whole stream is the same computation (a stage only reads the previous stage's output)
  uint32_t flag;
  int k = 0;
  do {
    BqStage st[1];
    st[0].b0 = def[0]; st[0].b1 = def[1]; st[0].b2 = def[2]; st[0].a1 = def[3]; st[0].a2 = def[4];
    bq_unpack_hist((uint32_t)def[5], st[0].x1, st[0].x2);
    bq_unpack_hist((uint32_t)def[6], st[0].y1, st[0].y2);
    st[0].res = def[7] & 0x3FFF;
    flag = (uint32_t)def[7] & 0x80000000u;
    for (uint32_t i = 0; i < n / 2; ++i) {
      const uint32_t w = d[i];
      int xe = (int)(w << 16), xo = (int)(w & 0xFFFF0000u);
      xe = bq_step(st[0], xe);
      xo = bq_step(st[0], xo);
      d[i] = __byte_perm((uint32_t)xe, (uint32_t)xo, 0x7632);
    }
    def[5] = (int32_t)bq_pack_hist(st[0].x1, st[0].x2);
    def[6] = (int32_t)bq_pack_hist(st[0].y1, st[0].y2);
    def[7] = (int32_t)((uint32_t)st[0].res | flag);
    def += 8;
    ++k;
  } while (flag && k < 4);
}
cudaError_t launch_biquad(int32_t *definition, int16_t *data, uint32_t rows, uint32_t n, size_t stride, cudaStream_t s)
{
  if (rows == 0 || n == 0) return cudaSuccess;
  biquad_kernel<<<(rows + 63) / 64, 64, 0, s>>>(definition, data, rows, n, stride);
  return cudaGetLastError();
}

// ---- AudioEffectFreqConv::update (freq_conv.cpp:30-116) -------------------------------------------------
__device__ __forceinline__ int mult_q15(int a, int b) { return ssat16((a * b) >> 15); } // arm_mult_q15
__global__ void freq_conv_kernel(int dir, int16_t *__restrict__ I, int16_t *__restrict__ Q, const int16_t *__restrict__ oscI,
                                 const int16_t *__restrict__ oscQ, uint32_t rows, uint32_t n, size_t stride)
{
  const size_t total = (size_t)rows * n;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t r = idx / n, i = idx - r * n;
    const size_t off = r * stride + i;
    const int vi = I[off], vq = Q[off], oi = oscI[i], oq = oscQ[i];
    if (!dir) { // I' = I*oscQ + Q*oscI ; Q' = Q*oscQ - I*oscI   (freq_conv.cpp:67-84)
      I[off] = (int16_t)ssat16(mult_q15(vi, oq) + mult_q15(vq, oi));
      Q[off] = (int16_t)ssat16(mult_q15(vq, oq) - mult_q15(vi, oi));
    } else {    // Q' = Q*oscQ + I*oscI ; I' = I*oscQ - Q*oscI   (freq_conv.cpp:86-104)
      Q[off] = (int16_t)ssat16(mult_q15(vq, oq) + mult_q15(vi, oi));
      I[off] = (int16_t)ssat16(mult_q15(vi, oq) - mult_q15(vq, oi));
    }
  }
}
cudaError_t launch_freq_conv(int dir, int16_t *I, int16_t *Q, const int16_t *oscI, const int16_t *oscQ, uint32_t rows, uint32_t n, size_t stride,
                             cudaStream_t s)
{
  const size_t total = (size_t)rows * n;
  if (total == 0) return cudaSuccess;
  const int grid = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
  freq_conv_kernel<<<grid, 256, 0, s>>>(dir, I, Q, oscI, oscQ, rows, n, stride);
  return cudaGetLastError();
}

// ---- arm_sqrt_q31 (arm_sqrt_q31.c:50-138) ---------------------------------------------------------------
__global__ void sqrt_q31_kernel(const int32_t *__restrict__ in, int32_t *__restrict__ out, int32_t *__restrict__ status, uint32_t n)
{
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int st;
    out[i] = sqrt_q31(in[i], &st);
    if (status) status[i] = st;
  }
}
cudaError_t launch_sqrt_q31(const int32_t *in, int32_t *out, int32_t *status, uint32_t n, cudaStream_t s)
{
  if (n == 0) return cudaSuccess;
  sqrt_q31_kernel<<<min((n + 255u) / 256u, 148u * 8u), 256, 0, s>>>(in, out, status, n);
  return cudaGetLastError();
}

// ---- AudioFilterBiquad::setCoefficients (filter_biquad.cpp:84-100) on the chain's SoA state -------------
__global__ void bq_setcoef_kernel(int32_t *__restrict__ bq, uint32_t Cpad, int object, uint32_t ch0, uint32_t nch, uint32_t stage, int c0, int c1, int c2,
                                  int c3, int c4)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nch) return;
  const uint32_t ch = ch0 + i;
  int32_t *b = bq + (size_t)((object * 4 + (int)stage) * 8) * Cpad + ch;
  if (stage > 0) {
    int32_t *prev7 = bq + (size_t)((object * 4 + (int)stage - 1) * 8 + 7) * Cpad + ch;
    *prev7 = (int32_t)((uint32_t)*prev7 | 0x80000000u);
  }
  b[0 * (size_t)Cpad] = c0;
  b[1 * (size_t)Cpad] = c1;
  b[2 * (size_t)Cpad] = c2;
  b[3 * (size_t)Cpad] = (int32_t)(0u - (uint32_t)c3);
  b[4 * (size_t)Cpad] = (int32_t)(0u - (uint32_t)c4);
  b[7 * (size_t)Cpad] = (int32_t)((uint32_t)b[7 * (size_t)Cpad] & 0x80000000u);
}
cudaError_t launch_bq_setcoef(int32_t *bq, uint32_t Cpad, int object, uint32_t ch0, uint32_t nch, uint32_t stage, const int32_t coef[5], cudaStream_t s)
{
  if (nch == 0) return cudaSuccess;
  bq_setcoef_kernel<<<(nch + 255) / 256, 256, 0, s>>>(bq, Cpad, object, ch0, nch, stage, coef[0], coef[1], coef[2], coef[3], coef[4]);
  return cudaGetLastError();
}


// exhaustive check of sqrt_rn_fast against __fsqrt_rn over the envelope's argument domain s in [0, 2^31)
__global__ void sqrt_check_kernel(unsigned long long *mismatch)
{
  unsigned long long bad = 0;
  for (unsigned long long s = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; s < 0x80000000ull; s += (unsigned long long)gridDim.x * blockDim.x) {
    const float f = __int2float_rn((int)s);
    if (__float_as_int(sqrt_rn_fast(f)) != __float_as_int(__fsqrt_rn(f))) ++bad;
  }
  if (bad) atomicAdd(mismatch, bad);
}
cudaError_t launch_sqrt_check(unsigned long long *d_mismatch, cudaStream_t s)
{
  sqrt_check_kernel<<<148 * 16, 256, 0, s>>>(d_mismatch);
  return cudaGetLastError();
}


// ---- glue for channels the fused kernel does not demodulate itself (mode SYNCAM with the f32 PLL): rows and biquad words are
// copied out to dense scratch arrays, run through the stage kernels, and copied back (msdr_capi.cu).  The chain channel of scratch row i
// is chmap[i] when a channel map is given (a channel-list update), else ch0 + rows[i].
__global__ void gather_rows_kernel(const uint32_t *__restrict__ rows, const uint32_t *__restrict__ chmap, uint32_t ch0, const int16_t *__restrict__ hist, uint32_t H,
                                   const int16_t *__restrict__ in, size_t stride, int16_t *__restrict__ raw, uint32_t L)
{
  const uint32_t s = blockIdx.y, row = rows[s];
  const size_t Lp = (size_t)H + L, ch = chmap ? (size_t)chmap[s] : (size_t)ch0 + row;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < Lp; i += (size_t)gridDim.x * blockDim.x)
    raw[s * Lp + i] = i < H ? hist[ch * H + i] : in[(size_t)row * stride + (i - H)];
}
__global__ void scatter_rows_kernel(const uint32_t *__restrict__ rows, const int16_t *__restrict__ audio, size_t astride, int16_t *__restrict__ out,
                                    size_t stride, uint32_t L)
{
  const uint32_t s = blockIdx.y, row = rows[s];
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < L; i += (size_t)gridDim.x * blockDim.x)
    out[(size_t)row * stride + i] = audio[s * astride + i];
}
// d_bq is [2 objects * 4 stages * 8 words][Cpad]; defs is [object][n][32]
__global__ void bq_words_kernel(int dir, const uint32_t *__restrict__ rows, const uint32_t *__restrict__ chmap, uint32_t ch0, int32_t *__restrict__ bq, uint32_t Cpad,
                                int32_t *__restrict__ defs, uint32_t n)
{
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 64u) return;
  const uint32_t s = i / 64u, w = i % 64u; // w = object * 32 + word
  int32_t *g = bq + (size_t)w * Cpad + (chmap ? chmap[s] : ch0 + rows[s]);
  int32_t *d = defs + ((size_t)(w / 32u) * n + s) * 32u + (w % 32u);
  if (dir == 0) *d = *g; else *g = *d;
}
// demodulation switch with a kind per row (255 = leave the row alone); I/Q rows of pitch `stride`, output rows of pitch `ostride`
__global__ void demod_rows_kernel(const uint8_t *__restrict__ kinds, const int16_t *__restrict__ I, const int16_t *__restrict__ Q, size_t stride,
                                  int16_t *__restrict__ out, size_t ostride, uint32_t n)
{
  const uint32_t r = blockIdx.y;
  const int kind = kinds[r];
  if (kind > 3) return;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[r * ostride + i] = (int16_t)demod_sample(kind, I[r * stride + i], Q[r * stride + i]);
}
cudaError_t launch_demod_rows(const uint8_t *kinds, const int16_t *I, const int16_t *Q, size_t stride, int16_t *out, size_t ostride, uint32_t rows, uint32_t n,
                              cudaStream_t s)
{
  if (rows == 0 || n == 0) return cudaSuccess;
  for (uint32_t r0 = 0; r0 < rows; r0 += 32768u) // gridDim.y limit
    demod_rows_kernel<<<dim3(8, std::min(rows - r0, 32768u)), 256, 0, s>>>(kinds + r0, I + (size_t)r0 * stride, Q + (size_t)r0 * stride, stride, out + (size_t)r0 * ostride, ostride, n);
  return cudaGetLastError();
}
cudaError_t launch_gather_rows(const uint32_t *rows, const uint32_t *chmap, uint32_t n, uint32_t ch0, const int16_t *hist, uint32_t H, const int16_t *in, size_t stride,
                               int16_t *raw, uint32_t L, cudaStream_t s)
{
  if (n == 0) return cudaSuccess;
  for (uint32_t r0 = 0; r0 < n; r0 += 32768u) // gridDim.y limit
    gather_rows_kernel<<<dim3(8, std::min(n - r0, 32768u)), 256, 0, s>>>(rows + r0, chmap ? chmap + r0 : nullptr, ch0, hist, H, in, stride,
                                                                         raw + (size_t)r0 * ((size_t)H + L), L);
  return cudaGetLastError();
}
cudaError_t launch_scatter_rows(const uint32_t *rows, uint32_t n, const int16_t *audio, size_t astride, int16_t *out, size_t stride, uint32_t L, cudaStream_t s)
{
  if (n == 0) return cudaSuccess;
  for (uint32_t r0 = 0; r0 < n; r0 += 32768u)
    scatter_rows_kernel<<<dim3(8, std::min(n - r0, 32768u)), 256, 0, s>>>(rows + r0, audio + (size_t)r0 * astride, astride, out, stride, L);
  return cudaGetLastError();
}
// zero the raw-sample history rows of a list of channels (init_FIR's memset of both delay lines, Minimal-SDR.ino:902-903)
__global__ void zero_hist_rows_kernel(int16_t *__restrict__ hist, uint32_t H, const uint32_t *__restrict__ channels, uint32_t n)
{
  const uint32_t hq = H / 8; // uint4 per row
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (size_t)n * hq; i += (size_t)gridDim.x * blockDim.x)
    reinterpret_cast<uint4 *>(hist + (size_t)channels[i / hq] * H)[i % hq] = make_uint4(0, 0, 0, 0);
}
cudaError_t launch_zero_hist_rows(int16_t *hist, uint32_t H, const uint32_t *channels, uint32_t n, cudaStream_t s)
{
  if (n == 0) return cudaSuccess;
  const size_t total = (size_t)n * (H / 8);
  zero_hist_rows_kernel<<<(unsigned)std::min<size_t>((total + 255) / 256, 148 * 16), 256, 0, s>>>(hist, H, channels, n);
  return cudaGetLastError();
}
cudaError_t launch_bq_words(int dir, const uint32_t *rows, const uint32_t *chmap, uint32_t n, uint32_t ch0, int32_t *bq, uint32_t Cpad, int32_t *defs, cudaStream_t s)
{
  if (n == 0) return cudaSuccess;
  bq_words_kernel<<<(n * 64u + 255u) / 256u, 256, 0, s>>>(dir, rows, chmap, ch0, bq, Cpad, defs, n);
  return cudaGetLastError();
}

} // namespace msdr
