// msdr_anr.cu — K5: LMS automatic notch / noise reduction (SURVEY 8f rank 3), Minimal-SDR.ino:702-770, batched over channels.
// In the sketch it sits between the demodulation switch and queue_dac (the biquads follow as audio objects); here it is a
// stand-alone stateful operator on demodulated int16 audio (not fused into K1).
//
// Variable-leak LMS after Warren Pratt's wdsp: 64 taps on a 512-entry delay line, 16 samples of decorrelation delay, per sample
//   y = sum w[j] d[idx], sigma = sum d[idx]^2, error = d[now] - y, leak index / ngamma update, w[j] = c0 w[j] + c1 d[idx].
// float32 state with the `double` sub-expressions C gives the literals 1.0 and 1e-10.  Bit-exactness with the reference compiled
// by gcc for the host: every operation is a separately rounded IEEE operation in source order (explicit _rn intrinsics, no FMA
// contraction, no re-association of the 64-term sums).  That serial sum is also the bound: ~1 k instructions per sample.
//
// One warp owns 32 channels (lane = channel): delay lines in shared memory ([index][lane], conflict-free), weights in
// registers, blocks global -> shared -> global with cp.async like the front-end kernel.
#include "msdr_device.cuh"
#include "msdr_internal.h"
#include "../../include/msdr.h"

#include <string>
#include <vector>

namespace msdr {
namespace anr {

constexpr int kBlock = 128, kPitchW = kBlock / 2 + 4;
constexpr int kDline = 512, kTaps = 64, kDelay = 16; // .ino:707-709

struct Params {
  int16_t *data; // [C][stride], in place
  size_t stride;
  uint32_t C, Cpad, n_blocks;
  int mode;      // 1 notch (output = error), 2 noise reduction (output = y), .ino:749-750
  const uint8_t *row_mode; // optional per-row mode (0 = leave the row alone); overrides `mode`
  const uint32_t *chmap;   // optional row -> state index (receive chain: its channels with ANR switched on)
  float *d;      // [kDline][Cpad]
  float *w;      // [kTaps][Cpad]
  float *lidx, *ngamma;
  int *in_idx;
};

__global__ void __launch_bounds__(32) anr_kernel(const Params p)
{
  extern __shared__ __align__(16) unsigned char smem[];
  float *dl = reinterpret_cast<float *>(smem);                               // [kDline][32]
  uint32_t *buf = reinterpret_cast<uint32_t *>(smem + kDline * 32 * 4);      // [2][32][kPitchW]
  const int lane = threadIdx.x;
  const uint32_t g = blockIdx.x, row_id = g * kGroup + lane;
  const int mode = row_id < p.C ? (p.row_mode ? (int)p.row_mode[row_id] : p.mode) : 0;
  const bool active = row_id < p.C && mode != 0;
  const uint32_t ch = active ? (p.chmap ? p.chmap[row_id] : row_id) : 0;
  const int nrows = min(kGroup, (int)(p.C - g * kGroup));

  const float two_mu = (float)0.001, gamma = (float)0.1, lidx_min = 0.0f, lidx_max = 200.0f, den_mult = (float)6.25e-10, lincr = 1.0f, ldecr = 3.0f;
  float w[kTaps];
  float lidx = 120.0f, ngamma = 0.001f;
  int in_idx = 0;
  if (active) {
#pragma unroll
    for (int j = 0; j < kTaps; ++j) w[j] = p.w[(size_t)j * p.Cpad + ch];
    for (int k = 0; k < kDline; ++k) dl[k * 32 + lane] = p.d[(size_t)k * p.Cpad + ch];
    lidx = p.lidx[ch]; ngamma = p.ngamma[ch]; in_idx = p.in_idx[ch];
  } else {
#pragma unroll
    for (int j = 0; j < kTaps; ++j) w[j] = 0.0f;
  }

  const int r0 = lane >> 4, c = lane & 15; // coalesced copies: 2 rows of 256 bytes per warp instruction
  unsigned char *gbase = reinterpret_cast<unsigned char *>(p.data + ((size_t)g * kGroup + r0) * p.stride) + c * 16;
  const size_t gstep = 2 * p.stride * 2;
  auto issue = [&](uint32_t b) {
    const uint32_t sdst = smem_u32(buf + (b & 1) * (kGroup * kPitchW)) + (uint32_t)(r0 * kPitchW * 4 + c * 16);
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (r0 + 2 * j < nrows)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sdst + (uint32_t)(j * 2 * kPitchW * 4)), "l"(gbase + (size_t)b * kBlock * 2 + (size_t)j * gstep) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  issue(0);
  for (uint32_t b = 0; b < p.n_blocks; ++b) {
    if (b + 1 < p.n_blocks) { issue(b + 1); asm volatile("cp.async.wait_group 1;" ::: "memory"); }
    else asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    int16_t *row = reinterpret_cast<int16_t *>(buf + (b & 1) * (kGroup * kPitchW) + lane * kPitchW);
    if (active) {
#pragma unroll 1
      for (int i = 0; i < kBlock; ++i) {
        const float dcur = (float)row[i];
        dl[in_idx * 32 + lane] = dcur;
        float y = 0.0f, sigma = 0.0f;
        const int base = in_idx + kDelay;
#pragma unroll
        for (int j = 0; j < kTaps; ++j) {
          const float dv = dl[((base + j) & (kDline - 1)) * 32 + lane];
          y = __fadd_rn(y, __fmul_rn(w[j], dv));
          sigma = __fadd_rn(sigma, __fmul_rn(dv, dv));
        }
        const float inv_sigp = __double2float_rn(__ddiv_rn(1.0, __dadd_rn((double)sigma, 1e-10)));
        const float error = __fsub_rn(dcur, y);
        row[i] = (int16_t)__float2int_rz(mode == 1 ? error : y);
        float nel = __double2float_rn(__dmul_rn((double)error, __dsub_rn(1.0, (double)__fmul_rn(__fmul_rn(two_mu, sigma), inv_sigp))));
        if (nel < 0.0f) nel = -nel;
        const float t2 = __fmul_rn(__fmul_rn(__fmul_rn(two_mu, error), sigma), inv_sigp);
        float nev = __double2float_rn(__dsub_rn(__dsub_rn((double)dcur, __dmul_rn(__dsub_rn(1.0, (double)__fmul_rn(two_mu, ngamma)), (double)y)), (double)t2));
        if (nev < 0.0f) nev = -nev;
        if (nev < nel) {
          lidx = __fadd_rn(lidx, lincr);
          if (lidx > lidx_max) lidx = lidx_max;
          else { lidx = __fsub_rn(lidx, ldecr); if (lidx < lidx_min) lidx = lidx_min; }
        }
        const float l2 = __fmul_rn(lidx, lidx);
        ngamma = __fmul_rn(__fmul_rn(__fmul_rn(gamma, l2), l2), den_mult);
        const float c0 = __double2float_rn(__dsub_rn(1.0, (double)__fmul_rn(two_mu, ngamma)));
        const float c1 = __fmul_rn(__fmul_rn(two_mu, error), inv_sigp);
#pragma unroll
        for (int j = 0; j < kTaps; ++j) {
          const float dv = dl[((base + j) & (kDline - 1)) * 32 + lane];
          w[j] = __fadd_rn(__fmul_rn(c0, w[j]), __fmul_rn(c1, dv));
        }
        in_idx = (in_idx + (kDline - 1)) & (kDline - 1);
      }
    }
    __syncwarp();
    {
      const unsigned char *ssrc = reinterpret_cast<const unsigned char *>(buf + (b & 1) * (kGroup * kPitchW)) + r0 * kPitchW * 4 + c * 16;
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (r0 + 2 * j < nrows)
          *reinterpret_cast<uint4 *>(gbase + (size_t)b * kBlock * 2 + (size_t)j * gstep) = *reinterpret_cast<const uint4 *>(ssrc + j * 2 * kPitchW * 4);
    }
    __syncwarp();
  }
  if (active) {
#pragma unroll
    for (int j = 0; j < kTaps; ++j) p.w[(size_t)j * p.Cpad + ch] = w[j];
    for (int k = 0; k < kDline; ++k) p.d[(size_t)k * p.Cpad + ch] = dl[k * 32 + lane];
    p.lidx[ch] = lidx; p.ngamma[ch] = ngamma; p.in_idx[ch] = in_idx;
  }
}

constexpr size_t kSmem = (size_t)kDline * 32 * 4 + 2 * kGroup * kPitchW * 4;

} // namespace anr

// rows of demodulated audio in place; per-row mode and state index (msdr_capi.cu: channels of a receive chain with ANR on)
cudaError_t launch_anr(int16_t *data, size_t stride, uint32_t rows, uint32_t n_blocks, const uint8_t *row_mode, const uint32_t *chmap, float *d, float *w,
                       float *lidx, float *ngamma, int *in_idx, uint32_t Cpad, cudaStream_t s)
{
  if (rows == 0 || n_blocks == 0) return cudaSuccess;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(anr::anr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)anr::kSmem);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  anr::Params p{};
  p.data = data; p.stride = stride; p.C = rows; p.Cpad = Cpad; p.n_blocks = n_blocks; p.mode = 0; p.row_mode = row_mode; p.chmap = chmap;
  p.d = d; p.w = w; p.lidx = lidx; p.ngamma = ngamma; p.in_idx = in_idx;
  anr::anr_kernel<<<(rows + kGroup - 1) / kGroup, 32, anr::kSmem, s>>>(p);
  return cudaGetLastError();
}
} // namespace msdr

struct msdr_anr {
  int device = 0;
  uint32_t C = 0, Cpad = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  float *d_d = nullptr, *d_w = nullptr, *d_lidx = nullptr, *d_ngamma = nullptr;
  int *d_in_idx = nullptr;
  int16_t *d_data = nullptr;
  size_t stage_samples = 0;
  uint64_t launches = 0;
  std::string err;
};

namespace {
thread_local std::string g_anr_error;
int anr_fail(msdr_anr *a, int code, const std::string &msg) { if (a) a->err = msg; else g_anr_error = msg; return code; }
#define ACK(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return anr_fail(anr, MSDR_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); } while (0)
}

extern "C" {

const char *msdr_anr_last_error(const msdr_anr *anr) { return anr ? anr->err.c_str() : g_anr_error.c_str(); }

int msdr_anr_create(msdr_anr **out, int device, uint32_t n_channels)
{
  if (!out || n_channels == 0) return anr_fail(nullptr, MSDR_ERR_ARGUMENT, "anr_create: bad arguments");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return anr_fail(nullptr, MSDR_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
  if (device < 0 || device >= ndev) return anr_fail(nullptr, MSDR_ERR_ARGUMENT, "anr_create: bad device");
  msdr_anr *anr = new msdr_anr();
  anr->device = device; anr->C = n_channels; anr->Cpad = (n_channels + 31u) & ~31u;
  const size_t cp = anr->Cpad;
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&anr->own_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaMalloc(&anr->d_d, msdr::anr::kDline * cp * 4);
  if (e == cudaSuccess) e = cudaMalloc(&anr->d_w, msdr::anr::kTaps * cp * 4);
  if (e == cudaSuccess) e = cudaMalloc(&anr->d_lidx, cp * 4);
  if (e == cudaSuccess) e = cudaMalloc(&anr->d_ngamma, cp * 4);
  if (e == cudaSuccess) e = cudaMalloc(&anr->d_in_idx, cp * 4);
  if (e == cudaSuccess) e = cudaMemset(anr->d_d, 0, msdr::anr::kDline * cp * 4);
  if (e == cudaSuccess) e = cudaMemset(anr->d_w, 0, msdr::anr::kTaps * cp * 4);
  if (e == cudaSuccess) e = cudaMemset(anr->d_in_idx, 0, cp * 4);
  if (e == cudaSuccess) {
    std::vector<float> l(cp, msdr::kAnrLidx0), n(cp, msdr::kAnrNgamma0);
    e = cudaMemcpy(anr->d_lidx, l.data(), cp * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(anr->d_ngamma, n.data(), cp * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaDeviceSynchronize(); // legacy-stream copies / memsets vs this object's non-blocking stream
  }
  if (e == cudaSuccess) e = cudaFuncSetAttribute(msdr::anr::anr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msdr::anr::kSmem);
  if (e != cudaSuccess) {
    g_anr_error = std::string("anr_create: ") + cudaGetErrorString(e);
    cudaFree(anr->d_d); cudaFree(anr->d_w); cudaFree(anr->d_lidx); cudaFree(anr->d_ngamma); cudaFree(anr->d_in_idx);
    if (anr->own_stream) cudaStreamDestroy(anr->own_stream);
    delete anr;
    return MSDR_ERR_CUDA;
  }
  anr->stream = anr->own_stream;
  *out = anr;
  return MSDR_OK;
}

void msdr_anr_destroy(msdr_anr *anr)
{
  if (!anr) return;
  cudaSetDevice(anr->device);
  if (anr->stream) cudaStreamSynchronize(anr->stream);
  cudaFree(anr->d_d); cudaFree(anr->d_w); cudaFree(anr->d_lidx); cudaFree(anr->d_ngamma); cudaFree(anr->d_in_idx); cudaFree(anr->d_data);
  if (anr->own_stream) cudaStreamDestroy(anr->own_stream);
  delete anr;
}

int msdr_anr_set_stream(msdr_anr *anr, void *cuda_stream)
{
  if (!anr) return MSDR_ERR_ARGUMENT;
  anr->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : anr->own_stream;
  return MSDR_OK;
}

int msdr_anr_synchronize(msdr_anr *anr)
{
  if (!anr) return MSDR_ERR_ARGUMENT;
  ACK(cudaSetDevice(anr->device));
  ACK(cudaStreamSynchronize(anr->stream));
  return MSDR_OK;
}

int msdr_anr_update_device(msdr_anr *anr, int mode, int16_t *d_data, uint32_t n_blocks, size_t stride)
{
  if (!anr) return MSDR_ERR_ARGUMENT;
  if (mode != 1 && mode != 2) return anr_fail(anr, MSDR_ERR_ARGUMENT, "anr_update: mode must be 1 (notch) or 2 (noise reduction); 0 = off is the caller not calling");
  if (n_blocks == 0) return MSDR_OK;
  if (!d_data || (uint64_t)n_blocks * MSDR_BLOCK_SAMPLES > stride) return anr_fail(anr, MSDR_ERR_ARGUMENT, "anr_update: bad buffer / stride < n_blocks*128");
  if (((uintptr_t)d_data & 15u) || (stride & 7u)) return anr_fail(anr, MSDR_ERR_ARGUMENT, "anr_update_device: buffer must be 16-byte aligned and stride a multiple of 8 samples");
  ACK(cudaSetDevice(anr->device));
  msdr::anr::Params p{};
  p.data = d_data; p.stride = stride; p.C = anr->C; p.Cpad = anr->Cpad; p.n_blocks = n_blocks; p.mode = mode; p.row_mode = nullptr; p.chmap = nullptr;
  p.d = anr->d_d; p.w = anr->d_w; p.lidx = anr->d_lidx; p.ngamma = anr->d_ngamma; p.in_idx = anr->d_in_idx;
  msdr::anr::anr_kernel<<<(anr->C + msdr::kGroup - 1) / msdr::kGroup, 32, msdr::anr::kSmem, anr->stream>>>(p);
  ACK(cudaGetLastError());
  anr->launches++;
  return MSDR_OK;
}

int msdr_anr_update(msdr_anr *anr, int mode, int16_t *data, uint32_t n_blocks, size_t stride)
{
  if (!anr) return MSDR_ERR_ARGUMENT;
  if (n_blocks == 0) return MSDR_OK;
  if (!data || (uint64_t)n_blocks * MSDR_BLOCK_SAMPLES > stride) return anr_fail(anr, MSDR_ERR_ARGUMENT, "anr_update: bad buffer / stride < n_blocks*128");
  ACK(cudaSetDevice(anr->device));
  const size_t L = (size_t)n_blocks * MSDR_BLOCK_SAMPLES, need = (size_t)anr->C * L;
  if (need > anr->stage_samples) {
    ACK(cudaStreamSynchronize(anr->stream));
    cudaFree(anr->d_data);
    anr->d_data = nullptr; anr->stage_samples = 0;
    ACK(cudaMalloc(&anr->d_data, need * 2));
    anr->stage_samples = need;
  }
  ACK(cudaMemcpy2DAsync(anr->d_data, L * 2, data, stride * 2, L * 2, anr->C, cudaMemcpyHostToDevice, anr->stream));
  ACK(cudaDeviceSynchronize()); // the copies ran in the legacy stream; this object's stream is non-blocking
  int st = msdr_anr_update_device(anr, mode, anr->d_data, n_blocks, L);
  if (st != MSDR_OK) return st;
  ACK(cudaMemcpy2DAsync(data, stride * 2, anr->d_data, L * 2, L * 2, anr->C, cudaMemcpyDeviceToHost, anr->stream));
  ACK(cudaStreamSynchronize(anr->stream));
  return MSDR_OK;
}

int msdr_anr_get_state(msdr_anr *anr, uint32_t ch, msdr_anr_state *out)
{
  if (!anr || !out || ch >= anr->C) return MSDR_ERR_ARGUMENT;
  ACK(cudaSetDevice(anr->device));
  ACK(cudaStreamSynchronize(anr->stream));
  ACK(cudaMemcpy2D(out->d, 4, anr->d_d + ch, (size_t)anr->Cpad * 4, 4, msdr::anr::kDline, cudaMemcpyDeviceToHost));
  ACK(cudaMemcpy2D(out->w, 4, anr->d_w + ch, (size_t)anr->Cpad * 4, 4, msdr::anr::kTaps, cudaMemcpyDeviceToHost));
  ACK(cudaMemcpy(&out->lidx, anr->d_lidx + ch, 4, cudaMemcpyDeviceToHost));
  ACK(cudaMemcpy(&out->ngamma, anr->d_ngamma + ch, 4, cudaMemcpyDeviceToHost));
  ACK(cudaMemcpy(&out->in_idx, anr->d_in_idx + ch, 4, cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

int msdr_anr_set_state(msdr_anr *anr, uint32_t ch, const msdr_anr_state *in)
{
  if (!anr || !in || ch >= anr->C || in->in_idx < 0 || in->in_idx >= msdr::anr::kDline) return MSDR_ERR_ARGUMENT;
  ACK(cudaSetDevice(anr->device));
  ACK(cudaStreamSynchronize(anr->stream));
  ACK(cudaMemcpy2D(anr->d_d + ch, (size_t)anr->Cpad * 4, in->d, 4, 4, msdr::anr::kDline, cudaMemcpyHostToDevice));
  ACK(cudaMemcpy2D(anr->d_w + ch, (size_t)anr->Cpad * 4, in->w, 4, 4, msdr::anr::kTaps, cudaMemcpyHostToDevice));
  ACK(cudaMemcpy(anr->d_lidx + ch, &in->lidx, 4, cudaMemcpyHostToDevice));
  ACK(cudaMemcpy(anr->d_ngamma + ch, &in->ngamma, 4, cudaMemcpyHostToDevice));
  ACK(cudaMemcpy(anr->d_in_idx + ch, &in->in_idx, 4, cudaMemcpyHostToDevice));
  ACK(cudaDeviceSynchronize()); // the copies ran in the legacy stream; this object's stream is non-blocking
  return MSDR_OK;
}

uint64_t msdr_anr_launch_count(const msdr_anr *anr) { return anr ? anr->launches : 0; }

} // extern "C"
