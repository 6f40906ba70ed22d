// msdr_frontend.cu — K4: front-end conditioning in front of the receive chain (SURVEY 8f rank 1), batched over channels:
//   raw unsigned ADC codes -> 1-pole DC-blocking high-pass in S1.30 (AudioInputAnalog::update, input_adc.cpp:198-212)
//   -> AudioAmplifier gain with SSAT16 (mixer.cpp:34-47,134-159, mixer.h:75-79) -> int16 IF samples,
//   and per 128-sample block the AGC of the sketch (Minimal-SDR.ino:445-515): block maximum of |x| through the halfword SIMD
//   idiom, 25-block history, float gain law, new amplifier multiplier for the blocks that follow.
// Signal order: adc1 -> amp_adc -> queue_adc (.ino:76-78), AGC(p_adc) on each block read from the queue (.ino:530-534).
// Batch semantics: zero queue latency, block k+1 is amplified with the gain AGC set after block k.
//
// The high-pass is a truncating recurrence per sample and the AGC a feedback per block: serial in time per channel, parallel
// over channels.  One warp owns 32 channels (lane = channel) for the whole call; half blocks travel global -> shared (cp.async,
// coalesced, three buffers) -> lane-per-row processing in place -> global.  Bound: per-sample dependent latency of the
// recurrence (~25 cycles) for few channels, HBM (4 B per sample) for many.
#include "msdr_device.cuh"
#include "msdr_frontend.cuh"
#include "msdr_internal.h"
#include "../../include/msdr.h"

#include <cstring>
#include <algorithm>
#include <string>
#include <vector>

namespace msdr {
namespace fe {

struct Params {
  const uint16_t *adc; // [C][stride] raw codes
  int16_t *out;        // [C][stride]
  size_t stride;
  uint32_t C, n_blocks;
  State *state;        // [C]
  float agc_max;
  int agc_on;
};

// Shared memory decides how many of these one-warp CTAs an SM holds: the blocks travel in pieces of kPart samples through a
// ring of kNBuf buffers (64 samples, three deep: 13.8 KB per CTA, 16 CTAs per SM).
// The warps of a CTA are independent (only __syncwarp): blockDim.x / 32 > 1 packs several channel groups onto one SM, which confines
// the kernel to a few SMs so that a chain kernel that leaves SMs free can run beside it (msdr_frontend_set_option "sms").
template <int kPart, int kNBuf>
__global__ void frontend_kernel(const Params p)
{
  constexpr int kPartPitchW = kPart / 2 + 4;     // 4 mod 32, conflict-free row-wise 128-bit access
  constexpr int RPI = 512 / (kPart * 2);         // rows per warp instruction
  constexpr int CPR = 32 / RPI;                  // 16-byte chunks per row
  extern __shared__ __align__(16) uint32_t fe_smem[];
  uint32_t (*buf)[kGroup * kPartPitchW] = reinterpret_cast<uint32_t (*)[kGroup * kPartPitchW]>(fe_smem + (size_t)(threadIdx.x >> 5) * kNBuf * kGroup * kPartPitchW);
  const int lane = threadIdx.x & 31;
  const uint32_t g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), row = g * kGroup + lane;
  if (g * kGroup >= p.C) return; // a warp past the last channel group (whole warps only: nothing below is block-wide)
  const bool active = row < p.C;
  const int nrows = min(kGroup, (int)(p.C - g * kGroup));
  State s;
  if (active) s = p.state[row];

  // coalesced mapping for the copies: 4 rows of 128 bytes per warp instruction
  const int r0 = lane / CPR, c = lane % CPR;
  const unsigned char *gin = reinterpret_cast<const unsigned char *>(p.adc + ((size_t)g * kGroup + r0) * p.stride) + c * 16;
  unsigned char *gout = reinterpret_cast<unsigned char *>(p.out + ((size_t)g * kGroup + r0) * p.stride) + c * 16;
  const size_t gstep = (size_t)RPI * p.stride * 2;
  const uint32_t nparts = p.n_blocks * (kBlock / kPart);
  auto issue = [&](uint32_t h) {
    if (h < nparts) {
      const uint32_t sdst = smem_u32(buf[h % kNBuf]) + (uint32_t)(r0 * kPartPitchW * 4 + c * 16);
#pragma unroll
      for (int j = 0; j < 32 / RPI; ++j)
        if (r0 + RPI * j < nrows)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sdst + (uint32_t)(j * RPI * kPartPitchW * 4)), "l"(gin + (size_t)h * kPart * 2 + (size_t)j * gstep) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory"); // one group per piece, empty past the end: the wait below stays uniform
  };
#pragma unroll
  for (int i = 0; i < kNBuf - 1; ++i) issue(i);
  int x1 = s.hpf_x1, y1 = s.hpf_y1;
  uint32_t maxv = kMaxInit, minv = kMinInit;
  for (uint32_t h = 0; h < nparts; ++h) {
    issue(h + kNBuf - 1); // its buffer held piece h - 1, written back (and fenced by the __syncwarp) at the end of the last iteration
    asm volatile("cp.async.wait_group %0;" ::"n"(kNBuf - 1) : "memory");
    __syncwarp();
    uint32_t *rowp = buf[h % kNBuf] + lane * kPartPitchW;
    if (active) {
      const int mult = s.mult;
#pragma unroll 1
      for (int q = 0; q < kPart / 8; ++q) {
        uint4 v = *reinterpret_cast<const uint4 *>(rowp + 4 * q);
        uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) w[i] = condition2(w[i], x1, y1, mult, maxv, minv);
        *reinterpret_cast<uint4 *>(rowp + 4 * q) = make_uint4(w[0], w[1], w[2], w[3]);
      }
      if ((h % (kBlock / kPart)) == kBlock / kPart - 1) { // an audio block is complete
        if (p.agc_on) agc_update(s, block_absmax(maxv, minv), p.agc_max);
        maxv = kMaxInit; minv = kMinInit;
      }
    }
    __syncwarp();
    { // write the piece back, coalesced
      const unsigned char *ssrc = reinterpret_cast<const unsigned char *>(buf[h % kNBuf]) + r0 * kPartPitchW * 4 + c * 16;
#pragma unroll
      for (int j = 0; j < 32 / RPI; ++j)
        if (r0 + RPI * j < nrows)
          *reinterpret_cast<uint4 *>(gout + (size_t)h * kPart * 2 + (size_t)j * gstep) = *reinterpret_cast<const uint4 *>(ssrc + j * RPI * kPartPitchW * 4);
    }
    __syncwarp(); // this buffer is the target of the copy issued at the top of the next iteration
  }
  s.hpf_x1 = x1; s.hpf_y1 = y1;
  if (active) p.state[row] = s;
}

} // namespace fe

// piece length / ring depth measured at 65 536 and 262 144 channels (profiles/r01_frontend.txt): <64, 3> 1018 / 1189 Gsamples/s,
// <128, 2> 914 / 1225, <64, 2> 1043 / 1153, <32, 4> 1040 / 1125, <32, 3> 1031 / 1027, <64, 4> 884 / 1195
cudaError_t launch_frontend(const uint16_t *adc, int16_t *out, size_t stride, uint32_t C, uint32_t n_blocks, fe::State *state, float agc_max,
                            int agc_on, int sms, cudaStream_t s)
{
  fe::Params p{};
  p.adc = adc; p.out = out; p.stride = stride; p.C = C; p.n_blocks = n_blocks; p.state = state;
  p.agc_max = agc_max; p.agc_on = agc_on;
  constexpr int kPart = 64, kNBuf = 3;
  const uint32_t groups = (C + kGroup - 1) / kGroup;
  const size_t warp_smem = (size_t)kNBuf * kGroup * (kPart / 2 + 4) * 4; // 13.8 KB per channel group
  uint32_t wpc = 1;
  if (sms > 0) wpc = std::min<uint32_t>(16, std::max<uint32_t>(1, (groups + (uint32_t)sms - 1) / (uint32_t)sms));
  auto kern = fe::frontend_kernel<kPart, kNBuf>;
  if (wpc * warp_smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(wpc * warp_smem));
    if (e != cudaSuccess) return e;
  }
  kern<<<(groups + wpc - 1) / wpc, 32 * wpc, wpc * warp_smem, s>>>(p);
  return cudaGetLastError();
}

} // namespace msdr

// ------------------------------------------------------------------------------------------------------------------------
struct msdr_frontend {
  int device = 0;
  uint32_t C = 0;
  float agc_start = 0.25f, agc_max = 40.0f;
  int agc_on = 1;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  msdr::fe::State *d_state = nullptr;
  uint16_t *d_in = nullptr;
  int16_t *d_out = nullptr;
  size_t stage_samples = 0;
  uint64_t launches = 0;
  int sms = 0; // option "sms": > 0 = pack the channel groups into about this many CTAs of several warps (one per SM)
  std::string err;
};

namespace {
thread_local std::string g_fe_error;
int fe_fail(msdr_frontend *f, int code, const std::string &msg) { if (f) f->err = msg; else g_fe_error = msg; return code; }
#define FCK(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fe_fail(fe, MSDR_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); } while (0)
}

extern "C" {

const char *msdr_frontend_last_error(const msdr_frontend *fe) { return fe ? fe->err.c_str() : g_fe_error.c_str(); }

int msdr_frontend_create(msdr_frontend **out, int device, uint32_t n_channels, float agc_start, float agc_max, int agc_on)
{
  if (!out || n_channels == 0) return fe_fail(nullptr, MSDR_ERR_ARGUMENT, "frontend_create: bad arguments");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fe_fail(nullptr, MSDR_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
  if (device < 0 || device >= ndev) return fe_fail(nullptr, MSDR_ERR_ARGUMENT, "frontend_create: bad device");
  msdr_frontend *fe = new msdr_frontend();
  fe->device = device; fe->C = n_channels; fe->agc_start = agc_start; fe->agc_max = agc_max; fe->agc_on = agc_on;
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&fe->own_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaMalloc(&fe->d_state, (size_t)n_channels * sizeof(msdr::fe::State));
  if (e != cudaSuccess) { g_fe_error = std::string("frontend_create: ") + cudaGetErrorString(e); delete fe; return MSDR_ERR_CUDA; }
  fe->stream = fe->own_stream;
  std::vector<msdr::fe::State> h(n_channels);
  for (auto &s : h) {
    s = msdr::fe::State{};
    s.agc_idx = msdr::fe::kAgcBuf;                    // .ino:451
    s.agc_val = agc_start;                            // .ino:104
    s.mult = msdr::fe::amp_multiplier(agc_start);     // .ino:385
  }
  e = cudaMemcpy(fe->d_state, h.data(), h.size() * sizeof(msdr::fe::State), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaDeviceSynchronize(); // legacy-stream copy vs this object's non-blocking stream
  if (e != cudaSuccess) { g_fe_error = std::string("frontend_create: ") + cudaGetErrorString(e); cudaFree(fe->d_state); delete fe; return MSDR_ERR_CUDA; }
  *out = fe;
  return MSDR_OK;
}

void msdr_frontend_destroy(msdr_frontend *fe)
{
  if (!fe) return;
  cudaSetDevice(fe->device);
  if (fe->stream) cudaStreamSynchronize(fe->stream);
  cudaFree(fe->d_state); cudaFree(fe->d_in); cudaFree(fe->d_out);
  if (fe->own_stream) cudaStreamDestroy(fe->own_stream);
  delete fe;
}

int msdr_frontend_set_stream(msdr_frontend *fe, void *cuda_stream)
{
  if (!fe) return MSDR_ERR_ARGUMENT;
  fe->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : fe->own_stream;
  return MSDR_OK;
}

int msdr_frontend_synchronize(msdr_frontend *fe)
{
  if (!fe) return MSDR_ERR_ARGUMENT;
  FCK(cudaSetDevice(fe->device));
  FCK(cudaStreamSynchronize(fe->stream));
  return MSDR_OK;
}

/* AudioInputAnalog::init (input_adc.cpp:59-63): x1 = first reading << 14, y1 = 0 */
int msdr_frontend_preset(msdr_frontend *fe, uint32_t ch0, uint32_t nch, uint16_t first_reading)
{
  if (!fe || (uint64_t)ch0 + nch > fe->C) return fe_fail(fe, MSDR_ERR_ARGUMENT, "frontend_preset: bad channel range");
  FCK(cudaSetDevice(fe->device));
  FCK(cudaStreamSynchronize(fe->stream));
  std::vector<msdr::fe::State> h(nch);
  if (nch == 0) return MSDR_OK;
  FCK(cudaMemcpy(h.data(), fe->d_state + ch0, nch * sizeof(msdr::fe::State), cudaMemcpyDeviceToHost));
  for (auto &s : h) { s.hpf_x1 = (int32_t)((uint32_t)first_reading << 14); s.hpf_y1 = 0; }
  FCK(cudaMemcpy(fe->d_state + ch0, h.data(), nch * sizeof(msdr::fe::State), cudaMemcpyHostToDevice));
  FCK(cudaDeviceSynchronize()); // the copies ran in the legacy stream; this object's stream is non-blocking
  return MSDR_OK;
}

int msdr_frontend_update_device(msdr_frontend *fe, const uint16_t *d_adc, int16_t *d_out, uint32_t n_blocks, size_t stride)
{
  if (!fe) return MSDR_ERR_ARGUMENT;
  if (n_blocks == 0) return MSDR_OK;
  if (!d_adc || !d_out || (uint64_t)n_blocks * MSDR_BLOCK_SAMPLES > stride) return fe_fail(fe, MSDR_ERR_ARGUMENT, "frontend_update: bad buffers / stride < n_blocks*128");
  if (((uintptr_t)d_adc & 15u) || ((uintptr_t)d_out & 15u) || (stride & 7u))
    return fe_fail(fe, MSDR_ERR_ARGUMENT, "frontend_update_device: buffers must be 16-byte aligned and stride a multiple of 8 samples");
  FCK(cudaSetDevice(fe->device));
  FCK(msdr::launch_frontend(d_adc, d_out, stride, fe->C, n_blocks, fe->d_state, fe->agc_max, fe->agc_on, fe->sms, fe->stream));
  fe->launches++;
  return MSDR_OK;
}

int msdr_frontend_update(msdr_frontend *fe, const uint16_t *adc, int16_t *out, uint32_t n_blocks, size_t stride)
{
  if (!fe) return MSDR_ERR_ARGUMENT;
  if (n_blocks == 0) return MSDR_OK;
  if (!adc || !out || (uint64_t)n_blocks * MSDR_BLOCK_SAMPLES > stride) return fe_fail(fe, MSDR_ERR_ARGUMENT, "frontend_update: bad buffers / stride < n_blocks*128");
  FCK(cudaSetDevice(fe->device));
  const size_t L = (size_t)n_blocks * MSDR_BLOCK_SAMPLES, need = (size_t)fe->C * L;
  if (need > fe->stage_samples) {
    FCK(cudaStreamSynchronize(fe->stream));
    cudaFree(fe->d_in); cudaFree(fe->d_out);
    fe->d_in = nullptr; fe->d_out = nullptr; fe->stage_samples = 0;
    FCK(cudaMalloc(&fe->d_in, need * 2));
    FCK(cudaMalloc(&fe->d_out, need * 2));
    fe->stage_samples = need;
  }
  FCK(cudaMemcpy2DAsync(fe->d_in, L * 2, adc, stride * 2, L * 2, fe->C, cudaMemcpyHostToDevice, fe->stream));
  FCK(cudaDeviceSynchronize()); // the copies ran in the legacy stream; this object's stream is non-blocking
  int st = msdr_frontend_update_device(fe, fe->d_in, fe->d_out, n_blocks, L);
  if (st != MSDR_OK) return st;
  FCK(cudaMemcpy2DAsync(out, stride * 2, fe->d_out, L * 2, L * 2, fe->C, cudaMemcpyDeviceToHost, fe->stream));
  FCK(cudaStreamSynchronize(fe->stream));
  return MSDR_OK;
}

int msdr_frontend_get_state(msdr_frontend *fe, uint32_t ch, msdr_frontend_state *out)
{
  if (!fe || !out || ch >= fe->C) return MSDR_ERR_ARGUMENT;
  static_assert(sizeof(msdr_frontend_state) == sizeof(msdr::fe::State), "public and device state layouts must match");
  FCK(cudaSetDevice(fe->device));
  FCK(cudaStreamSynchronize(fe->stream));
  FCK(cudaMemcpy(out, fe->d_state + ch, sizeof(*out), cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

int msdr_frontend_set_state(msdr_frontend *fe, uint32_t ch, const msdr_frontend_state *in)
{
  if (!fe || !in || ch >= fe->C) return MSDR_ERR_ARGUMENT;
  // agc_idx indexes the 25-entry block-maximum history after a pre-decrement (Minimal-SDR.ino:481): the sketch only ever holds
  // 0..25 there; anything else (a corrupt or foreign checkpoint) would be an out-of-bounds store in the kernel
  if (in->agc_idx < 0 || in->agc_idx > msdr::fe::kAgcBuf) {
    fe->err = "frontend_set_state: agc_idx outside [0, 25]";
    return MSDR_ERR_ARGUMENT;
  }
  FCK(cudaSetDevice(fe->device));
  FCK(cudaStreamSynchronize(fe->stream));
  FCK(cudaMemcpy(fe->d_state + ch, in, sizeof(*in), cudaMemcpyHostToDevice));
  FCK(cudaDeviceSynchronize()); // the copies ran in the legacy stream; this object's stream is non-blocking
  return MSDR_OK;
}

uint64_t msdr_frontend_launch_count(const msdr_frontend *fe) { return fe ? fe->launches : 0; }

int msdr_frontend_set_option(msdr_frontend *fe, const char *key, int value)
{
  if (!fe || !key) return MSDR_ERR_ARGUMENT;
  if (!strcmp(key, "sms")) { fe->sms = value < 0 ? 0 : value; return MSDR_OK; }
  return fe_fail(fe, MSDR_ERR_ARGUMENT, std::string("unknown option ") + key);
}

int32_t msdr_amp_gain_multiplier(float gain) { return msdr::fe::amp_multiplier(gain); }

} // extern "C"
