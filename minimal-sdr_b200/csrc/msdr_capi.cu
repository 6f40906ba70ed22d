// msdr_capi.cu — the C ABI declared in include/msdr.h: chain object, configuration, updates, stage operators.
// Host-side only plumbing; every computation is a CUDA kernel from the msdr_chain_v*.cu / msdr_stage_kernels.cu files.
#include "../../include/msdr.h"
#include "msdr_frontend.cuh"
#include "msdr_internal.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace msdr;

namespace {

thread_local std::string g_create_error;

struct FirSet {
  uint32_t T = 0;
  std::vector<int16_t> cI, cQ;
  uint32_t users = 0;
};

// Split one (cI, cQ) table into the four polyphase sub-filters of the fs/4 mix + FIR pair; KP = roundup4(T/2 + 1).
// With k' = d - (KP - T/2):  A[d] = cI[2k'], B[d] = cI[2k'+1], C[d] = cQ[2k'+1], D[d] = cQ[2(k'+1)], zero outside.
// Derivation in DESIGN.md ("Polyphase form of the fs/4 mix + FIR"); tc_build_bmat turns them into the Toeplitz operands.
void expand_set_int(uint32_t T, const int16_t *cI, const int16_t *cQ, std::vector<int> &A, std::vector<int> &B, std::vector<int> &C, std::vector<int> &D)
{
  const int half = (int)T / 2, KP = (int)kp_of_taps(T);
  A.assign(KP, 0); B.assign(KP, 0); C.assign(KP, 0); D.assign(KP, 0);
  for (int d = 0; d < KP; ++d) {
    const int kq = d - (KP - half);
    if (kq >= 0 && kq < half) { A[d] = cI[2 * kq]; B[d] = cI[2 * kq + 1]; C[d] = cQ[2 * kq + 1]; }
    if (kq + 1 >= 0 && kq + 1 < half) D[d] = cQ[2 * (kq + 1)];
  }
}

} // namespace

struct msdr_chain {
  int device = 0;
  uint32_t C = 0, Cpad = 0, max_taps = 0, KPmax = 0, H = 0, flags = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr, copy_in = nullptr, copy_out = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::vector<cudaEvent_t> pipe_ev;
  bool timed = false;
  // processor usage (AudioProcessorUsage / AudioProcessorUsageMax of the Teensy core, Minimal-SDR.ino:424-426): device time of an
  // update per 128-sample block, last and running maximum; `usage_pending` = events of the last timed update not read back yet
  bool usage_pending = false;
  uint32_t usage_blocks = 0;
  float usage_last_ms_per_block = 0.f, usage_max_ms_per_block = 0.f;

  std::vector<uint8_t> h_mode, h_set; // h_set: 0xFF = FIR not initialised
  uint32_t n_uninit = 0;
  std::vector<FirSet> sets;

  uint8_t *d_mode = nullptr, *d_set = nullptr;
  int16_t *d_hist = nullptr;
  int32_t *d_bq = nullptr;
  int *d_ctrl = nullptr;       // [2] chain kernel v4: work counter, spans taken

  // staging for host-buffer updates
  int16_t *d_in = nullptr, *d_out = nullptr;
  size_t stage_samples = 0; // per buffer
  int16_t *pin_in = nullptr, *pin_out = nullptr;
  size_t pin_samples = 0;

  // tensor-core FIR plan (chain kernel v4): rows sorted by tap table inside each wave of chains, see build_tc_plan()
  uint64_t meta_version = 1;  // bumped whenever a channel's table binding or a table's contents change
  struct TcPlan {
    uint64_t version = 0;
    uint32_t ch0 = 0, nch = 0, sms = 0, W = 0, K = 0, rings[4] = {0, 0, 0, 0}, n_rb = 0, n_waves = 0;
    bool want_dual = false, want_v6 = false, dual = false;
    uint32_t ring_v5 = 0;  // msdr_chain_v5.cu: operand ring depth, 0 = the window does not fit that kernel
    uint32_t ring_v5l = 0; // msdr_chain_v5l.cu (half-tile hand-offs, for the 256-tap window)
    uint32_t slots_v6 = 0, n_gb = 0; // msdr_chain_v6.cu: sub-tile slots (0 = the window does not fit), group blocks of 32 same-table rows
    uint32_t *d_rowmap32 = nullptr;
    uint4 *d_rb32 = nullptr;
    uint32_t *d_rowmap = nullptr, *d_wave_rb0 = nullptr;
    uint4 *d_rb = nullptr;
    uint8_t *d_bmat = nullptr;
    std::vector<uint32_t> list;  // a channel-list plan: row r is chain channel list[r] (ch0 = 0, nch = list size); empty for a range
    uint32_t *d_list = nullptr;  // the same on the device (ChainParams::chlist)
  };
  // one plan per updated channel range or channel list: msdr_chain_update cuts wide chains into channel chunks, each its own range
  static constexpr size_t kMaxPlans = 64;
  std::vector<TcPlan> plans;
  size_t plan_victim = 0;
  // channel-list updates: list_seen[c] == list_stamp marks a channel already met in the list being checked
  std::vector<uint32_t> list_seen;
  uint32_t list_stamp = 0;
  int *d_tile_cnt = nullptr;
  size_t tile_cnt_len = 0;

  // mode SYNCAM with the f32 PLL (.ino:631-688): a serial loop through sinf/cosf/atan2f per channel, run beside the fused kernel
  // on dense scratch copies of those channels (see syncam_lane_*)
  float *d_pll = nullptr;            // [3][Cpad] fil_out, omega2, phzerror
  // LMS notch / noise reduction between demodulation and the biquads (.ino:702-770), per channel 0 = off, 1, 2; same lane
  std::vector<uint8_t> h_anr;
  uint32_t n_anr = 0;                // channels with ANR on
  float *d_anr_d = nullptr, *d_anr_w = nullptr, *d_anr_lidx = nullptr, *d_anr_ngamma = nullptr; // allocated on first use
  int *d_anr_idx = nullptr;
  struct PllLane {
    std::vector<uint32_t> rows;      // launch-relative rows, ordered by tap table
    uint32_t *d_rows = nullptr, *d_chmap = nullptr;
    uint8_t *d_kind = nullptr, *d_anr_mode = nullptr;
    bool any_pll = false, any_anr = false;
    bool dirty = true;                 // modes / ANR switches changed: rebuild `channels`
    uint64_t epoch = 0;                // counts those changes
    // the index vectors of the last update's range stay valid (host copies persist: their uploads are asynchronous)
    bool cached = false;
    uint64_t key_epoch = 0, key_version = 0;
    uint32_t key_ch0 = 0, key_nch = 0;
    std::vector<uint32_t> key_list;    // the channel list of the last update; empty for a range
    std::vector<uint32_t> chmap;
    std::vector<uint8_t> kind, amode;
    std::vector<uint32_t> channels;    // every chain channel that needs the lane, ascending
    int16_t *d_raw = nullptr, *d_I = nullptr, *d_Q = nullptr, *d_If = nullptr, *d_Qf = nullptr, *d_taps = nullptr;
    int32_t *d_defs = nullptr;
    size_t cap_rows = 0, cap_samples = 0;
  } pll;

  int16_t *d_set_taps = nullptr;     // [MSDR_MAX_FIR_SETS][2][MSDR_MAX_TAPS] every live table's raw taps (the side lane's FIR launches read them)
  // ADC-code input (msdr_chain_enable_frontend): per-channel front end, and the conditioned IF samples of the composed path
  fe::State *d_fe = nullptr;         // [C]
  float fe_agc_start = 0.25f, fe_agc_max = 40.0f;
  int fe_agc_on = 1;
  int16_t *d_fe_if = nullptr;        // [rows][stride] of the largest composed update so far
  size_t fe_if_samples = 0;
  bool fe_composed = false;          // the last ADC update ran K4, then the int16 path

  // snapshots (msdr_chain_snapshot* / msdr_chain_restore*): host vectors their asynchronous uploads read from; `snap_ev` marks the
  // last such upload, and the next snapshot or restore waits for it before it writes them again
  std::vector<uint8_t> snap_host;
  std::vector<int16_t> snap_taps;
  fe::State snap_fe0{};
  cudaEvent_t snap_ev = nullptr;
  bool snap_pending = false;

  int variant = 0;
  uint32_t host_chunk_channels = 0, host_chunk_blocks = 0; // 0 = auto
  uint32_t spare_sms = 0;
  uint64_t launches = 0;
  std::string err;
  ChainLaunchInfo last_info{};
  std::string last_kernel = "none";
  uint64_t plan_builds = 0;
};

namespace {

int fail(msdr_chain *c, int code, const std::string &msg)
{
  if (c) c->err = msg; else g_create_error = msg;
  return code;
}
int cuda_fail(msdr_chain *c, cudaError_t e, const char *what)
{
  return fail(c, MSDR_ERR_CUDA, std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")");
}
#define CK(call)                                             \
  do {                                                       \
    cudaError_t e__ = (call);                                \
    if (e__ != cudaSuccess) return cuda_fail(chain, e__, #call); \
  } while (0)

bool range_ok(const msdr_chain *c, uint32_t ch0, uint32_t nch) { return (uint64_t)ch0 + nch <= c->C; }

// read back the events of the last timed update (blocks until it has finished) and fold it into the usage figures
int usage_resolve(msdr_chain *chain)
{
  if (!chain->usage_pending) return MSDR_OK;
  chain->usage_pending = false;
  float ms = 0.f;
  CK(cudaEventSynchronize(chain->ev1));
  CK(cudaEventElapsedTime(&ms, chain->ev0, chain->ev1));
  chain->usage_last_ms_per_block = ms / (float)std::max(1u, chain->usage_blocks);
  chain->usage_max_ms_per_block = std::max(chain->usage_max_ms_per_block, chain->usage_last_ms_per_block);
  return MSDR_OK;
}

int upload_set(msdr_chain *chain, uint32_t id)
{
  const FirSet &fs = chain->sets[id];
  int16_t *dst = chain->d_set_taps + (size_t)id * 2 * MSDR_MAX_TAPS;
  CK(cudaMemcpyAsync(dst, fs.cI.data(), fs.T * 2, cudaMemcpyHostToDevice, chain->stream));
  CK(cudaMemcpyAsync(dst + MSDR_MAX_TAPS, fs.cQ.data(), fs.T * 2, cudaMemcpyHostToDevice, chain->stream));
  CK(cudaStreamSynchronize(chain->stream)); // the taps' vectors may be reassigned as soon as this returns
  chain->meta_version++;
  return MSDR_OK;
}

// find or create a coefficient set; returns id or negative status
int intern_set(msdr_chain *chain, uint32_t T, const int16_t *cI, const int16_t *cQ)
{
  for (size_t i = 0; i < chain->sets.size(); ++i) {
    const FirSet &s = chain->sets[i];
    if (s.T == T && s.users > 0 && !memcmp(s.cI.data(), cI, T * 2) && !memcmp(s.cQ.data(), cQ, T * 2)) return (int)i;
  }
  size_t slot = chain->sets.size();
  for (size_t i = 0; i < chain->sets.size(); ++i)
    if (chain->sets[i].users == 0) { slot = i; break; }
  if (slot == chain->sets.size()) {
    if (slot >= MSDR_MAX_FIR_SETS) return fail(chain, MSDR_ERR_NOMEM, "more than MSDR_MAX_FIR_SETS distinct FIR tables in one chain");
    chain->sets.emplace_back();
  }
  FirSet &s = chain->sets[slot];
  s.T = T;
  s.cI.assign(cI, cI + T);
  s.cQ.assign(cQ, cQ + T);
  s.users = 0;
  int st = upload_set(chain, (uint32_t)slot);
  if (st != MSDR_OK) return st;
  return (int)slot;
}

int assign_set(msdr_chain *chain, uint32_t ch0, uint32_t nch, uint32_t id)
{
  for (uint32_t c = ch0; c < ch0 + nch; ++c) {
    const uint8_t old = chain->h_set[c];
    if (old == 0xFF) chain->n_uninit--; else chain->sets[old].users--;
    chain->h_set[c] = (uint8_t)id;
  }
  chain->sets[id].users += nch;
  chain->meta_version++;
  CK(cudaMemcpyAsync(chain->d_set + ch0, chain->h_set.data() + ch0, nch, cudaMemcpyHostToDevice, chain->stream));
  CK(cudaStreamSynchronize(chain->stream));
  return MSDR_OK;
}

// Before channels are bound to a new table, a table used by none but them gives its slot back (its channels stay unbound until the
// caller binds them): re-tuning a full chain (MSDR_MAX_FIR_SETS live tables) then does not fail for want of the slot it frees itself.
// A table that keeps another user keeps its slot, and nothing changes when no table is freed, so a refused table leaves the chain as
// it was.  Used by both FIR setters.  `each(f)` calls f(channel) for every channel to be re-bound, each channel once.
template <class Each> void release_sole_sets(msdr_chain *chain, Each each)
{
  uint32_t n[MSDR_MAX_FIR_SETS] = {0};
  each([&](uint32_t c) { if (chain->h_set[c] != 0xFF) n[chain->h_set[c]]++; });
  auto sole = [&](uint32_t sid) { return n[sid] && n[sid] == chain->sets[sid].users; };
  each([&](uint32_t c) {
    if (chain->h_set[c] != 0xFF && sole(chain->h_set[c])) { chain->h_set[c] = 0xFF; chain->n_uninit++; }
  });
  for (uint32_t sid = 0; sid < chain->sets.size(); ++sid)
    if (sole(sid)) chain->sets[sid].users = 0;
}

int ensure_stage(msdr_chain *chain, size_t samples)
{
  if (chain->stage_samples >= samples) return MSDR_OK;
  if (chain->d_in) cudaFree(chain->d_in);
  if (chain->d_out) cudaFree(chain->d_out);
  chain->d_in = chain->d_out = nullptr;
  chain->stage_samples = 0;
  CK(cudaMalloc(&chain->d_in, samples * sizeof(int16_t)));
  CK(cudaMalloc(&chain->d_out, samples * sizeof(int16_t)));
  chain->stage_samples = samples;
  return MSDR_OK;
}

} // namespace

extern "C" {

const char *msdr_version(void) { return "minimal-sdr_b200 0.1 (sm_100a)"; }

int msdr_chain_create(msdr_chain **out, int device, uint32_t n_channels, uint32_t max_taps, uint32_t flags)
{
  if (!out) return fail(nullptr, MSDR_ERR_ARGUMENT, "out == NULL");
  *out = nullptr;
  if (max_taps == 0) max_taps = 102;
  if (n_channels == 0 || (max_taps & 1u) || max_taps < 4 || max_taps > MSDR_MAX_TAPS)
    return fail(nullptr, MSDR_ERR_ARGUMENT, "n_channels must be > 0 and max_taps even in [4, MSDR_MAX_TAPS]");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return fail(nullptr, MSDR_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(nullptr, MSDR_ERR_ARGUMENT, "bad device index");
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return cuda_fail(nullptr, e, "cudaGetDeviceProperties");
  if (prop.major != 10) return fail(nullptr, MSDR_ERR_UNSUPPORTED, "kernels are built for sm_100a (B200) only");
  if ((e = cudaSetDevice(device)) != cudaSuccess) return cuda_fail(nullptr, e, "cudaSetDevice");

  msdr_chain *chain = new msdr_chain();
  chain->device = device;
  chain->C = n_channels;
  chain->Cpad = (n_channels + 31u) & ~31u;
  chain->max_taps = max_taps;
  chain->KPmax = kp_of_taps(max_taps);
  chain->H = hist_of_kp(chain->KPmax);
  chain->flags = flags;
  chain->h_mode.assign(n_channels, (uint8_t)MSDR_MODE_AM);
  chain->h_set.assign(n_channels, 0xFF);
  chain->n_uninit = n_channels;
  if (const char *ev = getenv("MSDR_VARIANT")) chain->variant = atoi(ev); // developer aid: default kernel variant (DESIGN.md 6)

  auto bail = [&](cudaError_t ee, const char *what) {
    int st = cuda_fail(nullptr, ee, what);
    msdr_chain_destroy(chain);
    return st;
  };
#define CKC(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return bail(e__, #call); } while (0)
  CKC(cudaStreamCreateWithFlags(&chain->own_stream, cudaStreamNonBlocking));
  CKC(cudaStreamCreateWithFlags(&chain->copy_in, cudaStreamNonBlocking));
  CKC(cudaStreamCreateWithFlags(&chain->copy_out, cudaStreamNonBlocking));
  chain->stream = chain->own_stream;
  CKC(cudaEventCreate(&chain->ev0));
  CKC(cudaEventCreate(&chain->ev1));
  CKC(cudaMalloc(&chain->d_mode, n_channels));
  CKC(cudaMalloc(&chain->d_set, n_channels));
  CKC(cudaMalloc(&chain->d_hist, (size_t)n_channels * chain->H * sizeof(int16_t)));
  CKC(cudaMalloc(&chain->d_bq, (size_t)kBqWords * chain->Cpad * sizeof(int32_t)));
  CKC(cudaMalloc(&chain->d_pll, (size_t)3 * chain->Cpad * sizeof(float)));
  CKC(cudaMemsetAsync(chain->d_pll, 0, (size_t)3 * chain->Cpad * sizeof(float), chain->own_stream));
  CKC(cudaMalloc(&chain->d_set_taps, (size_t)MSDR_MAX_FIR_SETS * 2 * MSDR_MAX_TAPS * sizeof(int16_t)));
  CKC(cudaMalloc(&chain->d_ctrl, 2 * sizeof(int)));
  CKC(cudaMemsetAsync(chain->d_mode, MSDR_MODE_AM, n_channels, chain->stream));
  CKC(cudaMemsetAsync(chain->d_set, 0, n_channels, chain->stream));
  CKC(cudaMemsetAsync(chain->d_hist, 0, (size_t)n_channels * chain->H * sizeof(int16_t), chain->stream));
  CKC(cudaMemsetAsync(chain->d_bq, 0, (size_t)kBqWords * chain->Cpad * sizeof(int32_t), chain->stream));
  CKC(cudaStreamSynchronize(chain->stream));
#undef CKC
  *out = chain;
  return MSDR_OK;
}

void msdr_chain_destroy(msdr_chain *chain)
{
  if (!chain) return;
  cudaSetDevice(chain->device);
  if (chain->stream) cudaStreamSynchronize(chain->stream);
  cudaFree(chain->d_mode); cudaFree(chain->d_set); cudaFree(chain->d_hist); cudaFree(chain->d_bq);
  for (auto &pl : chain->plans) { cudaFree(pl.d_rowmap); cudaFree(pl.d_wave_rb0); cudaFree(pl.d_rb); cudaFree(pl.d_bmat); cudaFree(pl.d_rowmap32); cudaFree(pl.d_rb32); }
  cudaFree(chain->d_tile_cnt); cudaFree(chain->d_pll);
  cudaFree(chain->d_anr_d); cudaFree(chain->d_anr_w); cudaFree(chain->d_anr_lidx); cudaFree(chain->d_anr_ngamma); cudaFree(chain->d_anr_idx);
  cudaFree(chain->pll.d_kind); cudaFree(chain->pll.d_anr_mode);
  cudaFree(chain->pll.d_rows); cudaFree(chain->pll.d_chmap); cudaFree(chain->pll.d_raw); cudaFree(chain->pll.d_I); cudaFree(chain->pll.d_Q);
  cudaFree(chain->pll.d_If); cudaFree(chain->pll.d_Qf); cudaFree(chain->pll.d_taps); cudaFree(chain->pll.d_defs);
  cudaFree(chain->d_set_taps); cudaFree(chain->d_ctrl);
  cudaFree(chain->d_in); cudaFree(chain->d_out);
  cudaFree(chain->d_fe); cudaFree(chain->d_fe_if);
  if (chain->pin_in) cudaFreeHost(chain->pin_in);
  if (chain->pin_out) cudaFreeHost(chain->pin_out);
  for (cudaEvent_t ev : chain->pipe_ev) cudaEventDestroy(ev);
  if (chain->ev0) cudaEventDestroy(chain->ev0);
  if (chain->ev1) cudaEventDestroy(chain->ev1);
  if (chain->snap_ev) cudaEventDestroy(chain->snap_ev);
  if (chain->own_stream) cudaStreamDestroy(chain->own_stream);
  if (chain->copy_in) cudaStreamDestroy(chain->copy_in);
  if (chain->copy_out) cudaStreamDestroy(chain->copy_out);
  delete chain;
}

int msdr_chain_set_stream(msdr_chain *chain, void *cuda_stream)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  CK(cudaSetDevice(chain->device));
  CK(cudaStreamSynchronize(chain->stream));
  chain->stream = cuda_stream ? (cudaStream_t)cuda_stream : chain->own_stream;
  return MSDR_OK;
}

int msdr_chain_synchronize(msdr_chain *chain)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  CK(cudaSetDevice(chain->device));
  CK(cudaStreamSynchronize(chain->stream));
  return MSDR_OK;
}

const char *msdr_last_error(const msdr_chain *chain) { return chain ? chain->err.c_str() : g_create_error.c_str(); }
uint32_t msdr_chain_channels(const msdr_chain *chain) { return chain ? chain->C : 0; }
uint64_t msdr_chain_launch_count(const msdr_chain *chain) { return chain ? chain->launches : 0; }
uint64_t msdr_chain_plan_build_count(const msdr_chain *chain) { return chain ? chain->plan_builds : 0; }
const char *msdr_chain_last_kernel(const msdr_chain *chain) { return chain ? chain->last_kernel.c_str() : ""; }
int msdr_chain_fir_taps(const msdr_chain *chain, uint32_t ch)
{
  if (!chain || ch >= chain->C) return MSDR_ERR_ARGUMENT;
  const uint8_t sid = chain->h_set[ch];
  return sid == 0xFF ? 0 : (int)chain->sets[sid].T;
}

int msdr_chain_set_mode(msdr_chain *chain, uint32_t ch0, uint32_t nch, int mode)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (!range_ok(chain, ch0, nch) || mode < 0 || mode > 4) return fail(chain, MSDR_ERR_ARGUMENT, "set_mode: bad channel range or mode");
  if (nch == 0) return MSDR_OK;
  CK(cudaSetDevice(chain->device));
  std::fill(chain->h_mode.begin() + ch0, chain->h_mode.begin() + ch0 + nch, (uint8_t)mode);
  chain->pll.dirty = true; chain->pll.epoch++;
  CK(cudaMemsetAsync(chain->d_mode + ch0, mode, nch, chain->stream));
  return MSDR_OK;
}

int msdr_chain_set_anr(msdr_chain *chain, uint32_t ch0, uint32_t nch, int anr_on)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (!range_ok(chain, ch0, nch) || anr_on < 0 || anr_on > 2) return fail(chain, MSDR_ERR_ARGUMENT, "set_anr: bad channel range or ANR_on (0 off, 1 notch, 2 noise reduction)");
  if (nch == 0) return MSDR_OK;
  CK(cudaSetDevice(chain->device));
  if (chain->h_anr.empty()) chain->h_anr.assign(chain->C, 0);
  if (anr_on && !chain->d_anr_d) { // LMS state: 512-entry delay line + 64 weights per channel, allocated on first use
    const size_t cp = chain->Cpad;
    CK(cudaStreamSynchronize(chain->stream));
    CK(cudaMalloc(&chain->d_anr_d, 512 * cp * 4)); CK(cudaMalloc(&chain->d_anr_w, 64 * cp * 4));
    CK(cudaMalloc(&chain->d_anr_lidx, cp * 4)); CK(cudaMalloc(&chain->d_anr_ngamma, cp * 4)); CK(cudaMalloc(&chain->d_anr_idx, cp * 4));
    CK(cudaMemset(chain->d_anr_d, 0, 512 * cp * 4)); CK(cudaMemset(chain->d_anr_w, 0, 64 * cp * 4)); CK(cudaMemset(chain->d_anr_idx, 0, cp * 4));
    std::vector<float> l(cp, 120.0f), g(cp, 0.001f); // Minimal-SDR.ino:715,718
    CK(cudaMemcpy(chain->d_anr_lidx, l.data(), cp * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(chain->d_anr_ngamma, g.data(), cp * 4, cudaMemcpyHostToDevice));
    CK(cudaDeviceSynchronize()); // legacy-stream copies / memsets vs the chain's non-blocking stream
  }
  for (uint32_t c = ch0; c < ch0 + nch; ++c) {
    chain->n_anr += (anr_on != 0) - (chain->h_anr[c] != 0);
    chain->h_anr[c] = (uint8_t)anr_on; // the LMS state is kept across on/off like the sketch's statics
  }
  chain->pll.dirty = true; chain->pll.epoch++;
  return MSDR_OK;
}

int msdr_chain_get_anr_state(msdr_chain *chain, uint32_t ch, msdr_anr_state *out)
{
  if (!chain || !out || ch >= chain->C) return MSDR_ERR_ARGUMENT;
  if (!chain->d_anr_d) return fail(chain, MSDR_ERR_NOT_INITIALISED, "get_anr_state: ANR was never switched on in this chain");
  CK(cudaSetDevice(chain->device));
  CK(cudaStreamSynchronize(chain->stream));
  const size_t pitch = (size_t)chain->Cpad * 4;
  CK(cudaMemcpy2D(out->d, 4, chain->d_anr_d + ch, pitch, 4, 512, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy2D(out->w, 4, chain->d_anr_w + ch, pitch, 4, 64, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(&out->lidx, chain->d_anr_lidx + ch, 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(&out->ngamma, chain->d_anr_ngamma + ch, 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(&out->in_idx, chain->d_anr_idx + ch, 4, cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

int msdr_chain_set_anr_state(msdr_chain *chain, uint32_t ch, const msdr_anr_state *in)
{
  if (!chain || !in || ch >= chain->C || in->in_idx < 0 || in->in_idx >= 512) return MSDR_ERR_ARGUMENT;
  if (!chain->d_anr_d) return fail(chain, MSDR_ERR_NOT_INITIALISED, "set_anr_state: switch ANR on (msdr_chain_set_anr) first");
  CK(cudaSetDevice(chain->device));
  CK(cudaStreamSynchronize(chain->stream));
  const size_t pitch = (size_t)chain->Cpad * 4;
  CK(cudaMemcpy2D(chain->d_anr_d + ch, pitch, in->d, 4, 4, 512, cudaMemcpyHostToDevice));
  CK(cudaMemcpy2D(chain->d_anr_w + ch, pitch, in->w, 4, 4, 64, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(chain->d_anr_lidx + ch, &in->lidx, 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(chain->d_anr_ngamma + ch, &in->ngamma, 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(chain->d_anr_idx + ch, &in->in_idx, 4, cudaMemcpyHostToDevice));
  CK(cudaDeviceSynchronize()); // legacy-stream copies vs the chain's non-blocking stream
  return MSDR_OK;
}

int msdr_fir_init_q15(msdr_chain *chain, uint32_t ch0, uint32_t nch, uint16_t numTaps, const int16_t *cI, const int16_t *cQ)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (numTaps & 1u) return fail(chain, MSDR_ERR_ARGUMENT, "arm_fir_init_q15: numTaps must be even (arm_fir_init_q15.c:93-96)");
  if (!cI || !cQ || !range_ok(chain, ch0, nch)) return fail(chain, MSDR_ERR_ARGUMENT, "fir_init: bad arguments");
  if (numTaps < 4 || numTaps > chain->max_taps) return fail(chain, MSDR_ERR_LENGTH, "fir_init: numTaps outside [4, max_taps of this chain]");
  if (nch == 0) return MSDR_OK;
  CK(cudaSetDevice(chain->device));
  release_sole_sets(chain, [&](auto &&f) { for (uint32_t c = ch0; c < ch0 + nch; ++c) f(c); });
  const int id = intern_set(chain, numTaps, cI, cQ);
  if (id < 0) return id;
  int st = assign_set(chain, ch0, nch, (uint32_t)id);
  if (st != MSDR_OK) return st;
  CK(cudaMemsetAsync(chain->d_hist + (size_t)ch0 * chain->H, 0, (size_t)nch * chain->H * sizeof(int16_t), chain->stream)); // init_FIR memset, .ino:902-903
  return MSDR_OK;
}

// ---- the same two setters for a LIST of channels: a batch of receivers whose modes interleave (mode = f(channel mod 4) in the
// benchmark layouts) is configured with one call per mode instead of one per channel
int msdr_chain_set_mode_list(msdr_chain *chain, const uint32_t *channels, uint32_t n, int mode)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if ((!channels && n) || mode < 0 || mode > 4) return fail(chain, MSDR_ERR_ARGUMENT, "set_mode_list: bad arguments");
  if (n == 0) return MSDR_OK;
  uint32_t lo = 0xFFFFFFFFu, hi = 0;
  for (uint32_t i = 0; i < n; ++i) {
    if (channels[i] >= chain->C) return fail(chain, MSDR_ERR_ARGUMENT, "set_mode_list: channel out of range");
    lo = std::min(lo, channels[i]); hi = std::max(hi, channels[i]);
  }
  CK(cudaSetDevice(chain->device));
  for (uint32_t i = 0; i < n; ++i) chain->h_mode[channels[i]] = (uint8_t)mode;
  chain->pll.dirty = true; chain->pll.epoch++;
  CK(cudaMemcpyAsync(chain->d_mode + lo, chain->h_mode.data() + lo, hi - lo + 1, cudaMemcpyHostToDevice, chain->stream));
  CK(cudaStreamSynchronize(chain->stream));
  return MSDR_OK;
}

int msdr_fir_init_q15_list(msdr_chain *chain, const uint32_t *channels, uint32_t n, uint16_t numTaps, const int16_t *cI, const int16_t *cQ)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (numTaps & 1u) return fail(chain, MSDR_ERR_ARGUMENT, "arm_fir_init_q15: numTaps must be even (arm_fir_init_q15.c:93-96)");
  if (!cI || !cQ || (!channels && n)) return fail(chain, MSDR_ERR_ARGUMENT, "fir_init_list: bad arguments");
  if (numTaps < 4 || numTaps > chain->max_taps) return fail(chain, MSDR_ERR_LENGTH, "fir_init: numTaps outside [4, max_taps of this chain]");
  if (n == 0) return MSDR_OK;
  uint32_t lo = 0xFFFFFFFFu, hi = 0;
  for (uint32_t i = 0; i < n; ++i) {
    if (channels[i] >= chain->C) return fail(chain, MSDR_ERR_ARGUMENT, "fir_init_list: channel out of range");
    lo = std::min(lo, channels[i]); hi = std::max(hi, channels[i]);
  }
  CK(cudaSetDevice(chain->device));
  {
    std::vector<uint32_t> uniq(channels, channels + n); // a channel listed twice is one user
    std::sort(uniq.begin(), uniq.end());
    uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
    release_sole_sets(chain, [&](auto &&f) { for (uint32_t c : uniq) f(c); });
  }
  const int id = intern_set(chain, numTaps, cI, cQ);
  if (id < 0) return id;
  uint32_t added = 0;
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t c = channels[i];
    const uint8_t old = chain->h_set[c];
    if (old == (uint8_t)id) continue; // listed twice, or already bound to this table
    if (old == 0xFF) chain->n_uninit--; else chain->sets[old].users--;
    chain->h_set[c] = (uint8_t)id;
    ++added;
  }
  chain->sets[id].users += added;
  chain->meta_version++;
  uint32_t *d_list = nullptr;
  CK(cudaMemcpyAsync(chain->d_set + lo, chain->h_set.data() + lo, hi - lo + 1, cudaMemcpyHostToDevice, chain->stream));
  CK(cudaMalloc(&d_list, (size_t)n * 4));
  cudaError_t e = cudaMemcpyAsync(d_list, channels, (size_t)n * 4, cudaMemcpyHostToDevice, chain->stream);
  if (e == cudaSuccess) e = launch_zero_hist_rows(chain->d_hist, chain->H, d_list, n, chain->stream); // init_FIR memset, .ino:902-903
  if (e == cudaSuccess) e = cudaStreamSynchronize(chain->stream);
  cudaFree(d_list);
  if (e != cudaSuccess) return cuda_fail(chain, e, "fir_init_list");
  chain->launches++;
  return MSDR_OK;
}

int msdr_fir_set_coefficients(msdr_chain *chain, uint32_t ch0, uint32_t nch, const int16_t *cI, const int16_t *cQ)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (!cI || !cQ || !range_ok(chain, ch0, nch) || nch == 0) return fail(chain, MSDR_ERR_ARGUMENT, "fir_set_coefficients: bad arguments");
  const uint8_t cur = chain->h_set[ch0];
  if (cur == 0xFF) return fail(chain, MSDR_ERR_NOT_INITIALISED, "fir_set_coefficients: FIR not initialised");
  for (uint32_t c = ch0; c < ch0 + nch; ++c)
    if (chain->h_set[c] != cur) return fail(chain, MSDR_ERR_ARGUMENT, "fir_set_coefficients: channels in the range do not share one table");
  CK(cudaSetDevice(chain->device));
  const uint32_t T = chain->sets[cur].T;
  if (chain->sets[cur].users == nch) { // every user is in the range: rewrite in place, like the sketch's single table
    chain->sets[cur].cI.assign(cI, cI + T);
    chain->sets[cur].cQ.assign(cQ, cQ + T);
    return upload_set(chain, cur);
  }
  const int id = intern_set(chain, T, cI, cQ);
  if (id < 0) return id;
  return assign_set(chain, ch0, nch, (uint32_t)id); // delay lines untouched
}

int msdr_biquad_set_coefficients(msdr_chain *chain, int object, uint32_t ch0, uint32_t nch, uint32_t stage, const int32_t *coef)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (object < 0 || object >= MSDR_BIQUAD_OBJECTS || !coef || !range_ok(chain, ch0, nch))
    return fail(chain, MSDR_ERR_ARGUMENT, "biquad_set_coefficients: bad arguments");
  if (stage >= 4 || nch == 0) return MSDR_OK; // filter_biquad.cpp:86: silently ignored
  CK(cudaSetDevice(chain->device));
  CK(launch_bq_setcoef(chain->d_bq, chain->Cpad, object, ch0, nch, stage, coef, chain->stream));
  chain->launches++;
  return MSDR_OK;
}

namespace {

void free_tc_plan(msdr_chain::TcPlan &pl)
{
  cudaFree(pl.d_rowmap); cudaFree(pl.d_wave_rb0); cudaFree(pl.d_rb); cudaFree(pl.d_bmat); cudaFree(pl.d_rowmap32); cudaFree(pl.d_rb32); cudaFree(pl.d_list);
  pl = msdr_chain::TcPlan{};
}

// Row plan of the tensor-core chain kernel for the channel range [ch0, ch0 + nch).  All 128 rows of a GEMM tile share the
// B operand, i.e. one tap table, and a chain wave (W groups of 32 channels, one per CTA) must get its FIR input first; so
// inside each wave the rows are sorted by table and cut into blocks of 128 (the last block of a table is padded).
// The epilogue finds each row's channel group in the row map and adds the group's rows to tile_cnt[group][unit]; a chain starts
// a unit when the count reaches the group's row count.
// want_dual: the caller would like waves of 2 x sms chains (two chain sets per SM); the plan is built with that width only if the
// window leaves room for the second set of chain slots (rings[3]), which is known before any row is sorted — so the wave width
// is chosen once and an unchanged configuration always hits the cache (256 taps beyond 148 groups used to rebuild twice per update).
// want_v6: also the group-block plan of the time-folded kernel (msdr_chain_v6.cu), if the window fits that kernel.
// list != NULL: the rows are the chain channels list[0 .. nch) (ch0 = 0) instead of the range; the plan keeps the list, and a lookup
// compares its contents.
int build_tc_plan(msdr_chain *chain, uint32_t ch0, uint32_t nch, const uint32_t *list, uint32_t sms, bool want_dual, bool want_v6,
                  const msdr_chain::TcPlan **out)
{
  for (const auto &c : chain->plans)
    if (c.version == chain->meta_version && c.ch0 == ch0 && c.nch == nch && c.sms == sms && c.want_dual == want_dual && c.want_v6 == want_v6 &&
        c.list.empty() == !list && (!list || std::equal(c.list.begin(), c.list.end(), list))) {
      *out = &c;
      return MSDR_OK;
    }
  auto chan = [&](uint32_t r) { return list ? list[r] : ch0 + r; }; // chain channel of row r
  uint32_t kp_max = 0;
  for (uint32_t r = 0; r < nch; ++r) kp_max = std::max(kp_max, kp_of_taps(chain->sets[chain->h_set[chan(r)]].T));
  const uint32_t K = tc_window_words_kp(kp_max);
  int smem_max = 0;
  CK(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, chain->device));
  uint32_t rings[4];
  if (!chain_v4_config(K, smem_max, rings)) // every window of up to MSDR_MAX_TAPS taps fits on a B200
    return fail(chain, MSDR_ERR_UNSUPPORTED, "update: the FIR window of " + std::to_string(K) + " words does not fit the chain kernel's shared memory");
  CK(cudaStreamSynchronize(chain->stream)); // a launch in flight may still read the plan that is replaced
  size_t slot = chain->plans.size();
  for (size_t i = 0; i < chain->plans.size(); ++i)
    if (chain->plans[i].version != chain->meta_version) { slot = i; break; } // stale: a table or a binding changed since
  if (slot == chain->plans.size()) {
    if (chain->plans.size() < msdr_chain::kMaxPlans) chain->plans.emplace_back();
    else slot = chain->plan_victim++ % msdr_chain::kMaxPlans;
  }
  msdr_chain::TcPlan &pl = chain->plans[slot];
  free_tc_plan(pl);
  *out = &pl;
  chain->plan_builds++;
  pl.version = chain->meta_version; pl.ch0 = ch0; pl.nch = nch; pl.sms = sms; pl.want_dual = want_dual; pl.want_v6 = want_v6;
  std::copy(rings, rings + 4, pl.rings);
  pl.K = K;
  pl.ring_v5 = chain_v5_config(K, smem_max);
  pl.ring_v5l = chain_v5l_config(K, smem_max);
  pl.slots_v6 = want_v6 ? chain_v6_config(K, smem_max) : 0u;
  pl.dual = want_dual && pl.rings[3] != 0;
  const uint32_t W = pl.W = sms * (pl.dual ? 2u : 1u);

  const uint32_t NG = (nch + kGroup - 1) / kGroup, n_sets = (uint32_t)chain->sets.size(), M = tc_tile_rows();
  std::vector<uint32_t> rowmap, wave_rb0;
  std::vector<uint4> rbs;
  std::vector<std::vector<uint32_t>> bucket(n_sets);
  wave_rb0.push_back(0);
  for (uint32_t g0 = 0; g0 < NG; g0 += W) {
    const uint32_t g1 = std::min(NG, g0 + W);
    for (auto &b : bucket) b.clear();
    for (uint32_t r = g0 * kGroup; r < std::min(nch, g1 * (uint32_t)kGroup); ++r) bucket[chain->h_set[chan(r)]].push_back(r);
    for (uint32_t sid = 0; sid < n_sets; ++sid) {
      const std::vector<uint32_t> &rows = bucket[sid];
      for (size_t i0 = 0; i0 < rows.size(); i0 += M) {
        for (size_t i = i0; i < i0 + M; ++i) rowmap.push_back(i < rows.size() ? rows[i] : 0xFFFFFFFFu);
        rbs.push_back(make_uint4(sid, 0, 0, 0));
      }
    }
    wave_rb0.push_back((uint32_t)rbs.size());
  }
  pl.n_rb = (uint32_t)rbs.size();
  pl.n_waves = (uint32_t)wave_rb0.size() - 1;
  // msdr_chain_v6.cu: the whole range sorted by table and cut into half blocks of 16 rows (the last one of a table is padded); a group
  // block is two half blocks, each with its own table.  The envelope demodulators (AM, CW: a square root per sample) cost the
  // epilogue several times what the SSB sums do and a CTA keeps its group block for the whole launch, so expensive halves are paired
  // with cheap ones: every CTA then carries the same load (with whole blocks per table the AM / CW CTAs finish 7 % after the SSB ones).
  std::vector<uint32_t> rowmap32;
  std::vector<uint4> rbs32;
  if (pl.slots_v6) {
    const uint32_t HR = chain_v6_group_rows() / 2;
    struct Half { uint32_t sid; size_t i0; bool costly; };
    std::vector<Half> costly, cheap;
    for (auto &b : bucket) b.clear();
    for (uint32_t r = 0; r < nch; ++r) bucket[chain->h_set[chan(r)]].push_back(r);
    for (uint32_t sid = 0; sid < n_sets; ++sid) {
      const std::vector<uint32_t> &rows = bucket[sid];
      for (size_t i0 = 0; i0 < rows.size(); i0 += HR) {
        bool env = false;
        for (size_t i = i0; i < std::min(rows.size(), i0 + HR); ++i) {
          const int md = chain->h_mode[chan(rows[i])];
          env |= !(md == MSDR_MODE_LSB || md == MSDR_MODE_USB);
        }
        (env ? costly : cheap).push_back(Half{sid, i0, env});
      }
    }
    std::vector<Half> order; // costly and cheap halves alternate while both last; the rest follows in table order
    size_t a = 0, b = 0;
    while (a < costly.size() || b < cheap.size()) {
      if (a < costly.size()) order.push_back(costly[a++]);
      if (b < cheap.size()) order.push_back(cheap[b++]);
    }
    for (size_t h0 = 0; h0 < order.size(); h0 += 2) {
      uint32_t sid2[2] = {order[h0].sid, order[h0].sid};
      for (size_t h = h0; h < h0 + 2; ++h) {
        if (h < order.size()) {
          const std::vector<uint32_t> &rows = bucket[order[h].sid];
          sid2[h - h0] = order[h].sid;
          for (size_t i = order[h].i0; i < order[h].i0 + HR; ++i) rowmap32.push_back(i < rows.size() ? rows[i] : 0xFFFFFFFFu);
        } else {
          for (uint32_t i = 0; i < HR; ++i) rowmap32.push_back(0xFFFFFFFFu);
        }
      }
      rbs32.push_back(make_uint4(sid2[0], sid2[1], 0, 0));
    }
    pl.n_gb = (uint32_t)rbs32.size();
  }

  // Toeplitz operands of every live table for the common window K
  const size_t bsz = (size_t)4 * tc_tile_samples() * K;
  std::vector<uint8_t> bm(bsz * n_sets, 0);
  for (uint32_t sid = 0; sid < n_sets; ++sid) {
    const FirSet &fs = chain->sets[sid];
    if (fs.users == 0 || kp_of_taps(fs.T) > kp_max) continue;
    std::vector<int> A, B, C, D;
    expand_set_int(fs.T, fs.cI.data(), fs.cQ.data(), A, B, C, D);
    tc_build_bmat(A.data(), B.data(), C.data(), D.data(), kp_of_taps(fs.T), K, bm.data() + bsz * sid);
  }
  CK(cudaMalloc(&pl.d_rowmap, rowmap.size() * 4));
  CK(cudaMalloc(&pl.d_wave_rb0, wave_rb0.size() * 4)); CK(cudaMalloc(&pl.d_rb, rbs.size() * sizeof(uint4))); CK(cudaMalloc(&pl.d_bmat, bm.size()));
  CK(cudaMemcpyAsync(pl.d_rowmap, rowmap.data(), rowmap.size() * 4, cudaMemcpyHostToDevice, chain->stream));
  CK(cudaMemcpyAsync(pl.d_wave_rb0, wave_rb0.data(), wave_rb0.size() * 4, cudaMemcpyHostToDevice, chain->stream));
  CK(cudaMemcpyAsync(pl.d_rb, rbs.data(), rbs.size() * sizeof(uint4), cudaMemcpyHostToDevice, chain->stream));
  CK(cudaMemcpyAsync(pl.d_bmat, bm.data(), bm.size(), cudaMemcpyHostToDevice, chain->stream));
  if (pl.n_gb) {
    CK(cudaMalloc(&pl.d_rowmap32, rowmap32.size() * 4)); CK(cudaMalloc(&pl.d_rb32, rbs32.size() * sizeof(uint4)));
    CK(cudaMemcpyAsync(pl.d_rowmap32, rowmap32.data(), rowmap32.size() * 4, cudaMemcpyHostToDevice, chain->stream));
    CK(cudaMemcpyAsync(pl.d_rb32, rbs32.data(), rbs32.size() * sizeof(uint4), cudaMemcpyHostToDevice, chain->stream));
  }
  if (list) {
    pl.list.assign(list, list + nch);
    CK(cudaMalloc(&pl.d_list, (size_t)nch * 4));
    CK(cudaMemcpyAsync(pl.d_list, pl.list.data(), (size_t)nch * 4, cudaMemcpyHostToDevice, chain->stream));
  }
  // On the chain's stream, NOT cudaMemcpy: a synchronous copy from pageable memory returns once the data is staged, its DMA runs in
  // the legacy stream, and the chain's stream is non-blocking - a kernel launched right after could read the plan before it had
  // arrived (seen as intermittent mismatches in the last, ragged channel chunk of msdr_chain_update).
  CK(cudaStreamSynchronize(chain->stream));
  return MSDR_OK;
}

} // namespace

namespace {

// ---- channels the fused kernel cannot finish: mode SYNCAM without MSDR_FLAG_AM_Q31 (the f32 PLL demodulator, Minimal-SDR.ino:631-688)
// and channels with the LMS notch / noise reduction switched on (.ino:702-770, between demodulation and the biquads) ---------------
// The fused kernel has no serial PLL stage and no LMS stage.  It processes these channels like any other (their result is thrown away); their
// real result is computed on dense scratch copies with the stage kernels and written over it:
//   before the fused kernel   gather  hist || in  rows and the biquad words of both objects
//   after it                  fs/4 mix -> FIR pair (zero initial state over hist || in: exact from sample 0 on, H >= taps - 1)
//                             -> demodulation switch or PLL (state per chain channel) -> LMS where it is on
//                             -> biquad object 1, 2 -> scatter audio and biquad words back
// The raw-sample history is the fused kernel's to update; it is correct for every channel.
// every chain channel that the side lane serves, ascending (one scan per configuration change, not per update)
const std::vector<uint32_t> &side_lane_channels(msdr_chain *chain)
{
  msdr_chain::PllLane &ln = chain->pll;
  if (ln.dirty) {
    const bool pll_build = !(chain->flags & MSDR_FLAG_AM_Q31);
    ln.channels.clear();
    for (uint32_t c = 0; c < chain->C; ++c)
      if ((pll_build && chain->h_mode[c] == MSDR_MODE_SYNCAM) || (chain->n_anr && chain->h_anr[c] != 0)) ln.channels.push_back(c);
    ln.dirty = false;
  }
  return ln.channels;
}

bool side_lane_in_range(msdr_chain *chain, uint32_t ch0, uint32_t nch)
{
  const std::vector<uint32_t> &ch = side_lane_channels(chain);
  const auto it = std::lower_bound(ch.begin(), ch.end(), ch0);
  return it != ch.end() && *it < ch0 + nch;
}

// list != NULL: the update's rows are the chain channels list[0 .. nch) (ch0 = 0)
int syncam_lane_prepare(msdr_chain *chain, uint32_t ch0, uint32_t nch, const uint32_t *list, const int16_t *d_in, size_t stride, uint32_t L)
{
  msdr_chain::PllLane &ln = chain->pll;
  const bool pll_build = !(chain->flags & MSDR_FLAG_AM_Q31); // Teensy 3.2 arithmetic: SYNCAM is the q31 envelope (.ino:618-620)
  // The lane's index vectors depend on the range or list, the modes / ANR switches (epoch) and the table bindings (meta_version) only: an
  // update that repeats the last one's configuration re-uses them on the device, and nothing in this function waits for the stream.
  const bool hit = ln.cached && ln.key_epoch == ln.epoch && ln.key_version == chain->meta_version && ln.key_ch0 == ch0 && ln.key_nch == nch &&
                   ln.key_list.empty() == !list && (!list || std::equal(ln.key_list.begin(), ln.key_list.end(), list));
  auto chan = [&](uint32_t r) { return list ? list[r] : ch0 + r; }; // chain channel of row r
  if (!hit) {
    ln.rows.clear();
    ln.any_pll = ln.any_anr = false;
    auto take = [&](uint32_t r) {
      const bool is_pll = pll_build && chain->h_mode[chan(r)] == MSDR_MODE_SYNCAM;
      const bool is_anr = chain->n_anr && chain->h_anr[chan(r)] != 0;
      if (!list || is_pll || is_anr) ln.rows.push_back(r);
      ln.any_pll |= is_pll; ln.any_anr |= is_anr;
    };
    const std::vector<uint32_t> &lane = side_lane_channels(chain);
    if (!list)
      for (auto it = std::lower_bound(lane.begin(), lane.end(), ch0); it != lane.end() && *it < ch0 + nch; ++it) take(*it - ch0);
    else if (!lane.empty())
      for (uint32_t r = 0; r < nch; ++r) take(r);
    std::stable_sort(ln.rows.begin(), ln.rows.end(), [&](uint32_t a, uint32_t b) { return chain->h_set[chan(a)] < chain->h_set[chan(b)]; });
    ln.cached = true; ln.key_epoch = ln.epoch; ln.key_version = chain->meta_version; ln.key_ch0 = ch0; ln.key_nch = nch;
    if (list) ln.key_list.assign(list, list + nch); else ln.key_list.clear();
  }
  if (ln.rows.empty()) return MSDR_OK;
  const uint32_t n = (uint32_t)ln.rows.size();
  const size_t Lp = (size_t)chain->H + L, samples = (size_t)n * Lp;
  bool upload = !hit;
  if (n > ln.cap_rows || samples > ln.cap_samples) {
    CK(cudaStreamSynchronize(chain->stream));
    cudaFree(ln.d_rows); cudaFree(ln.d_chmap); cudaFree(ln.d_raw); cudaFree(ln.d_I); cudaFree(ln.d_Q); cudaFree(ln.d_If); cudaFree(ln.d_Qf);
    cudaFree(ln.d_defs); cudaFree(ln.d_kind); cudaFree(ln.d_anr_mode);
    ln.d_kind = ln.d_anr_mode = nullptr;
    ln.d_rows = ln.d_chmap = nullptr; ln.d_raw = ln.d_I = ln.d_Q = ln.d_If = ln.d_Qf = nullptr; ln.d_defs = nullptr;
    ln.cap_rows = ln.cap_samples = 0;
    CK(cudaMalloc(&ln.d_rows, n * 4)); CK(cudaMalloc(&ln.d_chmap, n * 4)); CK(cudaMalloc(&ln.d_kind, n)); CK(cudaMalloc(&ln.d_anr_mode, n)); CK(cudaMalloc(&ln.d_defs, (size_t)n * 64 * 4));
    CK(cudaMalloc(&ln.d_raw, samples * 2)); CK(cudaMalloc(&ln.d_I, samples * 2)); CK(cudaMalloc(&ln.d_Q, samples * 2));
    CK(cudaMalloc(&ln.d_If, samples * 2)); CK(cudaMalloc(&ln.d_Qf, samples * 2));
    ln.cap_rows = n; ln.cap_samples = samples;
    upload = true;
  }
  if (upload) {
    ln.chmap.resize(n); ln.kind.resize(n); ln.amode.resize(n);
    for (uint32_t i = 0; i < n; ++i) {
      const uint32_t ch = chan(ln.rows[i]);
      ln.chmap[i] = ch;
      const int md = chain->h_mode[ch];
      // demodulation kind of the row (Minimal-SDR.ino:589-628); 255 = the PLL demodulator takes the row
      ln.kind[i] = (pll_build && md == MSDR_MODE_SYNCAM) ? 255 : md == MSDR_MODE_LSB ? 0 : md == MSDR_MODE_USB ? 1 : (md == MSDR_MODE_SYNCAM || !pll_build) ? 3 : 2;
      ln.amode[i] = chain->n_anr ? chain->h_anr[ch] : 0;
    }
    // pageable sources: the copies are staged before these calls return, and the vectors live in the lane until the next rebuild
    CK(cudaMemcpyAsync(ln.d_rows, ln.rows.data(), n * 4, cudaMemcpyHostToDevice, chain->stream));
    CK(cudaMemcpyAsync(ln.d_chmap, ln.chmap.data(), n * 4, cudaMemcpyHostToDevice, chain->stream));
    CK(cudaMemcpyAsync(ln.d_kind, ln.kind.data(), n, cudaMemcpyHostToDevice, chain->stream));
    CK(cudaMemcpyAsync(ln.d_anr_mode, ln.amode.data(), n, cudaMemcpyHostToDevice, chain->stream));
  }
  const uint32_t *d_chmap = list ? ln.d_chmap : nullptr;
  CK(launch_gather_rows(ln.d_rows, d_chmap, n, ch0, chain->d_hist, chain->H, d_in, stride, ln.d_raw, L, chain->stream));
  CK(launch_bq_words(0, ln.d_rows, d_chmap, n, ch0, chain->d_bq, chain->Cpad, ln.d_defs, chain->stream));
  chain->launches += 2;
  return MSDR_OK;
}

int syncam_lane_finish(msdr_chain *chain, uint32_t ch0, bool list, int16_t *d_out, size_t stride, uint32_t L)
{
  msdr_chain::PllLane &ln = chain->pll;
  if (ln.rows.empty()) return MSDR_OK;
  const uint32_t n = (uint32_t)ln.rows.size(), H = chain->H;
  const size_t Lp = (size_t)H + L;
  CK(launch_mix_fs4(ln.d_raw, ln.d_I, ln.d_Q, n, (uint32_t)Lp, Lp, chain->stream));
  for (uint32_t i0 = 0; i0 < n;) { // one FIR launch pair per run of channels sharing a tap table
    const uint8_t sid = chain->h_set[ln.chmap[i0]];
    uint32_t i1 = i0;
    while (i1 < n && chain->h_set[ln.chmap[i1]] == sid) ++i1;
    const FirSet &fs = chain->sets[sid];
    const int16_t *taps = chain->d_set_taps + (size_t)sid * 2 * MSDR_MAX_TAPS; // resident since upload_set: no copy, no wait per table
    CK(launch_fir_fast_q15(fs.T, taps, nullptr, nullptr, ln.d_I + i0 * Lp, ln.d_If + i0 * Lp, i1 - i0, (uint32_t)Lp, Lp, chain->stream));
    CK(launch_fir_fast_q15(fs.T, taps + MSDR_MAX_TAPS, nullptr, nullptr, ln.d_Q + i0 * Lp, ln.d_Qf + i0 * Lp, i1 - i0, (uint32_t)Lp, Lp, chain->stream));
    chain->launches += 2;
    i0 = i1;
  }
  int16_t *audio = ln.d_I; // reuse: [n][Lp], audio in the first L samples of every row
  CK(launch_demod_rows(ln.d_kind, ln.d_If + H, ln.d_Qf + H, Lp, audio, Lp, n, L, chain->stream));
  if (ln.any_pll) CK(launch_syncam(ln.d_If + H, ln.d_Qf + H, Lp, audio, Lp, n, L, chain->d_pll, chain->Cpad, ln.d_chmap, ln.d_kind, chain->stream));
  if (ln.any_anr)
    CK(launch_anr(audio, Lp, n, L / MSDR_BLOCK_SAMPLES, ln.d_anr_mode, ln.d_chmap, chain->d_anr_d, chain->d_anr_w, chain->d_anr_lidx, chain->d_anr_ngamma,
                  chain->d_anr_idx, chain->Cpad, chain->stream));
  CK(launch_biquad(ln.d_defs, audio, n, L, Lp, chain->stream));
  CK(launch_biquad(ln.d_defs + (size_t)n * 32, audio, n, L, Lp, chain->stream));
  CK(launch_scatter_rows(ln.d_rows, n, audio, Lp, d_out, stride, L, chain->stream));
  CK(launch_bq_words(1, ln.d_rows, list ? ln.d_chmap : nullptr, n, ch0, chain->d_bq, chain->Cpad, ln.d_defs, chain->stream));
  chain->launches += 6;
  return MSDR_OK;
}

// ---- the kernel choice -------------------------------------------------------------------------------------------------------
// variant bits the choice reads (study and parity-test knobs, include/msdr.h); the kernels read their own stage-form and ablation bits
constexpr int kV4Helper = 128;       // v4: the feed-forward helper-warp shape even beyond one channel group per SM
constexpr int kV4Classic = 256;      // v4: the classic shape (neither helper nor post warps)
constexpr int kV4OneSet = 512;       // v4: never two chain sets per SM
constexpr int kV4Post = 2048;        // v4: the post-warp shape (whole stages in the chain warps)
constexpr int kForceV5 = 4096;       // the row-block kernel for any channel count
constexpr int kNoV5 = 8192;          // never the row-block kernel
constexpr int kNoV6 = 16384;         // never the time-folded kernel
constexpr int kV5lAnyWindow = 32768; // the row-block kernel's half-tile form for any window
constexpr int kForceV6 = 65536;      // the time-folded kernel for any channel count
constexpr int kV4Study = kV4Helper | kV4Classic | kV4OneSet | kV4Post; // any of these: v4, one chain set per SM

enum Kernel { kV6, kV4, kV5, kV5l };
struct Choice {
  Kernel kernel = kV4;
  const msdr_chain::TcPlan *plan = nullptr;
  uint32_t shape = 0; // v4 (tc_ff): 0 post warps, 1 classic, 2 feed-forward helper warps, 3 two chain sets per SM
};

// The fused kernel for the range [ch0, ch0 + nch) (or the channel list[0 .. nch)) of NG channel groups on `sms` SMs, and the row plan
// it runs from.
int choose_kernel(msdr_chain *chain, uint32_t ch0, uint32_t nch, const uint32_t *list, uint32_t NG, int sms, Choice &ch)
{
  const int v = chain->variant;
  if (list) {
    // A channel list has no chain kernel v4 form (its chain warps own contiguous 32-channel groups): the time-folded kernel when its
    // group blocks fit one per SM, else the row-block kernels whatever the channel count.  The plan has one wave (sms = NG), and the
    // v6 group blocks are only asked for when the list's channel groups alone fit.
    const int v6_sms = std::max(1, sms - (int)chain->spare_sms);
    const bool want_v6 = !(v & (kNoV6 | kForceV5)) && ((v & kForceV6) || NG <= (uint32_t)v6_sms);
    const int st = build_tc_plan(chain, 0, nch, list, NG, false, want_v6, &ch.plan);
    if (st != MSDR_OK) return st;
    const msdr_chain::TcPlan &pl = *ch.plan;
    if (pl.slots_v6 && ((v & kForceV6) || pl.n_gb <= (uint32_t)v6_sms)) ch.kernel = kV6;
    else if (pl.ring_v5 || pl.ring_v5l) ch.kernel = !pl.ring_v5 || ((v & kV5lAnyWindow) && pl.ring_v5l) ? kV5l : kV5;
    else return fail(chain, MSDR_ERR_UNSUPPORTED, "update_list: the FIR window of " + std::to_string(pl.K) + " words fits no kernel with a channel-list form");
    return MSDR_OK;
  }
  // Many channels: the row-block kernel (msdr_chain_v5.cu), one CTA per 128 channels of one tap table walking through time.  It
  // needs enough row blocks to fill the SMs (kV5MinChannels: below that the pinned chains of msdr_chain_v4.cu win).
  // (more channel groups than one wave of two chain sets per SM holds - 9472 channels on 148 SMs - would make msdr_chain_v4.cu walk a
  // second, mostly empty wave: 11 264 channels 172 Gsamples/s there against ~200 here)
  const uint32_t kV5MinChannels = std::min<uint32_t>(12288u, 2u * (uint32_t)sms * (uint32_t)kGroup + 1u);
  if (((v & kForceV5) || nch >= kV5MinChannels) && !(v & (kNoV5 | kV4Study))) {
    // does the longest live table's window fit that kernel at all?  (known without sorting a single row: 256 taps do not)
    int smem_max = 0;
    CK(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, chain->device));
    uint32_t kp_live = 0;
    for (const FirSet &fs : chain->sets)
      if (fs.users) kp_live = std::max(kp_live, kp_of_taps(fs.T));
    const uint32_t K = tc_window_words_kp(kp_live);
    if (chain_v5_config(K, smem_max) || chain_v5l_config(K, smem_max)) { // a plan with ONE wave: rows sorted by table over the range
      const int st = build_tc_plan(chain, ch0, nch, nullptr, NG, false, false, &ch.plan);
      if (st != MSDR_OK) return st;
      const msdr_chain::TcPlan &pl = *ch.plan;
      if (pl.ring_v5 || pl.ring_v5l) { // else no row-block form fits this window: the kernels below
        ch.kernel = !pl.ring_v5 || ((v & kV5lAnyWindow) && pl.ring_v5l) ? kV5l : kV5; // 256 taps: the half-tile form
        return MSDR_OK;
      }
    }
  }
  // Few channels: the time-folded kernel (msdr_chain_v6.cu), one CTA per 32 same-table channels, nothing leaves the SM.  One group
  // block per SM: a second round would double the launch, and beyond that the two chain sets per SM of msdr_chain_v4.cu (then the
  // row-block kernel) are faster, so its plan is only asked for up to 8192 channels unless kForceV6 runs it anyway.
  const bool want_v6 = !(v & (kNoV6 | kV4Study)) && (nch <= 8192u || (v & kForceV6));
  // more channel groups than SMs: two chain sets per SM (waves of 2 x SMs groups)
  const bool want_dual = NG > (uint32_t)sms && !(v & kV4Study);
  const int st = build_tc_plan(chain, ch0, nch, nullptr, (uint32_t)sms, want_dual, want_v6, &ch.plan);
  if (st != MSDR_OK) return st;
  const msdr_chain::TcPlan &pl = *ch.plan;
  if (pl.slots_v6 && ((v & kForceV6) || pl.n_gb <= (uint32_t)std::max(1, sms - (int)chain->spare_sms))) {
    ch.kernel = kV6;
    return MSDR_OK;
  }
  // v4 shape: feed-forward helper warps where they fit, else post warps, else the plain classic shape; two chain sets per SM when
  // the plan has them (false when the second set of chain slots does not fit next to the window: 256 taps)
  ch.kernel = kV4;
  ch.shape = pl.rings[2] ? 2u : pl.rings[0] ? 0u : 1u;
  if ((v & kV4Post) && pl.rings[0]) ch.shape = 0u;
  if ((v & kV4Classic) && pl.rings[1]) ch.shape = 1u;
  if ((v & kV4Helper) && pl.rings[2]) ch.shape = 2u;
  if (pl.dual) ch.shape = 3u;
  return MSDR_OK;
}

// msdr_chain_last_kernel names "msdr::<ns>::chain_kernel (fused mix + ...; <form>)"; MSDR_PROF prints role r's counters i = 0..3,
// which each kernel keeps at prof[cta * 64 + r * 4 + i]
struct KernelNames {
  const char *ns, *form;   // v4: the form is the shape's name
  const char *prof, *items; // MSDR_PROF header "<prof> grid g[, n <items>], ..."
  int n_roles;
  const char *role[9];
};
const KernelNames kNames[4] = {
    {"v6", "one CTA per 32-channel group block, tile rows folded over time", "[msdr prof v6]", "group blocks", 9,
     {"convert", "mma", "epilogue", "chainA", "chainB", "load", "store", "ff1", "ff2"}},
    {"v4", nullptr, "[msdr prof]", nullptr, 8, {"convert", "mma", "epilogue", "chainA", "chainB", "load", "store", "ff2/post"}},
    {"v5", "one CTA per 128-channel row block", "[msdr prof v5]", "row blocks", 7, {"convert", "mma", "epilogue", "biquad1", "biquad2", "load", "store"}},
    {"v5l", "one CTA per 128-channel row block, half-tile hand-offs for the long window", "[msdr prof v5]", "row blocks", 7,
     {"convert", "mma", "epilogue", "biquad1", "biquad2", "load", "store"}},
};
const char *const kV4ShapeNames[4] = {"post-warp shape", "classic shape", "feed-forward helper-warp shape", "two chain sets per SM"};

// MSDR_PROF (developer aid): the mean of every role's counters over the g CTAs on stderr; the time-folded kernel adds their maxima,
// the time from kernel entry to the end of chain B and, with MSDR_PROF_CTAS, one line per CTA
int prof_dump(msdr_chain *chain, Kernel k, long long *d_prof, uint32_t g, uint32_t items)
{
  const KernelNames &kn = kNames[k];
  std::vector<long long> h((size_t)g * 64);
  CK(cudaMemcpyAsync(h.data(), d_prof, h.size() * sizeof(long long), cudaMemcpyDeviceToHost, chain->stream));
  CK(cudaStreamSynchronize(chain->stream));
  cudaFree(d_prof);
  auto at = [&](uint32_t b, int i) { return h[(size_t)b * 64 + i]; };
  if (kn.items) fprintf(stderr, "%s grid %u, %u %s, mean cycles per CTA (counter 0..3):\n", kn.prof, g, items, kn.items);
  else fprintf(stderr, "%s grid %u, mean cycles per CTA (counter 0..3):\n", kn.prof, g);
  for (int r = 0; r < kn.n_roles; ++r) {
    double m[4] = {0, 0, 0, 0}, mx[4] = {0, 0, 0, 0};
    for (uint32_t b = 0; b < g; ++b)
      for (int i = 0; i < 4; ++i) { m[i] += (double)at(b, r * 4 + i) / g; mx[i] = std::max(mx[i], (double)at(b, r * 4 + i)); }
    fprintf(stderr, "  %-9s %10.0f %10.0f %10.0f %10.0f", kn.role[r], m[0], m[1], m[2], m[3]);
    if (k == kV6) fprintf(stderr, "   max %10.0f %10.0f %10.0f %10.0f", mx[0], mx[1], mx[2], mx[3]);
    fprintf(stderr, "\n");
  }
  if (k != kV6) return MSDR_OK;
  double c = 0, n = 0, cm = 0, nm = 0;
  for (uint32_t b = 0; b < g; ++b) { c += (double)at(b, 40) / g; n += (double)at(b, 41) / g; cm = std::max(cm, (double)at(b, 40)); nm = std::max(nm, (double)at(b, 41)); }
  fprintf(stderr, "  kernel entry -> chain B done: %.0f cycles, %.0f ns (mean); max %.0f cycles, %.0f ns\n", c, n, cm, nm);
  if (getenv("MSDR_PROF_CTAS")) // per-CTA totals of chain A (wait, work) and the epilogue
    for (uint32_t b = 0; b < g; ++b)
      fprintf(stderr, "  cta %3u sm %3lld start %8lld ns total %9lld cyc  chainA %9lld %9lld %9lld  ff1 %9lld %9lld yfull %9lld  epilogue %9lld %9lld %9lld %9lld\n", b,
              at(b, 42), at(b, 43) - h[43], at(b, 40), at(b, 12), at(b, 13), at(b, 14), at(b, 28), at(b, 29), at(b, 31), at(b, 8), at(b, 9), at(b, 10), at(b, 11));
  return MSDR_OK;
}

// Refuses a channel list with a channel outside the chain or listed twice (two rows would race on one channel's state).
int check_list(msdr_chain *chain, const uint32_t *list, uint32_t n)
{
  if (chain->list_seen.size() != chain->C) { chain->list_seen.assign(chain->C, 0u); chain->list_stamp = 0; }
  if (++chain->list_stamp == 0) { std::fill(chain->list_seen.begin(), chain->list_seen.end(), 0u); chain->list_stamp = 1; }
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t c = list[i];
    if (c >= chain->C) return fail(chain, MSDR_ERR_ARGUMENT, "update_list: channel " + std::to_string(c) + " is not in the chain");
    if (chain->list_seen[c] == chain->list_stamp) return fail(chain, MSDR_ERR_ARGUMENT, "update_list: channel " + std::to_string(c) + " is listed twice");
    chain->list_seen[c] = chain->list_stamp;
  }
  return MSDR_OK;
}

// d_adc != NULL: the rows are raw ADC codes for the chain's front end.  Where the int16 input would run the row-block kernels and no
// channel of the range is on the side lane (which gathers IF samples from `d_in`), the front end runs inside their converters; in
// every other case K4 conditions the range into a scratch buffer first and the int16 path follows.  Both are bit-exact.
// list != NULL (int16 input only, ch0 = 0): row r of d_in / d_out is chain channel list[r] instead of ch0 + r.
int update_range(msdr_chain *chain, uint32_t ch0, uint32_t nch, const uint32_t *list, const int16_t *d_in, int16_t *d_out, uint32_t n_blocks,
                 size_t stride, const uint16_t *d_adc)
{
  if (n_blocks == 0 || nch == 0) return MSDR_OK;
  const uint64_t L64 = (uint64_t)n_blocks * MSDR_BLOCK_SAMPLES;
  if (list) {
    const int st = check_list(chain, list, nch);
    if (st != MSDR_OK) return st;
  } else if (!range_ok(chain, ch0, nch)) {
    return fail(chain, MSDR_ERR_ARGUMENT, "update: bad channel range");
  }
  const void *src_rows = d_adc ? static_cast<const void *>(d_adc) : static_cast<const void *>(d_in);
  if (!src_rows || !d_out || L64 > stride || L64 > 0x7FFFFF00ull) return fail(chain, MSDR_ERR_ARGUMENT, "update: bad buffers / stride < n_blocks*128");
  if (((uintptr_t)src_rows & 15u) || ((uintptr_t)d_out & 15u) || (stride & 7u))
    return fail(chain, MSDR_ERR_ARGUMENT, "update_device: buffers must be 16-byte aligned and stride a multiple of 8 samples");
  if (chain->n_uninit) return fail(chain, MSDR_ERR_NOT_INITIALISED, "update: some channels have no FIR bound (call msdr_fir_init_q15)");
  CK(cudaSetDevice(chain->device));
  chain->fe_composed = false;

  int sms = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, chain->device));
  const uint32_t NG = (nch + kGroup - 1) / kGroup;
  Choice ch;
  int st = choose_kernel(chain, ch0, nch, list, NG, sms, ch);
  if (st != MSDR_OK) return st;
  const msdr_chain::TcPlan &pl = *ch.plan;
  if (d_adc && ((ch.kernel != kV5 && ch.kernel != kV5l) || side_lane_in_range(chain, ch0, nch))) {
    // K4 over the range into the scratch rows (same stride as `d_out`), then the int16 path reads them
    const size_t need = (size_t)nch * stride;
    if (need > chain->fe_if_samples) {
      CK(cudaStreamSynchronize(chain->stream));
      cudaFree(chain->d_fe_if);
      chain->d_fe_if = nullptr; chain->fe_if_samples = 0;
      CK(cudaMalloc(&chain->d_fe_if, need * sizeof(int16_t)));
      chain->fe_if_samples = need;
    }
    CK(launch_frontend(d_adc, chain->d_fe_if, stride, nch, n_blocks, chain->d_fe + ch0, chain->fe_agc_max, chain->fe_agc_on, 0, chain->stream));
    chain->launches++;
    d_in = chain->d_fe_if;
    d_adc = nullptr;
    chain->fe_composed = true;
  }

  ChainParams p{};
  p.in = d_in; p.out = d_out; p.stride = stride;
  p.C = nch; p.ch0 = ch0; p.Cpad = chain->Cpad; p.L = (uint32_t)L64; p.H = chain->H;
  p.hist = chain->d_hist; p.bq = chain->d_bq; p.mode = chain->d_mode; p.setid = chain->d_set;
  p.am_q31 = (chain->flags & MSDR_FLAG_AM_Q31) ? 1u : 0u;
  p.spare_sms = chain->spare_sms;
  p.NG = NG; p.tc_K = pl.K; p.tc_bmat = pl.d_bmat;
  p.chlist = pl.d_list; // NULL for a range
  if (d_adc) { // fused: the converters read codes and condition them (msdr_chain_v5_common.cuh: FeRow)
    p.in = reinterpret_cast<const int16_t *>(d_adc);
    p.fe = chain->d_fe; p.agc_max = chain->fe_agc_max; p.agc_on = chain->fe_agc_on ? 1u : 0u;
  }
  switch (ch.kernel) {
  case kV5:
  case kV5l:
    p.n_items = pl.n_rb; p.tc_rowmap = pl.d_rowmap; p.tc_rb = pl.d_rb;
    p.tc_ring = ch.kernel == kV5l ? pl.ring_v5l : pl.ring_v5;
    break;
  case kV6:
    p.n_items = pl.n_gb; p.tc_rowmap = pl.d_rowmap32; p.tc_rb = pl.d_rb32;
    p.tc_ring = pl.slots_v6;
    break;
  case kV4: {
    p.NT = (p.L + chain_v4_span_samples() - 1) / chain_v4_span_samples();
    p.W = pl.W; // chains per wave
    p.n_items = pl.n_rb * p.NT;
    p.tc_rowmap = pl.d_rowmap; p.tc_rb = pl.d_rb; p.tc_wave_rb0 = pl.d_wave_rb0;
    p.tc_ring = pl.rings[ch.shape]; p.tc_ff = ch.shape;
    p.NU = p.L / chain_v4_unit_samples();
    const size_t n_cnt = (size_t)NG * p.NU;
    if (n_cnt > chain->tile_cnt_len) {
      CK(cudaStreamSynchronize(chain->stream));
      cudaFree(chain->d_tile_cnt);
      chain->d_tile_cnt = nullptr; chain->tile_cnt_len = 0;
      CK(cudaMalloc(&chain->d_tile_cnt, (n_cnt + 1024) * sizeof(int)));
      chain->tile_cnt_len = n_cnt + 1024;
    }
    CK(cudaMemsetAsync(chain->d_ctrl, 0, 2 * sizeof(int), chain->stream));
    CK(cudaMemsetAsync(chain->d_tile_cnt, 0, n_cnt * sizeof(int), chain->stream));
    p.ctrl = chain->d_ctrl; p.tile_cnt = chain->d_tile_cnt;
    break;
  }
  }

  if (chain->timed) {
    if ((st = usage_resolve(chain)) != MSDR_OK) return st; // the event pair is reused: fold the previous update in first
    CK(cudaEventRecord(chain->ev0, chain->stream));
  }
  if ((st = syncam_lane_prepare(chain, ch0, nch, list, d_in, stride, p.L)) != MSDR_OK) return st;
  static const bool prof_on = getenv("MSDR_PROF") != nullptr; // developer aid: per-role cycle counters on stderr
  long long *d_prof = nullptr;
  if (prof_on) {
    const size_t bytes = (size_t)(ch.kernel == kV4 ? p.W : (uint32_t)sms) * 64 * sizeof(long long);
    CK(cudaMalloc(&d_prof, bytes));
    CK(cudaMemsetAsync(d_prof, 0, bytes, chain->stream));
    p.prof = d_prof;
  }
  switch (ch.kernel) {
  case kV6: CK(launch_chain_v6(p, chain->stream, chain->variant, std::max(1, sms - (int)chain->spare_sms), &chain->last_info)); break;
  case kV4: CK(launch_chain_v4(p, chain->stream, chain->variant, &chain->last_info)); break;
  case kV5: CK(launch_chain_v5(p, chain->stream, chain->variant, sms, &chain->last_info)); break;
  case kV5l: CK(launch_chain_v5l(p, chain->stream, chain->variant, sms, &chain->last_info)); break;
  }
  chain->last_kernel = std::string("msdr::") + kNames[ch.kernel].ns + "::chain_kernel (fused mix + tensor-core FIR pair + demod + biquad cascade; " +
                       (ch.kernel == kV4 ? kV4ShapeNames[ch.shape] : kNames[ch.kernel].form) + ")";
  if (p.fe) chain->last_kernel += "; front end fused into the converters";
  if (list) chain->last_kernel += "; channel list";
  if ((st = syncam_lane_finish(chain, ch0, list != nullptr, d_out, stride, p.L)) != MSDR_OK) return st;
  if (chain->timed) {
    CK(cudaEventRecord(chain->ev1, chain->stream));
    chain->usage_pending = true;
    chain->usage_blocks = n_blocks;
  }
  chain->launches++;
  if (d_prof) return prof_dump(chain, ch.kernel, d_prof, ch.kernel == kV4 ? p.W : (uint32_t)chain->last_info.grid, p.n_items);
  return MSDR_OK;
}

} // namespace

int msdr_chain_update_range_device(msdr_chain *chain, uint32_t ch0, uint32_t nch, const int16_t *d_in, int16_t *d_out, uint32_t n_blocks,
                                   size_t stride)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  return update_range(chain, ch0, nch, nullptr, d_in, d_out, n_blocks, stride, nullptr);
}

int msdr_chain_update_list_device(msdr_chain *chain, const uint32_t *channels, uint32_t n, const int16_t *d_in, int16_t *d_out, uint32_t n_blocks,
                                  size_t stride)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (n && !channels) return fail(chain, MSDR_ERR_ARGUMENT, "update_list: NULL channel list");
  return update_range(chain, 0, n, channels, d_in, d_out, n_blocks, stride, nullptr);
}

int msdr_chain_update_device(msdr_chain *chain, const int16_t *d_in, int16_t *d_out, uint32_t n_blocks, size_t stride)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  return msdr_chain_update_range_device(chain, 0, chain->C, d_in, d_out, n_blocks, stride);
}

namespace {

// Host buffers: channels are cut into chunks that flow through a 3-slot device ring — H2D copy (stream copy_in),
// fused kernel (chain stream), D2H copy (stream copy_out) — so PCIe traffic in both directions overlaps the kernels.
// adc: `in` holds uint16 ADC codes (2 bytes a sample like int16 IF samples) for the chain's front end.
// list != NULL: the rows of `in` / `out` are the n chain channels list[0 .. n), cut into chunks of the list instead of the chain.
int host_pipeline(msdr_chain *chain, const int16_t *in, int16_t *out, uint32_t n_blocks, size_t stride, bool adc, const uint32_t *list = nullptr,
                  uint32_t n = 0)
{
  const uint32_t rows = list ? n : chain->C;
  const size_t L = (size_t)n_blocks * MSDR_BLOCK_SAMPLES;
  if (!in || !out || L > stride) return fail(chain, MSDR_ERR_ARGUMENT, "update: bad buffers / stride < n_blocks*128");
  if (chain->n_uninit) return fail(chain, MSDR_ERR_NOT_INITIALISED, "update: some channels have no FIR bound (call msdr_fir_init_q15)");
  CK(cudaSetDevice(chain->device));
  constexpr int kSlots = 3;
  // chunk = (channel range) x (block range).  Whole channel set and ~64 MiB per direction when it fits, so each kernel
  // still sees thousands of channels; huge chains are cut along channels as well.
  uint32_t Cc = chain->host_chunk_channels;
  uint32_t nbk = chain->host_chunk_blocks;
  if (Cc == 0) {
    // wide chains: keep the chunks deep in time (a kernel over a handful of blocks is all start-up) and cut along the channels
    // instead, ~128 MiB per direction and chunk; every distinct channel range has its own cached row plan (kMaxPlans)
    const uint32_t deep = std::min<uint32_t>(n_blocks, nbk ? nbk : 64u);
    const size_t want = ((size_t)128 << 20) / ((size_t)deep * MSDR_BLOCK_SAMPLES * 2);
    Cc = (uint32_t)std::min<size_t>(1u << 19, std::max<size_t>(8192, (want + 4095) / 4096 * 4096));
  }
  Cc = std::max<uint32_t>(kGroup, std::min(Cc, (rows + kGroup - 1) / kGroup * kGroup) / kGroup * kGroup);
  if (nbk == 0) nbk = (uint32_t)std::max<size_t>(64, ((size_t)64 << 20) / ((size_t)std::min(Cc, rows) * MSDR_BLOCK_SAMPLES * 2));
  nbk = std::min(nbk, n_blocks);
  const size_t Lc = (size_t)nbk * MSDR_BLOCK_SAMPLES; // device row pitch of a chunk
  const size_t slot_samples = (size_t)Cc * Lc;
  int st = ensure_stage(chain, slot_samples * kSlots);
  if (st != MSDR_OK) return st;
  if (chain->pipe_ev.empty()) {
    chain->pipe_ev.resize(3 * kSlots);
    for (auto &ev : chain->pipe_ev) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  }
  cudaEvent_t *ev_h2d = chain->pipe_ev.data(), *ev_k = ev_h2d + kSlots, *ev_d2h = ev_k + kSlots;
  // everything queued so far on the chain stream (setters, earlier updates) precedes this update's first kernel by stream order
  uint32_t k = 0;
  for (uint32_t c0 = 0; c0 < rows; c0 += Cc) {
    const uint32_t nc = std::min(Cc, rows - c0);
    for (uint32_t b0 = 0; b0 < n_blocks; b0 += nbk, ++k) { // time order within a channel range: state carries
      const uint32_t nb = std::min(nbk, n_blocks - b0);
      const size_t w = (size_t)nb * MSDR_BLOCK_SAMPLES * 2; // bytes per row in this chunk
      const int slot = (int)(k % kSlots);
      int16_t *din = chain->d_in + (size_t)slot * slot_samples, *dout = chain->d_out + (size_t)slot * slot_samples;
      const size_t hoff = (size_t)c0 * stride + (size_t)b0 * MSDR_BLOCK_SAMPLES;
      if (k >= (uint32_t)kSlots) { // slot reuse: its previous kernel has read d_in, its previous D2H has drained d_out
        CK(cudaStreamWaitEvent(chain->copy_in, ev_k[slot], 0));
        CK(cudaStreamWaitEvent(chain->stream, ev_d2h[slot], 0));
      }
      CK(cudaMemcpy2DAsync(din, Lc * 2, in + hoff, stride * 2, w, nc, cudaMemcpyHostToDevice, chain->copy_in));
      CK(cudaEventRecord(ev_h2d[slot], chain->copy_in));
      CK(cudaStreamWaitEvent(chain->stream, ev_h2d[slot], 0));
      st = list ? msdr_chain_update_list_device(chain, list + c0, nc, din, dout, nb, Lc)
           : adc ? msdr_chain_update_adc_range_device(chain, c0, nc, reinterpret_cast<const uint16_t *>(din), dout, nb, Lc)
                 : msdr_chain_update_range_device(chain, c0, nc, din, dout, nb, Lc);
      if (st != MSDR_OK) return st;
      CK(cudaEventRecord(ev_k[slot], chain->stream));
      CK(cudaStreamWaitEvent(chain->copy_out, ev_k[slot], 0));
      CK(cudaMemcpy2DAsync(out + hoff, stride * 2, dout, Lc * 2, w, nc, cudaMemcpyDeviceToHost, chain->copy_out));
      CK(cudaEventRecord(ev_d2h[slot], chain->copy_out));
    }
  }
  CK(cudaStreamSynchronize(chain->copy_out));
  CK(cudaStreamSynchronize(chain->stream));
  return MSDR_OK;
}

} // namespace

int msdr_chain_update(msdr_chain *chain, const int16_t *in, int16_t *out, uint32_t n_blocks, size_t stride)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (n_blocks == 0) return MSDR_OK;
  return host_pipeline(chain, in, out, n_blocks, stride, false);
}

int msdr_chain_update_list(msdr_chain *chain, const uint32_t *channels, uint32_t n, const int16_t *in, int16_t *out, uint32_t n_blocks, size_t stride)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (n && !channels) return fail(chain, MSDR_ERR_ARGUMENT, "update_list: NULL channel list");
  if (n == 0 || n_blocks == 0) return MSDR_OK;
  const int st = check_list(chain, channels, n); // the whole list before the first chunk is queued
  if (st != MSDR_OK) return st;
  return host_pipeline(chain, in, out, n_blocks, stride, false, channels, n);
}

// ---- ADC-code input: the front end of msdr_frontend.cu per chain channel, in front of the chain ------------------------------------
int msdr_chain_enable_frontend(msdr_chain *chain, float agc_start, float agc_max, int agc_on)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  CK(cudaSetDevice(chain->device));
  CK(cudaStreamSynchronize(chain->stream));
  if (!chain->d_fe) CK(cudaMalloc(&chain->d_fe, (size_t)chain->C * sizeof(fe::State)));
  chain->fe_agc_start = agc_start; chain->fe_agc_max = agc_max; chain->fe_agc_on = agc_on ? 1 : 0;
  fe::State s{};
  s.agc_idx = fe::kAgcBuf;                // .ino:451
  s.agc_val = agc_start;                  // .ino:104
  s.mult = fe::amp_multiplier(agc_start); // .ino:385
  std::vector<fe::State> h(chain->C, s);
  CK(cudaMemcpy(chain->d_fe, h.data(), h.size() * sizeof(fe::State), cudaMemcpyHostToDevice));
  CK(cudaDeviceSynchronize()); // legacy-stream copy vs the chain's non-blocking stream
  return MSDR_OK;
}

/* AudioInputAnalog::init (input_adc.cpp:59-63): x1 = first reading << 14, y1 = 0 */
int msdr_chain_frontend_preset(msdr_chain *chain, uint32_t ch0, uint32_t nch, uint16_t first_reading)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (!range_ok(chain, ch0, nch)) return fail(chain, MSDR_ERR_ARGUMENT, "frontend_preset: bad channel range");
  if (!chain->d_fe) return fail(chain, MSDR_ERR_NOT_INITIALISED, "frontend_preset: call msdr_chain_enable_frontend first");
  if (nch == 0) return MSDR_OK;
  CK(cudaSetDevice(chain->device));
  CK(cudaStreamSynchronize(chain->stream));
  std::vector<fe::State> h(nch);
  CK(cudaMemcpy(h.data(), chain->d_fe + ch0, nch * sizeof(fe::State), cudaMemcpyDeviceToHost));
  for (auto &s : h) { s.hpf_x1 = (int32_t)((uint32_t)first_reading << 14); s.hpf_y1 = 0; }
  CK(cudaMemcpy(chain->d_fe + ch0, h.data(), nch * sizeof(fe::State), cudaMemcpyHostToDevice));
  CK(cudaDeviceSynchronize());
  return MSDR_OK;
}

int msdr_chain_update_adc_range_device(msdr_chain *chain, uint32_t ch0, uint32_t nch, const uint16_t *d_adc, int16_t *d_out, uint32_t n_blocks,
                                       size_t stride)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (!chain->d_fe) return fail(chain, MSDR_ERR_NOT_INITIALISED, "update_adc: call msdr_chain_enable_frontend first");
  const int st = update_range(chain, ch0, nch, nullptr, nullptr, d_out, n_blocks, stride, d_adc);
  if (st == MSDR_OK && chain->fe_composed) chain->last_kernel = "msdr::fe::frontend_kernel (front end), then " + chain->last_kernel;
  return st;
}

int msdr_chain_update_adc_device(msdr_chain *chain, const uint16_t *d_adc, int16_t *d_out, uint32_t n_blocks, size_t stride)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  return msdr_chain_update_adc_range_device(chain, 0, chain->C, d_adc, d_out, n_blocks, stride);
}

int msdr_chain_update_adc(msdr_chain *chain, const uint16_t *adc, int16_t *out, uint32_t n_blocks, size_t stride)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (n_blocks == 0) return MSDR_OK;
  if (!chain->d_fe) return fail(chain, MSDR_ERR_NOT_INITIALISED, "update_adc: call msdr_chain_enable_frontend first");
  return host_pipeline(chain, reinterpret_cast<const int16_t *>(adc), out, n_blocks, stride, true);
}

int msdr_chain_get_frontend_state(msdr_chain *chain, uint32_t ch, msdr_frontend_state *out)
{
  if (!chain || !out || ch >= chain->C) return MSDR_ERR_ARGUMENT;
  if (!chain->d_fe) return fail(chain, MSDR_ERR_NOT_INITIALISED, "get_frontend_state: call msdr_chain_enable_frontend first");
  static_assert(sizeof(msdr_frontend_state) == sizeof(fe::State), "public and device state layouts must match");
  CK(cudaSetDevice(chain->device));
  CK(cudaStreamSynchronize(chain->stream));
  CK(cudaMemcpy(out, chain->d_fe + ch, sizeof(*out), cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

int msdr_chain_set_frontend_state(msdr_chain *chain, uint32_t ch, const msdr_frontend_state *in)
{
  if (!chain || !in || ch >= chain->C) return MSDR_ERR_ARGUMENT;
  if (!chain->d_fe) return fail(chain, MSDR_ERR_NOT_INITIALISED, "set_frontend_state: call msdr_chain_enable_frontend first");
  // agc_idx indexes the 25-entry history after a pre-decrement (Minimal-SDR.ino:481): anything outside 0..25 would be an out-of-bounds store
  if (in->agc_idx < 0 || in->agc_idx > fe::kAgcBuf) return fail(chain, MSDR_ERR_ARGUMENT, "set_frontend_state: agc_idx outside [0, 25]");
  CK(cudaSetDevice(chain->device));
  CK(cudaStreamSynchronize(chain->stream));
  CK(cudaMemcpy(chain->d_fe + ch, in, sizeof(*in), cudaMemcpyHostToDevice));
  CK(cudaDeviceSynchronize());
  return MSDR_OK;
}

int msdr_chain_last_update_ms(msdr_chain *chain, float *ms)
{
  if (!chain || !ms) return MSDR_ERR_ARGUMENT;
  if (!chain->timed) return fail(chain, MSDR_ERR_ARGUMENT, "enable with msdr_chain_set_option(chain, \"timing\", 1)");
  CK(cudaSetDevice(chain->device));
  CK(cudaEventSynchronize(chain->ev1));
  CK(cudaEventElapsedTime(ms, chain->ev0, chain->ev1));
  return MSDR_OK;
}

int msdr_chain_processor_usage(msdr_chain *chain, double sample_rate_hz, float *last_percent, float *max_percent)
{
  if (!chain || !(sample_rate_hz > 0.0)) return MSDR_ERR_ARGUMENT;
  CK(cudaSetDevice(chain->device));
  chain->timed = true; // from now on every update is bracketed by events
  int st = usage_resolve(chain);
  if (st != MSDR_OK) return st;
  const double block_ms = 1e3 * MSDR_BLOCK_SAMPLES / sample_rate_hz; // the real-time budget of one block (Minimal-SDR.ino:425)
  if (last_percent) *last_percent = (float)(100.0 * chain->usage_last_ms_per_block / block_ms);
  if (max_percent) *max_percent = (float)(100.0 * chain->usage_max_ms_per_block / block_ms);
  return MSDR_OK;
}

int msdr_chain_processor_usage_max_reset(msdr_chain *chain)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  CK(cudaSetDevice(chain->device));
  int st = usage_resolve(chain);
  chain->usage_max_ms_per_block = 0.f;
  return st;
}

int msdr_chain_set_option(msdr_chain *chain, const char *key, int value)
{
  if (!chain || !key) return MSDR_ERR_ARGUMENT;
  if (!strcmp(key, "variant")) { chain->variant = value; return MSDR_OK; }
  if (!strcmp(key, "timing")) { chain->timed = value != 0; return MSDR_OK; }
  if (!strcmp(key, "host_chunk_channels")) { chain->host_chunk_channels = (uint32_t)value; return MSDR_OK; }
  if (!strcmp(key, "host_chunk_blocks")) { chain->host_chunk_blocks = (uint32_t)value; return MSDR_OK; }
  if (!strcmp(key, "spare_sms")) { chain->spare_sms = value < 0 ? 0u : (uint32_t)value; return MSDR_OK; }
  return fail(chain, MSDR_ERR_ARGUMENT, std::string("unknown option ") + key);
}

int msdr_chain_get_state(msdr_chain *chain, uint32_t ch, msdr_channel_state *out)
{
  if (!chain || !out || ch >= chain->C) return MSDR_ERR_ARGUMENT;
  CK(cudaSetDevice(chain->device));
  CK(cudaStreamSynchronize(chain->stream));
  memset(out, 0, sizeof(*out));
  out->mode = chain->h_mode[ch];
  const uint8_t sid = chain->h_set[ch];
  out->fir_set = sid == 0xFF ? -1 : (int32_t)sid;
  out->num_taps = sid == 0xFF ? 0 : chain->sets[sid].T;
  std::vector<int16_t> h(chain->H);
  CK(cudaMemcpy(h.data(), chain->d_hist + (size_t)ch * chain->H, chain->H * sizeof(int16_t), cudaMemcpyDeviceToHost));
  if (out->num_taps) {
    const uint32_t n = out->num_taps - 1;
    memcpy(out->fir_history, h.data() + (chain->H - n), n * sizeof(int16_t));
  }
  int32_t bq[kBqWords];
  CK(cudaMemcpy2D(bq, sizeof(int32_t), chain->d_bq + ch, (size_t)chain->Cpad * sizeof(int32_t), sizeof(int32_t), kBqWords, cudaMemcpyDeviceToHost));
  memcpy(out->biquad_definition, bq, sizeof(bq));
  CK(cudaMemcpy2D(out->syncam_pll, sizeof(float), chain->d_pll + ch, (size_t)chain->Cpad * sizeof(float), sizeof(float), 3, cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

int msdr_chain_set_state(msdr_chain *chain, uint32_t ch, const msdr_channel_state *in)
{
  if (!chain || !in || ch >= chain->C) return MSDR_ERR_ARGUMENT;
  if (in->mode < 0 || in->mode > 4) return fail(chain, MSDR_ERR_ARGUMENT, "set_state: bad mode");
  const uint8_t sid = chain->h_set[ch];
  if (sid == 0xFF || chain->sets[sid].T != in->num_taps)
    return fail(chain, MSDR_ERR_ARGUMENT, "set_state: bind the FIR (msdr_fir_init_q15) with the same tap count first");
  CK(cudaSetDevice(chain->device));
  CK(cudaStreamSynchronize(chain->stream));
  int st = msdr_chain_set_mode(chain, ch, 1, in->mode);
  if (st != MSDR_OK) return st;
  std::vector<int16_t> h(chain->H, 0);
  const uint32_t n = in->num_taps - 1;
  memcpy(h.data() + (chain->H - n), in->fir_history, n * sizeof(int16_t));
  CK(cudaMemcpy(chain->d_hist + (size_t)ch * chain->H, h.data(), chain->H * sizeof(int16_t), cudaMemcpyHostToDevice));
  CK(cudaMemcpy2D(chain->d_bq + ch, (size_t)chain->Cpad * sizeof(int32_t), in->biquad_definition, sizeof(int32_t), sizeof(int32_t), kBqWords,
                  cudaMemcpyHostToDevice));
  CK(cudaMemcpy2D(chain->d_pll + ch, (size_t)chain->Cpad * sizeof(float), in->syncam_pll, sizeof(float), sizeof(float), 3, cudaMemcpyHostToDevice));
  CK(cudaDeviceSynchronize()); // legacy-stream copies vs the chain's non-blocking stream
  return MSDR_OK;
}

// ---- snapshots of channel ranges: checkpoint, resume, migration, re-sharding (format: DESIGN.md 7) ------------------------------
// Every state section is a plain (2D) copy of one SoA array of the chain; the copy engines do the work, no kernel is involved.
namespace {

constexpr char kSnapMagic[8] = {'M', 'S', 'D', 'R', 'S', 'N', 'A', 'P'};
constexpr uint32_t kSnapVersion = 1;
constexpr uint32_t kSnapHeaderBytes = 256;
constexpr uint32_t kSnapFrontend = 1u, kSnapAnr = 2u; // header `sections`
constexpr uint8_t kNoTable = 0xFF;

struct SnapTable {
  uint32_t T;
  int16_t cI[MSDR_MAX_TAPS], cQ[MSDR_MAX_TAPS];
};
static_assert(sizeof(SnapTable) == 1028, "snapshot table entry layout");

enum { kOffTables, kOffMeta, kOffHist, kOffBq, kOffPll, kOffFe, kOffAnrD, kOffAnrW, kOffAnrLidx, kOffAnrNgamma, kOffAnrIdx, kNumOff };

struct SnapHeader {
  char magic[8];
  uint32_t version, header_bytes;
  uint64_t total_bytes;
  uint32_t nch, flags, hist_len, sections;
  float agc_start, agc_max;
  int32_t agc_on;
  uint32_t n_tables, max_taps_needed, reserved;
  uint64_t off[kNumOff]; // 0 = section absent
  uint8_t zero[kSnapHeaderBytes - 64 - 8 * kNumOff];
};
static_assert(sizeof(SnapHeader) == kSnapHeaderBytes, "snapshot header is 256 bytes");

struct SnapLayout {
  uint64_t off[kNumOff], size[kNumOff];
  uint64_t total;
};

// the whole layout follows from (nch, hist_len, sections): every section starts on a 256-byte boundary, absent sections have offset 0
SnapLayout snap_layout(uint64_t nch, uint32_t hist_len, uint32_t sections)
{
  SnapLayout l{};
  uint64_t p = kSnapHeaderBytes;
  auto put = [&](int k, uint64_t bytes) { l.off[k] = p; l.size[k] = bytes; p = (p + bytes + 255u) & ~(uint64_t)255u; };
  put(kOffTables, (uint64_t)MSDR_MAX_FIR_SETS * sizeof(SnapTable));
  put(kOffMeta, 4 * nch);
  put(kOffHist, 2 * nch * hist_len);
  put(kOffBq, 4 * kBqWords * nch);
  put(kOffPll, 4 * 3 * nch);
  if (sections & kSnapFrontend) put(kOffFe, sizeof(fe::State) * nch);
  if (sections & kSnapAnr) {
    put(kOffAnrD, 4 * 512 * nch); put(kOffAnrW, 4 * 64 * nch);
    put(kOffAnrLidx, 4 * nch); put(kOffAnrNgamma, 4 * nch); put(kOffAnrIdx, 4 * nch);
  }
  l.total = p;
  return l;
}

uint32_t chain_sections(const msdr_chain *c) { return (c->d_fe ? kSnapFrontend : 0u) | (c->d_anr_d ? kSnapAnr : 0u); }

// header checks that need no device: 0, or a status with `why` set
int snap_parse_header(const void *buf, size_t bytes, SnapHeader &h, const char *&why)
{
  why = "";
  if (!buf || bytes < kSnapHeaderBytes) { why = "snapshot: buffer shorter than the 256-byte header"; return MSDR_ERR_ARGUMENT; }
  memcpy(&h, buf, sizeof(h));
  if (memcmp(h.magic, kSnapMagic, sizeof(kSnapMagic))) { why = "snapshot: bad magic"; return MSDR_ERR_ARGUMENT; }
  if (h.version != kSnapVersion) { why = "snapshot: format version not supported by this library"; return MSDR_ERR_UNSUPPORTED; }
  const uint32_t hist_max = hist_of_kp(kp_of_taps(MSDR_MAX_TAPS));
  if (h.header_bytes != kSnapHeaderBytes || h.nch == 0 || h.hist_len == 0 || h.hist_len > hist_max || (h.sections & ~(kSnapFrontend | kSnapAnr)) ||
      (h.flags & ~MSDR_FLAG_AM_Q31) || h.n_tables > MSDR_MAX_FIR_SETS || h.max_taps_needed > MSDR_MAX_TAPS) {
    why = "snapshot: header field out of range";
    return MSDR_ERR_ARGUMENT;
  }
  const SnapLayout l = snap_layout(h.nch, h.hist_len, h.sections);
  if (h.total_bytes != l.total || memcmp(h.off, l.off, sizeof(l.off))) { why = "snapshot: section offsets or total size do not match the layout"; return MSDR_ERR_ARGUMENT; }
  return MSDR_OK;
}

// before writing the staging vectors again, the uploads that read them must have run
int snap_wait(msdr_chain *chain)
{
  if (!chain->snap_ev) CK(cudaEventCreateWithFlags(&chain->snap_ev, cudaEventDisableTiming));
  if (chain->snap_pending) CK(cudaEventSynchronize(chain->snap_ev));
  chain->snap_pending = false;
  return MSDR_OK;
}

int snap_uploaded(msdr_chain *chain)
{
  CK(cudaEventRecord(chain->snap_ev, chain->stream));
  chain->snap_pending = true;
  return MSDR_OK;
}

// header, tables and meta of channels [ch0, ch0+nch) into chain->snap_host (the first l.off[kOffHist] bytes of the snapshot)
void snap_build_prefix(msdr_chain *chain, uint32_t ch0, uint32_t nch, const SnapLayout &l)
{
  std::vector<uint8_t> &b = chain->snap_host;
  b.assign(l.off[kOffHist], 0);
  SnapHeader h{};
  memcpy(h.magic, kSnapMagic, sizeof(h.magic));
  h.version = kSnapVersion; h.header_bytes = kSnapHeaderBytes; h.total_bytes = l.total;
  h.nch = nch; h.flags = chain->flags; h.hist_len = chain->H; h.sections = chain_sections(chain);
  if (chain->d_fe) { h.agc_start = chain->fe_agc_start; h.agc_max = chain->fe_agc_max; h.agc_on = chain->fe_agc_on; }
  memcpy(h.off, l.off, sizeof(h.off));
  uint8_t dense[MSDR_MAX_FIR_SETS];
  memset(dense, kNoTable, sizeof(dense));
  SnapTable *tab = reinterpret_cast<SnapTable *>(b.data() + l.off[kOffTables]);
  uint8_t *meta = b.data() + l.off[kOffMeta];
  for (uint32_t i = 0; i < nch; ++i) {
    const uint32_t c = ch0 + i;
    const uint8_t sid = chain->h_set[c];
    if (sid != kNoTable && dense[sid] == kNoTable) { // tables renumbered densely, in order of first use
      const FirSet &fs = chain->sets[sid];
      SnapTable &t = tab[h.n_tables];
      t.T = fs.T;
      memcpy(t.cI, fs.cI.data(), fs.T * 2);
      memcpy(t.cQ, fs.cQ.data(), fs.T * 2);
      h.max_taps_needed = std::max(h.max_taps_needed, fs.T);
      dense[sid] = (uint8_t)h.n_tables++;
    }
    meta[4 * i + 0] = chain->h_mode[c];
    meta[4 * i + 1] = sid == kNoTable ? kNoTable : dense[sid];
    meta[4 * i + 2] = chain->h_anr.empty() ? 0 : chain->h_anr[c];
  }
  memcpy(b.data(), &h, sizeof(h));
}

// the state sections of channels [ch0, ch0+nch) into dst (host or device), on the chain's stream
int snap_copy_state_out(msdr_chain *chain, uint32_t ch0, uint32_t nch, uint8_t *dst, const SnapLayout &l, cudaMemcpyKind kind)
{
  cudaStream_t s = chain->stream;
  const size_t cp = (size_t)chain->Cpad * 4, w = (size_t)nch * 4;
  CK(cudaMemcpyAsync(dst + l.off[kOffHist], chain->d_hist + (size_t)ch0 * chain->H, (size_t)nch * chain->H * 2, kind, s));
  CK(cudaMemcpy2DAsync(dst + l.off[kOffBq], w, chain->d_bq + ch0, cp, w, kBqWords, kind, s));
  CK(cudaMemcpy2DAsync(dst + l.off[kOffPll], w, chain->d_pll + ch0, cp, w, 3, kind, s));
  if (chain->d_fe) CK(cudaMemcpyAsync(dst + l.off[kOffFe], chain->d_fe + ch0, (size_t)nch * sizeof(fe::State), kind, s));
  for (int k = kOffHist; k < kNumOff; ++k) { // the alignment padding after each state section is zero: equal chains give equal snapshots
    if (!l.off[k]) continue;
    const uint64_t end = l.off[k] + l.size[k], pad = ((end + 255u) & ~(uint64_t)255u) - end;
    if (!pad) continue;
    if (kind == cudaMemcpyDeviceToHost) memset(dst + end, 0, pad);
    else CK(cudaMemsetAsync(dst + end, 0, pad, s));
  }
  if (chain->d_anr_d) {
    CK(cudaMemcpy2DAsync(dst + l.off[kOffAnrD], w, chain->d_anr_d + ch0, cp, w, 512, kind, s));
    CK(cudaMemcpy2DAsync(dst + l.off[kOffAnrW], w, chain->d_anr_w + ch0, cp, w, 64, kind, s));
    CK(cudaMemcpyAsync(dst + l.off[kOffAnrLidx], chain->d_anr_lidx + ch0, w, kind, s));
    CK(cudaMemcpyAsync(dst + l.off[kOffAnrNgamma], chain->d_anr_ngamma + ch0, w, kind, s));
    CK(cudaMemcpyAsync(dst + l.off[kOffAnrIdx], chain->d_anr_idx + ch0, w, kind, s));
  }
  return MSDR_OK;
}

int snap_begin(msdr_chain *chain, uint32_t ch0, uint32_t nch, size_t bytes, const void *buf, SnapLayout &l)
{
  if (!buf || nch == 0 || !range_ok(chain, ch0, nch)) return fail(chain, MSDR_ERR_ARGUMENT, "snapshot: bad buffer or channel range");
  l = snap_layout(nch, chain->H, chain_sections(chain));
  if (bytes < l.total) return fail(chain, MSDR_ERR_ARGUMENT, "snapshot: buffer smaller than msdr_chain_snapshot_bytes");
  CK(cudaSetDevice(chain->device));
  return snap_wait(chain);
}

// `count` copies of the element at host address `elem` (which outlives the copies) from d on: one upload, then doubling copies
int replicate(msdr_chain *chain, void *d, size_t elem_bytes, size_t count, const void *elem)
{
  if (!count) return MSDR_OK;
  uint8_t *p = static_cast<uint8_t *>(d);
  CK(cudaMemcpyAsync(p, elem, elem_bytes, cudaMemcpyHostToDevice, chain->stream));
  for (size_t done = 1; done < count; done *= 2)
    CK(cudaMemcpyAsync(p + done * elem_bytes, p, std::min(done, count - done) * elem_bytes, cudaMemcpyDeviceToDevice, chain->stream));
  return MSDR_OK;
}

const float kAnrLidx0 = 120.0f, kAnrNgamma0 = 0.001f; // Minimal-SDR.ino:715,718

// initial LMS state (msdr_chain_set_anr's) for channels [ch0, ch0+n)
int anr_initial(msdr_chain *chain, uint32_t ch0, uint32_t n)
{
  const size_t cp = (size_t)chain->Cpad * 4, w = (size_t)n * 4;
  CK(cudaMemset2DAsync(chain->d_anr_d + ch0, cp, 0, w, 512, chain->stream));
  CK(cudaMemset2DAsync(chain->d_anr_w + ch0, cp, 0, w, 64, chain->stream));
  CK(cudaMemsetAsync(chain->d_anr_idx + ch0, 0, w, chain->stream));
  int st = replicate(chain, chain->d_anr_lidx + ch0, 4, n, &kAnrLidx0);
  if (st == MSDR_OK) st = replicate(chain, chain->d_anr_ngamma + ch0, 4, n, &kAnrNgamma0);
  return st;
}

// Restore channels [ch0, ch0+n) from snapshot channels [first, first+n).  `pre` is a host copy of the snapshot from byte 0 through
// the meta of channel first+n-1; `src` is the whole snapshot (host or device, `kind`).  Every check runs before anything changes.
int snap_restore(msdr_chain *chain, uint32_t ch0, const uint8_t *pre, size_t pre_bytes, const uint8_t *src, size_t bytes, uint32_t first, uint32_t n,
                 cudaMemcpyKind kind)
{
  SnapHeader h;
  const char *why;
  int st = snap_parse_header(pre, pre_bytes, h, why);
  if (st != MSDR_OK) return fail(chain, st, why);
  if (bytes < h.total_bytes) return fail(chain, MSDR_ERR_ARGUMENT, "restore: buffer shorter than the snapshot's total size");
  if ((uint64_t)first + n > h.nch || !range_ok(chain, ch0, n)) return fail(chain, MSDR_ERR_ARGUMENT, "restore: channel range outside the snapshot or the chain");
  if (h.flags != chain->flags) return fail(chain, MSDR_ERR_ARGUMENT, "restore: the snapshot's chain flags (MSDR_FLAG_AM_Q31) differ from this chain's");
  const bool has_fe = h.sections & kSnapFrontend, has_anr = h.sections & kSnapAnr;
  if (has_fe && chain->d_fe && (h.agc_start != chain->fe_agc_start || h.agc_max != chain->fe_agc_max || (h.agc_on != 0) != (chain->fe_agc_on != 0)))
    return fail(chain, MSDR_ERR_ARGUMENT, "restore: the snapshot's AGC parameters differ from this chain's front end");
  if (n == 0) return MSDR_OK;
  const SnapTable *tab = reinterpret_cast<const SnapTable *>(pre + h.off[kOffTables]);
  const uint8_t *meta = pre + h.off[kOffMeta] + 4 * (size_t)first;
  uint32_t used[MSDR_MAX_FIR_SETS] = {0};
  for (uint32_t i = 0; i < n; ++i) {
    const uint8_t *m = meta + 4 * i;
    if (m[0] > MSDR_MODE_CW || (m[1] != kNoTable && m[1] >= h.n_tables) || m[2] > 2 || (m[2] && !has_anr))
      return fail(chain, MSDR_ERR_ARGUMENT, "restore: bad channel entry in the snapshot's meta section");
    if (m[1] != kNoTable) used[m[1]]++;
  }
  for (uint32_t k = 0; k < h.n_tables; ++k)
    if (used[k] && (tab[k].T < 4 || (tab[k].T & 1u) || tab[k].T > chain->max_taps))
      return fail(chain, MSDR_ERR_ARGUMENT, "restore: a table of the snapshot is longer than this chain's max_taps (or malformed)");
  if (kind == cudaMemcpyHostToDevice) { // host snapshots: the indices the kernels use are checked like the per-channel setters check them
    for (uint32_t i = 0; has_fe && i < n; ++i) {
      int32_t idx;
      memcpy(&idx, src + h.off[kOffFe] + ((size_t)first + i) * sizeof(fe::State) + offsetof(fe::State, agc_idx), 4);
      if (idx < 0 || idx > fe::kAgcBuf) return fail(chain, MSDR_ERR_ARGUMENT, "restore: front-end agc_idx outside [0, 25]");
    }
    for (uint32_t i = 0; has_anr && i < n; ++i) {
      int32_t idx;
      memcpy(&idx, src + h.off[kOffAnrIdx] + ((size_t)first + i) * 4, 4);
      if (idx < 0 || idx >= 512) return fail(chain, MSDR_ERR_ARGUMENT, "restore: ANR in_idx outside [0, 512)");
    }
  }
  // table slots: the range gives its bindings back (release_sole_sets frees tables only it used), then the snapshot's tables are
  // interned; count the live tables that would need before anything changes
  auto same = [&](const FirSet &s, const SnapTable &t) {
    return s.T == t.T && !memcmp(s.cI.data(), t.cI, t.T * 2) && !memcmp(s.cQ.data(), t.cQ, t.T * 2);
  };
  auto same_tab = [](const SnapTable &a, const SnapTable &b) { return a.T == b.T && !memcmp(a.cI, b.cI, a.T * 2) && !memcmp(a.cQ, b.cQ, a.T * 2); };
  {
    uint32_t left[MSDR_MAX_FIR_SETS] = {0};
    for (size_t s = 0; s < chain->sets.size(); ++s) left[s] = chain->sets[s].users;
    for (uint32_t c = ch0; c < ch0 + n; ++c)
      if (chain->h_set[c] != kNoTable) left[chain->h_set[c]]--;
    uint32_t live = 0;
    for (size_t s = 0; s < chain->sets.size(); ++s) live += left[s] > 0;
    for (uint32_t k = 0; k < h.n_tables; ++k) {
      if (!used[k]) continue;
      bool found = false;
      for (size_t s = 0; s < chain->sets.size() && !found; ++s) found = left[s] > 0 && same(chain->sets[s], tab[k]);
      for (uint32_t j = 0; j < k && !found; ++j) found = used[j] && same_tab(tab[j], tab[k]);
      live += !found;
    }
    if (live > MSDR_MAX_FIR_SETS) return fail(chain, MSDR_ERR_NOMEM, "restore: more than MSDR_MAX_FIR_SETS distinct FIR tables in one chain");
  }

  // ---- from here on the chain changes
  CK(cudaSetDevice(chain->device));
  if ((st = snap_wait(chain)) != MSDR_OK) return st;
  release_sole_sets(chain, [&](auto &&f) { for (uint32_t c = ch0; c < ch0 + n; ++c) f(c); });
  for (uint32_t c = ch0; c < ch0 + n; ++c)
    if (chain->h_set[c] != kNoTable) { chain->sets[chain->h_set[c]].users--; chain->h_set[c] = kNoTable; chain->n_uninit++; }
  uint8_t map[MSDR_MAX_FIR_SETS];
  chain->snap_taps.resize((size_t)MSDR_MAX_FIR_SETS * 2 * MSDR_MAX_TAPS);
  for (uint32_t k = 0; k < h.n_tables; ++k) {
    if (!used[k]) continue;
    const SnapTable &t = tab[k];
    size_t slot = chain->sets.size();
    for (size_t s = 0; s < chain->sets.size() && slot == chain->sets.size(); ++s)
      if (chain->sets[s].users > 0 && same(chain->sets[s], t)) slot = s;
    if (slot == chain->sets.size()) { // a new table: first free slot, uploaded from the staging vectors
      for (size_t s = 0; s < chain->sets.size(); ++s)
        if (chain->sets[s].users == 0) { slot = s; break; }
      if (slot == chain->sets.size()) chain->sets.emplace_back();
      FirSet &fs = chain->sets[slot];
      fs.T = t.T;
      fs.cI.assign(t.cI, t.cI + t.T);
      fs.cQ.assign(t.cQ, t.cQ + t.T);
      int16_t *tp = chain->snap_taps.data() + slot * 2 * MSDR_MAX_TAPS;
      std::copy(t.cI, t.cI + t.T, tp);
      std::copy(t.cQ, t.cQ + t.T, tp + MSDR_MAX_TAPS);
      CK(cudaMemcpyAsync(chain->d_set_taps + slot * 2 * MSDR_MAX_TAPS, tp, 2 * MSDR_MAX_TAPS * 2, cudaMemcpyHostToDevice, chain->stream));
    }
    chain->sets[slot].users += used[k]; // counted at once: an identical later entry finds this slot
    map[k] = (uint8_t)slot;
  }
  // host mirrors, then the device copies of mode and table id
  if (has_anr && chain->h_anr.empty()) chain->h_anr.assign(chain->C, 0);
  std::vector<uint8_t> &hb = chain->snap_host;
  hb.resize(2 * (size_t)n);
  for (uint32_t i = 0; i < n; ++i) {
    const uint8_t *m = meta + 4 * i;
    const uint32_t c = ch0 + i;
    chain->h_mode[c] = m[0];
    if (m[1] != kNoTable) { chain->h_set[c] = map[m[1]]; chain->n_uninit--; }
    if (!chain->h_anr.empty()) { chain->n_anr += (m[2] != 0) - (chain->h_anr[c] != 0); chain->h_anr[c] = m[2]; }
    hb[i] = chain->h_mode[c];
    hb[n + i] = chain->h_set[c];
  }
  chain->meta_version++;
  chain->pll.dirty = true; chain->pll.epoch++;
  cudaStream_t s = chain->stream;
  CK(cudaMemcpyAsync(chain->d_mode + ch0, hb.data(), n, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(chain->d_set + ch0, hb.data() + n, n, cudaMemcpyHostToDevice, s));

  // state sections: one (2D) copy each; the snapshot side has pitch nch, the chain side Cpad
  const size_t H = chain->H, Hs = h.hist_len, m = std::min(H, Hs), cp = (size_t)chain->Cpad * 4, sp = (size_t)h.nch * 4, w = (size_t)n * 4;
  if (Hs == H) {
    CK(cudaMemcpyAsync(chain->d_hist + (size_t)ch0 * H, src + h.off[kOffHist] + (size_t)first * Hs * 2, (size_t)n * H * 2, kind, s));
  } else { // the last min(H, hist_len) samples of each row go to the end of the row, the front is zero (msdr_chain_set_state)
    CK(cudaMemcpy2DAsync(chain->d_hist + (size_t)ch0 * H + (H - m), H * 2, src + h.off[kOffHist] + ((size_t)first * Hs + (Hs - m)) * 2, Hs * 2, m * 2, n,
                         kind, s));
    if (H > m) CK(cudaMemset2DAsync(chain->d_hist + (size_t)ch0 * H, H * 2, 0, (H - m) * 2, n, s));
  }
  CK(cudaMemcpy2DAsync(chain->d_bq + ch0, cp, src + h.off[kOffBq] + 4 * (size_t)first, sp, w, kBqWords, kind, s));
  CK(cudaMemcpy2DAsync(chain->d_pll + ch0, cp, src + h.off[kOffPll] + 4 * (size_t)first, sp, w, 3, kind, s));

  if (has_fe || chain->d_fe) {
    const bool fe_new = !chain->d_fe;
    if (fe_new) { // the snapshot brings a front end: enable it with its parameters, every other channel starts as enable_frontend starts it
      CK(cudaMalloc(&chain->d_fe, (size_t)chain->C * sizeof(fe::State)));
      chain->fe_agc_start = h.agc_start; chain->fe_agc_max = h.agc_max; chain->fe_agc_on = h.agc_on ? 1 : 0;
    }
    fe::State &s0 = chain->snap_fe0;
    s0 = fe::State{};
    s0.agc_idx = fe::kAgcBuf;                          // .ino:451
    s0.agc_val = chain->fe_agc_start;                  // .ino:104
    s0.mult = fe::amp_multiplier(chain->fe_agc_start); // .ino:385
    if (fe_new) st = replicate(chain, chain->d_fe, sizeof(fe::State), chain->C, &s0);
    if (st == MSDR_OK && has_fe)
      CK(cudaMemcpyAsync(chain->d_fe + ch0, src + h.off[kOffFe] + (size_t)first * sizeof(fe::State), (size_t)n * sizeof(fe::State), kind, s));
    else if (st == MSDR_OK)
      st = replicate(chain, chain->d_fe + ch0, sizeof(fe::State), n, &s0); // the snapshot has no front end: restored channels start fresh
    if (st != MSDR_OK) return st;
  }

  if (has_anr && !chain->d_anr_d) { // LMS arrays on first need, as msdr_chain_set_anr allocates them; every channel starts at the initial state
    const size_t cpb = (size_t)chain->Cpad * 4;
    CK(cudaMalloc(&chain->d_anr_d, 512 * cpb)); CK(cudaMalloc(&chain->d_anr_w, 64 * cpb));
    CK(cudaMalloc(&chain->d_anr_lidx, cpb)); CK(cudaMalloc(&chain->d_anr_ngamma, cpb)); CK(cudaMalloc(&chain->d_anr_idx, cpb));
    if ((st = anr_initial(chain, 0, chain->Cpad)) != MSDR_OK) return st;
  }
  if (has_anr) {
    CK(cudaMemcpy2DAsync(chain->d_anr_d + ch0, cp, src + h.off[kOffAnrD] + 4 * (size_t)first, sp, w, 512, kind, s));
    CK(cudaMemcpy2DAsync(chain->d_anr_w + ch0, cp, src + h.off[kOffAnrW] + 4 * (size_t)first, sp, w, 64, kind, s));
    CK(cudaMemcpyAsync(chain->d_anr_lidx + ch0, src + h.off[kOffAnrLidx] + 4 * (size_t)first, w, kind, s));
    CK(cudaMemcpyAsync(chain->d_anr_ngamma + ch0, src + h.off[kOffAnrNgamma] + 4 * (size_t)first, w, kind, s));
    CK(cudaMemcpyAsync(chain->d_anr_idx + ch0, src + h.off[kOffAnrIdx] + 4 * (size_t)first, w, kind, s));
  } else if (chain->d_anr_d) {
    if ((st = anr_initial(chain, ch0, n)) != MSDR_OK) return st;
  }
  return snap_uploaded(chain);
}

} // namespace

size_t msdr_chain_snapshot_bytes(const msdr_chain *chain, uint32_t nch)
{
  if (!chain || nch == 0) return 0;
  return snap_layout(nch, chain->H, chain_sections(chain)).total;
}

int msdr_chain_snapshot(msdr_chain *chain, uint32_t ch0, uint32_t nch, void *buf, size_t bytes)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  SnapLayout l;
  int st = snap_begin(chain, ch0, nch, bytes, buf, l);
  if (st != MSDR_OK) return st;
  snap_build_prefix(chain, ch0, nch, l);
  memcpy(buf, chain->snap_host.data(), chain->snap_host.size());
  if ((st = snap_copy_state_out(chain, ch0, nch, static_cast<uint8_t *>(buf), l, cudaMemcpyDeviceToHost)) != MSDR_OK) return st;
  CK(cudaStreamSynchronize(chain->stream));
  return MSDR_OK;
}

int msdr_chain_snapshot_device(msdr_chain *chain, uint32_t ch0, uint32_t nch, void *d_buf, size_t bytes)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  SnapLayout l;
  int st = snap_begin(chain, ch0, nch, bytes, d_buf, l);
  if (st != MSDR_OK) return st;
  snap_build_prefix(chain, ch0, nch, l);
  uint8_t *d = static_cast<uint8_t *>(d_buf);
  CK(cudaMemcpyAsync(d, chain->snap_host.data(), chain->snap_host.size(), cudaMemcpyHostToDevice, chain->stream));
  if ((st = snap_copy_state_out(chain, ch0, nch, d, l, cudaMemcpyDeviceToDevice)) != MSDR_OK) return st;
  return snap_uploaded(chain);
}

int msdr_chain_restore(msdr_chain *chain, uint32_t ch0, const void *buf, size_t bytes, uint32_t first, uint32_t n)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (!buf) return fail(chain, MSDR_ERR_ARGUMENT, "restore: buf == NULL");
  const uint8_t *b = static_cast<const uint8_t *>(buf);
  // the meta of snapshot channels [first, first+n) must lie inside `bytes` before the header is trusted with anything
  const uint64_t need = snap_layout(0, 8, 0).off[kOffMeta] + 4 * ((uint64_t)first + n);
  int st = snap_restore(chain, ch0, b, (size_t)std::min<uint64_t>(bytes, need), b, bytes, first, n, cudaMemcpyHostToDevice);
  if (st != MSDR_OK) return st;
  CK(cudaStreamSynchronize(chain->stream)); // the caller may free the blob on return
  return MSDR_OK;
}

int msdr_chain_restore_device(msdr_chain *chain, uint32_t ch0, const void *d_buf, size_t bytes, uint32_t first, uint32_t n)
{
  if (!chain) return MSDR_ERR_ARGUMENT;
  if (!d_buf) return fail(chain, MSDR_ERR_ARGUMENT, "restore_device: d_buf == NULL");
  // header, tables and the meta of the restored channels: one small synchronous read (stream-ordered after the chain's earlier work)
  const uint64_t need = snap_layout(0, 8, 0).off[kOffMeta] + 4 * ((uint64_t)first + n);
  const size_t pre = (size_t)std::min<uint64_t>(bytes, need);
  if (pre < kSnapHeaderBytes) return fail(chain, MSDR_ERR_ARGUMENT, "snapshot: buffer shorter than the 256-byte header");
  CK(cudaSetDevice(chain->device));
  std::vector<uint8_t> h(pre);
  CK(cudaMemcpyAsync(h.data(), d_buf, pre, cudaMemcpyDeviceToHost, chain->stream));
  CK(cudaStreamSynchronize(chain->stream));
  return snap_restore(chain, ch0, h.data(), pre, static_cast<const uint8_t *>(d_buf), bytes, first, n, cudaMemcpyDeviceToDevice);
}

int msdr_snapshot_info(const void *header, size_t bytes, uint32_t *n_channels, uint32_t *max_taps_needed, uint32_t *flags)
{
  SnapHeader h;
  const char *why;
  const int st = snap_parse_header(header, bytes, h, why);
  if (st != MSDR_OK) return st;
  if (n_channels) *n_channels = h.nch;
  if (max_taps_needed) *max_taps_needed = h.max_taps_needed;
  if (flags) *flags = h.flags | (h.sections & kSnapFrontend ? MSDR_SNAPSHOT_FRONTEND : 0u) | (h.sections & kSnapAnr ? MSDR_SNAPSHOT_ANR : 0u);
  return MSDR_OK;
}

void *msdr_host_alloc(size_t bytes)
{
  void *p = nullptr;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
  return p;
}
void msdr_host_free(void *p) { if (p) cudaFreeHost(p); }

} // extern "C"

// ---- stage-level operators ----------------------------------------------------------------------------

namespace {
struct DevBuf {
  void *p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
  cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 16); }
  template <class T> T *as() { return static_cast<T *>(p); }
};
int op_fail(cudaError_t e, const char *what) { g_create_error = std::string(what) + ": " + cudaGetErrorString(e); return MSDR_ERR_CUDA; }
#define OPCK(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return op_fail(e__, #call); } while (0)
int op_begin(int device)
{
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { g_create_error = "no CUDA device: this library has no CPU fallback"; return MSDR_ERR_CUDA; }
  if (device < 0 || device >= ndev) return MSDR_ERR_ARGUMENT;
  OPCK(cudaSetDevice(device));
  return MSDR_OK;
}
} // namespace

extern "C" {

int msdr_op_mix_fs4(int device, const int16_t *in, int16_t *outI, int16_t *outQ, uint32_t rows, uint32_t n, size_t stride)
{
  if (!in || !outI || !outQ || (n & 3u) || n > stride) return MSDR_ERR_ARGUMENT;
  int st = op_begin(device); if (st) return st;
  DevBuf a, b, c;
  const size_t bytes = (size_t)rows * n * 2;
  OPCK(a.alloc(bytes)); OPCK(b.alloc(bytes)); OPCK(c.alloc(bytes));
  OPCK(cudaMemcpy2D(a.p, (size_t)n * 2, in, stride * 2, (size_t)n * 2, rows, cudaMemcpyHostToDevice));
  OPCK(launch_mix_fs4(a.as<int16_t>(), b.as<int16_t>(), c.as<int16_t>(), rows, n, n, nullptr));
  OPCK(cudaMemcpy2D(outI, stride * 2, b.p, (size_t)n * 2, (size_t)n * 2, rows, cudaMemcpyDeviceToHost));
  OPCK(cudaMemcpy2D(outQ, stride * 2, c.p, (size_t)n * 2, (size_t)n * 2, rows, cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

int msdr_op_fir_fast_q15(int device, uint16_t numTaps, const int16_t *coeffs, int16_t *history, const int16_t *in, int16_t *out, uint32_t rows,
                         uint32_t n, size_t stride)
{
  if (numTaps & 1u) return MSDR_ERR_ARGUMENT; // arm_fir_init_q15.c:93-96
  if (!coeffs || !in || !out || numTaps < 2 || n > stride) return MSDR_ERR_ARGUMENT;
  int st = op_begin(device); if (st) return st;
  DevBuf dc, dh, dh2, di, dout;
  const size_t bytes = (size_t)rows * n * 2, hbytes = (size_t)rows * (numTaps - 1) * 2;
  OPCK(dc.alloc(numTaps * 2)); OPCK(di.alloc(bytes)); OPCK(dout.alloc(bytes));
  OPCK(cudaMemcpy(dc.p, coeffs, numTaps * 2, cudaMemcpyHostToDevice));
  if (history) { OPCK(dh.alloc(hbytes)); OPCK(dh2.alloc(hbytes)); OPCK(cudaMemcpy(dh.p, history, hbytes, cudaMemcpyHostToDevice)); }
  OPCK(cudaMemcpy2D(di.p, (size_t)n * 2, in, stride * 2, (size_t)n * 2, rows, cudaMemcpyHostToDevice));
  OPCK(launch_fir_fast_q15(numTaps, dc.as<int16_t>(), history ? dh.as<int16_t>() : nullptr, history ? dh2.as<int16_t>() : nullptr, di.as<int16_t>(),
                           dout.as<int16_t>(), rows, n, n, nullptr));
  OPCK(cudaMemcpy2D(out, stride * 2, dout.p, (size_t)n * 2, (size_t)n * 2, rows, cudaMemcpyDeviceToHost));
  if (history) OPCK(cudaMemcpy(history, dh2.p, hbytes, cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

int msdr_op_demod(int device, int kind, const int16_t *I, const int16_t *Q, int16_t *out, uint32_t rows, uint32_t n, size_t stride)
{
  if (!I || !Q || !out || kind < 0 || kind > 3 || n > stride) return MSDR_ERR_ARGUMENT;
  int st = op_begin(device); if (st) return st;
  DevBuf a, b, c;
  const size_t bytes = (size_t)rows * n * 2;
  OPCK(a.alloc(bytes)); OPCK(b.alloc(bytes)); OPCK(c.alloc(bytes));
  OPCK(cudaMemcpy2D(a.p, (size_t)n * 2, I, stride * 2, (size_t)n * 2, rows, cudaMemcpyHostToDevice));
  OPCK(cudaMemcpy2D(b.p, (size_t)n * 2, Q, stride * 2, (size_t)n * 2, rows, cudaMemcpyHostToDevice));
  OPCK(launch_demod(kind, a.as<int16_t>(), b.as<int16_t>(), c.as<int16_t>(), rows, n, n, nullptr));
  OPCK(cudaMemcpy2D(out, stride * 2, c.p, (size_t)n * 2, (size_t)n * 2, rows, cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

int msdr_op_dac_codes(int device, const int16_t *in, uint16_t *out, uint32_t rows, uint32_t n, size_t stride)
{
  if (!in || !out || n > stride) return MSDR_ERR_ARGUMENT;
  int st = op_begin(device); if (st) return st;
  DevBuf a, b;
  OPCK(a.alloc((size_t)rows * n * 2)); OPCK(b.alloc((size_t)rows * n * 2));
  OPCK(cudaMemcpy2D(a.p, (size_t)n * 2, in, stride * 2, (size_t)n * 2, rows, cudaMemcpyHostToDevice));
  OPCK(launch_dac_codes(a.as<int16_t>(), b.as<uint16_t>(), rows, n, n, nullptr));
  OPCK(cudaMemcpy2D(out, stride * 2, b.p, (size_t)n * 2, (size_t)n * 2, rows, cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

int msdr_op_amplifier(int device, const int32_t *multipliers, int16_t *data, uint32_t rows, uint32_t n, size_t stride)
{
  if (!multipliers || !data || n > stride) return MSDR_ERR_ARGUMENT;
  int st = op_begin(device); if (st) return st;
  DevBuf d, m;
  OPCK(d.alloc((size_t)rows * n * 2)); OPCK(m.alloc((size_t)rows * 4));
  OPCK(cudaMemcpy2D(d.p, (size_t)n * 2, data, stride * 2, (size_t)n * 2, rows, cudaMemcpyHostToDevice));
  OPCK(cudaMemcpy(m.p, multipliers, (size_t)rows * 4, cudaMemcpyHostToDevice));
  OPCK(launch_amplifier(m.as<int32_t>(), d.as<int16_t>(), rows, n, n, nullptr));
  OPCK(cudaMemcpy2D(data, stride * 2, d.p, (size_t)n * 2, (size_t)n * 2, rows, cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

int msdr_op_biquad(int device, int32_t *definition, int16_t *data, uint32_t rows, uint32_t n, size_t stride)
{
  if (!definition || !data || (n & 1u) || n > stride) return MSDR_ERR_ARGUMENT;
  int st = op_begin(device); if (st) return st;
  DevBuf dd, dx;
  const size_t n2 = (n + 7u) & ~7u; // keep rows 16-byte aligned
  OPCK(dd.alloc((size_t)rows * 32 * 4)); OPCK(dx.alloc((size_t)rows * n2 * 2));
  OPCK(cudaMemcpy(dd.p, definition, (size_t)rows * 32 * 4, cudaMemcpyHostToDevice));
  OPCK(cudaMemcpy2D(dx.p, n2 * 2, data, stride * 2, (size_t)n * 2, rows, cudaMemcpyHostToDevice));
  OPCK(launch_biquad(dd.as<int32_t>(), dx.as<int16_t>(), rows, n, n2, nullptr));
  OPCK(cudaMemcpy2D(data, stride * 2, dx.p, n2 * 2, (size_t)n * 2, rows, cudaMemcpyDeviceToHost));
  OPCK(cudaMemcpy(definition, dd.p, (size_t)rows * 32 * 4, cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

int msdr_op_freq_conv(int device, int dir, int pass, int16_t *I, int16_t *Q, const int16_t *oscI, const int16_t *oscQ, uint32_t rows, uint32_t n,
                      size_t stride)
{
  if (!I || !Q || !oscI || !oscQ || n > stride) return MSDR_ERR_ARGUMENT;
  int st = op_begin(device); if (st) return st;
  if (!pass) return MSDR_OK; // freq_conv.cpp:49-56: inputs forwarded unchanged
  DevBuf a, b, oi, oq;
  const size_t bytes = (size_t)rows * n * 2;
  OPCK(a.alloc(bytes)); OPCK(b.alloc(bytes)); OPCK(oi.alloc((size_t)n * 2)); OPCK(oq.alloc((size_t)n * 2));
  OPCK(cudaMemcpy2D(a.p, (size_t)n * 2, I, stride * 2, (size_t)n * 2, rows, cudaMemcpyHostToDevice));
  OPCK(cudaMemcpy2D(b.p, (size_t)n * 2, Q, stride * 2, (size_t)n * 2, rows, cudaMemcpyHostToDevice));
  OPCK(cudaMemcpy(oi.p, oscI, (size_t)n * 2, cudaMemcpyHostToDevice));
  OPCK(cudaMemcpy(oq.p, oscQ, (size_t)n * 2, cudaMemcpyHostToDevice));
  OPCK(launch_freq_conv(dir, a.as<int16_t>(), b.as<int16_t>(), oi.as<int16_t>(), oq.as<int16_t>(), rows, n, n, nullptr));
  OPCK(cudaMemcpy2D(I, stride * 2, a.p, (size_t)n * 2, (size_t)n * 2, rows, cudaMemcpyDeviceToHost));
  OPCK(cudaMemcpy2D(Q, stride * 2, b.p, (size_t)n * 2, (size_t)n * 2, rows, cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

// K3 study operator: mix + FIR pair + demod on the tensor cores (no biquad).  kinds: per-row demod kind or NULL (kind0 for all).
int msdr_op_fir_demod_tc(int device, uint16_t numTaps, const int16_t *cI, const int16_t *cQ, const uint8_t *kinds, int kind0, const int16_t *in,
                         int16_t *out, uint32_t rows, uint32_t n, size_t stride)
{
  if ((numTaps & 1u) || numTaps < 4 || numTaps > MSDR_MAX_TAPS) return MSDR_ERR_ARGUMENT;
  if (!cI || !cQ || !in || !out || n > stride || (n % tc_tile_samples()) || kind0 < 0 || kind0 > 3) return MSDR_ERR_ARGUMENT;
  int st = op_begin(device); if (st) return st;
  const uint32_t K = tc_window_words(numTaps), KP = kp_of_taps(numTaps);
  const uint32_t pad = 2 * (K - tc_tile_samples() / 2); // samples of (zero) history in front of every row
  const size_t dstride = (size_t)pad + n;
  std::vector<int> A, B, C, D;
  expand_set_int(numTaps, cI, cQ, A, B, C, D);
  std::vector<uint8_t> bm((size_t)4 * tc_tile_samples() * K);
  tc_build_bmat(A.data(), B.data(), C.data(), D.data(), KP, K, bm.data());
  std::vector<uint8_t> hk(rows, (uint8_t)kind0), hs(rows, 0);
  if (kinds) memcpy(hk.data(), kinds, rows);
  DevBuf din, dout, dbm, dk, ds, dctr;
  OPCK(dctr.alloc(sizeof(int)));
  OPCK(din.alloc(rows * dstride * 2)); OPCK(dout.alloc((size_t)rows * n * 2)); OPCK(dbm.alloc(bm.size())); OPCK(dk.alloc(rows)); OPCK(ds.alloc(rows));
  OPCK(cudaMemset(din.p, 0, rows * dstride * 2));
  OPCK(cudaMemcpy2D(din.as<int16_t>() + pad, dstride * 2, in, stride * 2, (size_t)n * 2, rows, cudaMemcpyHostToDevice));
  OPCK(cudaMemcpy(dbm.p, bm.data(), bm.size(), cudaMemcpyHostToDevice));
  OPCK(cudaMemcpy(dk.p, hk.data(), rows, cudaMemcpyHostToDevice));
  OPCK(cudaMemcpy(ds.p, hs.data(), rows, cudaMemcpyHostToDevice));
  OPCK(launch_fir_demod_tc(din.as<int16_t>() + pad, dstride, dout.as<int16_t>(), n, rows, n, K, dbm.as<uint8_t>(), ds.as<uint8_t>(), dk.as<uint8_t>(), dctr.as<int>(), nullptr));
  OPCK(cudaDeviceSynchronize());
  OPCK(cudaMemcpy2D(out, stride * 2, dout.p, (size_t)n * 2, (size_t)n * 2, rows, cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

// Study check: the branch-free float square root of the tensor-core epilogue equals __fsqrt_rn for every envelope argument.
int msdr_study_sqrt_check(int device, uint64_t *mismatches)
{
  if (!mismatches) return MSDR_ERR_ARGUMENT;
  int st = op_begin(device); if (st) return st;
  DevBuf d;
  OPCK(d.alloc(8));
  OPCK(cudaMemset(d.p, 0, 8));
  OPCK(launch_sqrt_check(d.as<unsigned long long>(), nullptr));
  OPCK(cudaDeviceSynchronize());
  unsigned long long h = 0;
  OPCK(cudaMemcpy(&h, d.p, 8, cudaMemcpyDeviceToHost));
  *mismatches = h;
  return MSDR_OK;
}

// K3 study timing: device-resident pseudo-random input, `iters` launches timed with CUDA events; returns ms per launch.
int msdr_study_fir_demod_tc_time(int device, uint16_t numTaps, uint32_t rows, uint32_t n, int kind0, int iters, float *ms_per_iter)
{
  if ((numTaps & 1u) || numTaps < 4 || numTaps > MSDR_MAX_TAPS || !ms_per_iter || (n % tc_tile_samples()) || iters < 1) return MSDR_ERR_ARGUMENT;
  int st = op_begin(device); if (st) return st;
  const uint32_t K = tc_window_words(numTaps), KP = kp_of_taps(numTaps);
  const uint32_t pad = 2 * (K - tc_tile_samples() / 2);
  const size_t dstride = (size_t)pad + n;
  std::vector<int16_t> cI(numTaps), cQ(numTaps);
  uint32_t lcg = 12345u;
  for (uint32_t i = 0; i < numTaps; ++i) { lcg = lcg * 1664525u + 1013904223u; cI[i] = (int16_t)((int)(lcg >> 20) - 2048); cQ[numTaps - 1 - i] = cI[i]; }
  std::vector<int> A, B, C, D;
  expand_set_int(numTaps, cI.data(), cQ.data(), A, B, C, D);
  std::vector<uint8_t> bm((size_t)4 * tc_tile_samples() * K);
  tc_build_bmat(A.data(), B.data(), C.data(), D.data(), KP, K, bm.data());
  std::vector<int16_t> hrow(dstride);
  for (size_t i = 0; i < dstride; ++i) { lcg = lcg * 1664525u + 1013904223u; hrow[i] = (int16_t)(lcg >> 16); }
  DevBuf din, dout, dbm, dk, ds, dctr;
  OPCK(dctr.alloc(sizeof(int)));
  OPCK(din.alloc(rows * dstride * 2)); OPCK(dout.alloc((size_t)rows * n * 2)); OPCK(dbm.alloc(bm.size())); OPCK(dk.alloc(rows)); OPCK(ds.alloc(rows));
  { // the same row pattern everywhere is fine for timing (no data-dependent work): upload 64 rows, replicate on the device
    const uint32_t rep = std::min<uint32_t>(64, rows);
    std::vector<int16_t> blockrows((size_t)rep * dstride);
    for (uint32_t r = 0; r < rep; ++r) memcpy(blockrows.data() + (size_t)r * dstride, hrow.data(), dstride * 2);
    OPCK(cudaMemcpy(din.p, blockrows.data(), blockrows.size() * 2, cudaMemcpyHostToDevice));
    for (uint32_t r = rep; r < rows; r += rep)
      OPCK(cudaMemcpy(din.as<int16_t>() + (size_t)r * dstride, din.p, (size_t)std::min(rep, rows - r) * dstride * 2, cudaMemcpyDeviceToDevice));
  }
  OPCK(cudaMemcpy(dbm.p, bm.data(), bm.size(), cudaMemcpyHostToDevice));
  OPCK(cudaMemset(dk.p, kind0, rows));
  OPCK(cudaMemset(ds.p, 0, rows));
  cudaEvent_t e0, e1;
  OPCK(cudaEventCreate(&e0)); OPCK(cudaEventCreate(&e1));
  for (int w = 0; w < 3; ++w)
    OPCK(launch_fir_demod_tc(din.as<int16_t>() + pad, dstride, dout.as<int16_t>(), n, rows, n, K, dbm.as<uint8_t>(), ds.as<uint8_t>(), dk.as<uint8_t>(), dctr.as<int>(), nullptr));
  OPCK(cudaDeviceSynchronize());
  OPCK(cudaEventRecord(e0, nullptr));
  for (int it = 0; it < iters; ++it)
    OPCK(launch_fir_demod_tc(din.as<int16_t>() + pad, dstride, dout.as<int16_t>(), n, rows, n, K, dbm.as<uint8_t>(), ds.as<uint8_t>(), dk.as<uint8_t>(), dctr.as<int>(), nullptr));
  OPCK(cudaEventRecord(e1, nullptr));
  OPCK(cudaEventSynchronize(e1));
  float ms = 0.f;
  OPCK(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  *ms_per_iter = ms / (float)iters;
  return MSDR_OK;
}

int msdr_op_sqrt_q31(int device, const int32_t *in, int32_t *out, int32_t *status, uint32_t n)
{
  if (!in || !out) return MSDR_ERR_ARGUMENT;
  int st = op_begin(device); if (st) return st;
  DevBuf a, b, c;
  OPCK(a.alloc((size_t)n * 4)); OPCK(b.alloc((size_t)n * 4)); OPCK(c.alloc((size_t)n * 4));
  OPCK(cudaMemcpy(a.p, in, (size_t)n * 4, cudaMemcpyHostToDevice));
  OPCK(launch_sqrt_q31(a.as<int32_t>(), b.as<int32_t>(), c.as<int32_t>(), n, nullptr));
  OPCK(cudaMemcpy(out, b.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
  if (status) OPCK(cudaMemcpy(status, c.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
  return MSDR_OK;
}

} // extern "C"
