// msdr_internal.h — host/device shared declarations (not part of the public ABI).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace msdr {

namespace fe { struct State; } // msdr_frontend.cuh

constexpr int kGroup = 32;            // channels per work group (one biquad lane each)
constexpr int kBqWords = 64;          // 2 objects x 4 stages x 8 words (filter_biquad.h:152)
constexpr float kAnrLidx0 = 120.0f, kAnrNgamma0 = 0.001f; // initial LMS leak index and noise gain (Minimal-SDR.ino:715,718)

// taps per polyphase sub-filter, padded: KP = roundup4(T/2 + 1)
inline __host__ __device__ uint32_t kp_of_taps(uint32_t T) { return ((T / 2u + 1u) + 3u) & ~3u; }
// raw-sample halo carried in front of each tile: H = roundup8(2*KP - 2) >= T - 1
inline __host__ __device__ uint32_t hist_of_kp(uint32_t KP) { return ((2u * KP - 2u) + 7u) & ~7u; }

struct ChainParams {
  const int16_t *in;      // [C][stride]
  int16_t *out;           // [C][stride]
  size_t stride;          // samples
  uint32_t C;             // channels processed by this launch: chain channels [ch0, ch0 + C)
  uint32_t ch0;           // first chain channel (indexes hist/bq/mode/setid); in/out rows are launch-relative
  uint32_t Cpad;          // row pitch of the SoA state arrays (multiple of 32)
  uint32_t L;             // samples per channel in this launch (multiple of 128)
  uint32_t H;             // history / halo length in samples (multiple of 8)
  int16_t *hist;          // [C][H]   last H raw ADC samples per channel
  int32_t *bq;            // [64][Cpad] biquad definition words, SoA
  const uint8_t *mode;    // [C] msdr_mode
  const uint8_t *setid;   // [C] FIR coefficient-set id
  uint32_t NG;            // channel groups
  uint32_t NT;            // spans per channel in this launch (v4)
  uint32_t n_items;       // work items: v4 row blocks x spans, v5 / v5l row blocks, v6 group blocks
  int *ctrl;              // v4: [0] work counter, [1] spans the loaders have taken (flow control)
  uint32_t W;             // v4: biquad chains per wave
  uint32_t ablate;        // study only: bit 0 skip the FIR arithmetic, bit 1 skip the biquad arithmetic (results are wrong)
  uint32_t am_q31;
  // tensor-core FIR plan (chain kernel v4, msdr_chain_v4.cu)
  const uint32_t *tc_rowmap;   // [n_rb][128] launch-relative row, 0xFFFFFFFF = padding
  const uint4 *tc_rb;          // [n_rb] .x = table id, the other words 0 (v6: [n_items] .x, .y = the tables of the two half blocks)
  const uint32_t *tc_wave_rb0; // [n_waves + 1] first row block of each wave
  const uint8_t *tc_bmat;      // [n_sets][4 * 64 * K] Toeplitz operands
  uint32_t tc_K, tc_ring, tc_sub, tc_ff; // tc_ff: kernel shape 0/1/2 (msdr_chain_v4.cu: chain_v4_config)
  uint32_t NU;                 // readiness units per channel (v4)
  uint32_t spare_sms;          // v4: launch this many fewer CTAs than a wave has slots (never fewer than there are chains to pin)
  long long *prof;             // developer profile buffer [grid][64] or NULL
  int *tile_cnt;               // [NG][NU] rows of group g whose unit u is in `out` (zeroed before the launch)
  // ADC-code input (row-block kernels only): non-NULL = `in` holds raw uint16 codes and the converters run the front end first
  fe::State *fe;               // [chain channels] front-end state, indexed like hist
  float agc_max;
  uint32_t agc_on;
  // channel list (v5, v5l, v6 int16 only): non-NULL = launch row r is chain channel chlist[r] instead of ch0 + r
  const uint32_t *chlist;
};

struct ChainLaunchInfo {
  int grid, block;
  size_t smem;
  int tile;
};

// Fused mix + FIR pair + demod + biquad cascade (K1, msdr_chain_v4.cu). variant: 0 = default.
cudaError_t launch_chain_v4(const ChainParams &p, cudaStream_t stream, int variant, ChainLaunchInfo *info);
uint32_t chain_v4_span_samples();
uint32_t chain_v4_unit_samples();
bool chain_v4_config(uint32_t K, int smem_max, uint32_t rings[4]);
// K4 (msdr_frontend.cu) over C rows: raw codes -> conditioned int16 IF samples; state = the first row's front-end state, or with
// map != NULL the state array that row r indexes at map[r] (the rows' codes and outputs stay row r).
// sms > 0 packs the channel groups into about that many CTAs.
// launch_frontend_preset: hpf_x1 = first_reading << 14, hpf_y1 = 0 in state[channels[i]] for the n device-resident channels, or with
// channels == NULL in state[ch0 + i].
cudaError_t launch_frontend_preset(fe::State *state, const uint32_t *channels, uint32_t ch0, uint32_t n, uint16_t first_reading, cudaStream_t s);
cudaError_t launch_frontend(const uint16_t *adc, int16_t *out, size_t stride, uint32_t C, uint32_t n_blocks, fe::State *state, float agc_max,
                            int agc_on, int sms, cudaStream_t s, const uint32_t *map = nullptr);
// row-block kernel for many channels (msdr_chain_v5.cu): p.n_items = number of row blocks, p.tc_ring from chain_v5_config of the same
// form (0 = does not fit).  half_tile: the form with half-tile hand-offs, for windows too long for whole tiles (256 taps).
// p.fe != NULL selects the ADC-code instantiation (default biquad form only), p.chlist != NULL the channel-list one (the same)
cudaError_t launch_chain_v5(const ChainParams &p, cudaStream_t stream, int variant, int sms, bool half_tile, ChainLaunchInfo *info);
uint32_t chain_v5_config(uint32_t K, int smem_max, bool half_tile);
// pinned 32-channel group blocks with the tile rows folded over time (msdr_chain_v6.cu): p.tc_rowmap = [n_items][32] rows,
// p.tc_rb[i].x / .y = the tables of its two half blocks, p.tc_ring = sub-tile slots from chain_v6_config (0 = the window does not fit)
cudaError_t launch_chain_v6(const ChainParams &p, cudaStream_t stream, int variant, int sms, ChainLaunchInfo *info);
uint32_t chain_v6_config(uint32_t K, int smem_max);
uint32_t chain_v6_group_rows();

// stage-level kernels on device buffers
cudaError_t launch_mix_fs4(const int16_t *in, int16_t *I, int16_t *Q, uint32_t rows, uint32_t n, size_t stride, cudaStream_t s);
cudaError_t launch_fir_fast_q15(uint32_t T, const int16_t *coef, const int16_t *hist_in, int16_t *hist_out, const int16_t *in, int16_t *out,
                                uint32_t rows, uint32_t n, size_t stride, cudaStream_t s);
cudaError_t launch_demod(int kind, const int16_t *I, const int16_t *Q, int16_t *out, uint32_t rows, uint32_t n, size_t stride, cudaStream_t s);
// side-lane glue (msdr_stage_kernels.cu): chmap != NULL gives the chain channel of each scratch row, else it is ch0 + rows[i]
cudaError_t launch_gather_rows(const uint32_t *rows, const uint32_t *chmap, uint32_t n, uint32_t ch0, const int16_t *hist, uint32_t H, const int16_t *in, size_t stride,
                               int16_t *raw, uint32_t L, cudaStream_t s);
cudaError_t launch_scatter_rows(const uint32_t *rows, uint32_t n, const int16_t *audio, size_t astride, int16_t *out, size_t stride, uint32_t L, cudaStream_t s);
cudaError_t launch_zero_hist_rows(int16_t *hist, uint32_t H, const uint32_t *channels, uint32_t n, cudaStream_t s);
cudaError_t launch_bq_words(int dir, const uint32_t *rows, const uint32_t *chmap, uint32_t n, uint32_t ch0, int32_t *bq, uint32_t Cpad, int32_t *defs, cudaStream_t s);
cudaError_t launch_demod_rows(const uint8_t *kinds, const int16_t *I, const int16_t *Q, size_t stride, int16_t *out, size_t ostride, uint32_t rows, uint32_t n,
                              cudaStream_t s);
cudaError_t launch_anr(int16_t *data, size_t stride, uint32_t rows, uint32_t n_blocks, const uint8_t *row_mode, const uint32_t *chmap, float *d, float *w,
                       float *lidx, float *ngamma, int *in_idx, uint32_t Cpad, cudaStream_t s);
cudaError_t launch_syncam(const int16_t *I, const int16_t *Q, size_t stride, int16_t *out, size_t ostride, uint32_t rows, uint32_t n, float *state,
                          uint32_t Cpad, const uint32_t *chmap, const uint8_t *row_sel, cudaStream_t s);
cudaError_t launch_dac_codes(const int16_t *in, uint16_t *out, uint32_t rows, uint32_t n, size_t stride, cudaStream_t s);
cudaError_t launch_amplifier(const int32_t *mult, int16_t *data, uint32_t rows, uint32_t n, size_t stride, cudaStream_t s);
cudaError_t launch_biquad(int32_t *definition, int16_t *data, uint32_t rows, uint32_t n, size_t stride, cudaStream_t s);
cudaError_t launch_freq_conv(int dir, int16_t *I, int16_t *Q, const int16_t *oscI, const int16_t *oscQ, uint32_t rows, uint32_t n, size_t stride,
                             cudaStream_t s);
// K3 study: tensor-core FIR + demod (msdr_fir_tc.cu)
uint32_t tc_window_words(uint32_t T);
uint32_t tc_window_words_kp(uint32_t KP);
uint32_t tc_tile_samples();
uint32_t tc_tile_rows();
void tc_build_bmat(const int *cA, const int *cB, const int *cC, const int *cD, uint32_t KP, uint32_t K, uint8_t *out);
cudaError_t launch_fir_demod_tc(const int16_t *in, size_t stride, int16_t *out, size_t ostride, uint32_t rows, uint32_t L, uint32_t K, const uint8_t *bmat,
                                const uint8_t *row_set, const uint8_t *row_kind, int *counter, cudaStream_t s);
cudaError_t launch_sqrt_check(unsigned long long *d_mismatch, cudaStream_t s);
cudaError_t launch_sqrt_q31(const int32_t *in, int32_t *out, int32_t *status, uint32_t n, cudaStream_t s);
cudaError_t launch_bq_setcoef(int32_t *bq, uint32_t Cpad, int object, uint32_t ch0, uint32_t nch, uint32_t stage, const int32_t coef[5], cudaStream_t s);

} // namespace msdr
