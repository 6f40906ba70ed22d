/* msdr.h — C ABI of the B200-native Minimal-SDR receive DSP chain.
 *
 * Drop-in boundary for ONE path of FrankBoesing/Minimal-SDR: what `demodulation()`
 * (Minimal-SDR.ino:518-775) does per 128-sample block — fs/4 mix, arm_fir_fast_q15 on I and Q,
 * SSB / AM demodulation — followed by the two AudioFilterBiquad objects of the audio graph
 * (Minimal-SDR.ino:71-72, src/Audio/filter_biquad.cpp:33-82), batched over independent channels and
 * executed by hand-written CUDA kernels for sm_100a.  There is no CPU fallback: every entry point that
 * computes needs a CUDA device and fails with MSDR_ERR_CUDA otherwise.
 *
 * Conventions
 *   - plain C types only; all buffers are caller-owned; a chain owns its device state and its copies of
 *     the coefficients (the reference's FIR borrows the table pointer, arm_fir_init_q15.c:103 — here
 *     msdr_fir_set_coefficients() models an in-place rewrite of that table, Minimal-SDR.ino:222).
 *   - sample buffers are int16 [n_channels][stride] row-major, `n_blocks*128` samples used per row.
 *   - return value: 0 = success; negative = error.  -1..-6 carry the values of CMSIS `arm_status`
 *     (arm_math.h:404-413) so `msdr_fir_init_q15` reports odd tap counts exactly like
 *     `arm_fir_init_q15` (arm_fir_init_q15.c:93-96).
 *   - a chain is not thread-safe; setters are stream-ordered and take effect at the next update, i.e. at
 *     a block boundary, like the reference's __disable_irq()/AudioNoInterrupts() sections
 *     (filter_biquad.cpp:88-99, Minimal-SDR.ino:336-367).
 */
#ifndef MSDR_H
#define MSDR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSDR_BLOCK_SAMPLES 128   /* AUDIO_BLOCK_SAMPLES (Teensy core; Minimal-SDR.ino:113-114) */
#define MSDR_MAX_TAPS 256        /* BASELINE config 4: 255 taps + zero pad (arm_fir_init_q15.c:55-64) */
#define MSDR_MAX_FIR_SETS 32     /* distinct (numTaps, cI, cQ) tables alive in one chain */
#define MSDR_BIQUAD_OBJECTS 2    /* biquad1_dac, biquad2_dac (Minimal-SDR.ino:71-72) */
#define MSDR_BIQUAD_STAGES 4     /* filter_biquad.h:152: int32_t definition[32] = 4 stages x 8 words */

typedef enum {
  MSDR_OK = 0,
  MSDR_ERR_ARGUMENT = -1,       /* == ARM_MATH_ARGUMENT_ERROR */
  MSDR_ERR_LENGTH = -2,         /* == ARM_MATH_LENGTH_ERROR */
  MSDR_ERR_CUDA = -100,         /* CUDA runtime/driver failure or no device; see msdr_last_error() */
  MSDR_ERR_UNSUPPORTED = -101,
  MSDR_ERR_NOMEM = -102,
  MSDR_ERR_NOT_INITIALISED = -103 /* update() on a channel whose FIR was never initialised */
} msdr_status;

/* stations.h:4  enum { SYNCAM, AM, LSB, USB, CW } — same numeric values */
typedef enum { MSDR_MODE_SYNCAM = 0, MSDR_MODE_AM = 1, MSDR_MODE_LSB = 2, MSDR_MODE_USB = 3, MSDR_MODE_CW = 4 } msdr_mode;

/* chain flags */
#define MSDR_FLAG_AM_Q31 1u /* Teensy 3.2 arithmetic: AM/CW/SYNCAM envelope via arm_sqrt_q31 (Minimal-SDR.ino:617-627)
                               instead of the Teensy 3.5/3.6 arm_sqrt_f32 path (:606-616) */

typedef struct msdr_chain msdr_chain;

/* Per-channel state, for checkpoint / resume / migration between GPUs. */
typedef struct {
  int32_t mode;                                 /* msdr_mode */
  uint32_t num_taps;                            /* 0 = FIR not initialised */
  int32_t fir_set;                              /* coefficient-set id inside this chain, -1 = none */
  int16_t fir_history[MSDR_MAX_TAPS];           /* last num_taps-1 RAW ADC samples, oldest first, in [0, num_taps-1);
                                                   the reference's two pState delay lines (arm_fir_fast_q15.c:296-327) are
                                                   this sequence after the fs/4 mix */
  int32_t biquad_definition[MSDR_BIQUAD_OBJECTS][32]; /* filter_biquad.h:152 layout, verbatim */
  float syncam_pll[3];                          /* fil_out, omega2, phzerror of the SYNCAM PLL (Minimal-SDR.ino:643-645) */
} msdr_channel_state;

/* ---- lifetime -------------------------------------------------------------------------------- */

/* Creates a chain of n_channels independent receive channels on CUDA device `device`.
 * max_taps (even, 4..MSDR_MAX_TAPS; 0 = 102, the reference's MAX_num_taps, Minimal-SDR.ino:110) bounds the FIR
 * length and sizes the per-channel history.  All channels start in mode AM (Minimal-SDR.ino:98) with
 * both biquad objects zeroed — "by default, the filter will not pass anything" (filter_biquad.h:36-39) —
 * and no FIR bound (the sketch always calls init_FIR() in setup(), Minimal-SDR.ino:404). */
int msdr_chain_create(msdr_chain **out, int device, uint32_t n_channels, uint32_t max_taps, uint32_t flags);
void msdr_chain_destroy(msdr_chain *chain);
/* Runs the chain's work on a caller-provided cudaStream_t (e.g. torch's current stream); NULL = the chain's own non-blocking
 * stream, which is NOT ordered with the legacy default stream - pass cudaStreamLegacy ((cudaStream_t)1) to run there. */
int msdr_chain_set_stream(msdr_chain *chain, void *cuda_stream);
int msdr_chain_synchronize(msdr_chain *chain);
const char *msdr_last_error(const msdr_chain *chain); /* chain may be NULL: error of the last failed create */
uint32_t msdr_chain_channels(const msdr_chain *chain);

/* ---- configuration (the reference's globals and setters, per channel range [ch0, ch0+nch)) ---- */

/* `mode = ...` (Minimal-SDR.ino:98; UI.cpp mode menu).  Only selects the demodulation branch
 * (Minimal-SDR.ino:589); like the reference, re-binding FIR tables is a separate call (init_FIR via tune()). */
int msdr_chain_set_mode(msdr_chain *chain, uint32_t ch0, uint32_t nch, int mode);

/* arm_fir_init_q15 x2 as in init_FIR() (Minimal-SDR.ino:901-930; arm_math.h:1106-1128): zeroes the delay lines of
 * the channels and binds taps cI (I branch) and cQ (Q branch), `numTaps` each, in the reference's
 * "time reversed" order (arm_fir_init_q15.c:50-54).  Odd numTaps -> MSDR_ERR_ARGUMENT and nothing changes. */
int msdr_fir_init_q15(msdr_chain *chain, uint32_t ch0, uint32_t nch, uint16_t numTaps, const int16_t *cI, const int16_t *cQ);

/* The same two setters for a list of channels (n entries, any order): configures interleaved mode families with one call each. */
int msdr_chain_set_mode_list(msdr_chain *chain, const uint32_t *channels, uint32_t n, int mode);
int msdr_fir_init_q15_list(msdr_chain *chain, const uint32_t *channels, uint32_t n, uint16_t numTaps, const int16_t *cI, const int16_t *cQ);

/* In-place rewrite of the bound tables (calc_demod_filter(), Minimal-SDR.ino:221-223 / UI.cpp:337-345): same tap
 * count, delay lines kept.  All channels in the range must currently share one table. */
int msdr_fir_set_coefficients(msdr_chain *chain, uint32_t ch0, uint32_t nch, const int16_t *cI, const int16_t *cQ);
/* numTaps of the FIR pair bound to channel `ch` (arm_fir_instance_q15::numTaps, arm_math.h:1027-1032): what
 * msdr_fir_set_coefficients reads from cI and cQ.  0 = not initialised; negative = bad argument. */
int msdr_chain_fir_taps(const msdr_chain *chain, uint32_t ch);

/* AudioFilterBiquad::setCoefficients(stage, const int *) (filter_biquad.cpp:84-100) on object `object`
 * (0 = biquad1_dac, 1 = biquad2_dac): coef = {b0,b1,b2,a1,a2} in Q2.30; a1,a2 are stored negated; the previous
 * stage gets its "another stage follows" flag; x/y history kept; residual cleared; stage >= 4 silently ignored. */
int msdr_biquad_set_coefficients(msdr_chain *chain, int object, uint32_t ch0, uint32_t nch, uint32_t stage, const int32_t *coef);

/* ---- the hot path ------------------------------------------------------------------------------ */

/* One `update_all()` worth of work for every channel, n_blocks AudioStream blocks deep:
 * out[c][n] = biquad2(biquad1(demod(FIR_I(mixI(in[c])), FIR_Q(mixQ(in[c]))))), state carried across calls.
 * HOST buffers: copies in, runs, copies out, returns when `out` is complete.  Pinned buffers
 * (msdr_host_alloc) make the copies overlap the kernels. */
int msdr_chain_update(msdr_chain *chain, const int16_t *in, int16_t *out, uint32_t n_blocks, size_t stride);

/* Same on DEVICE buffers, asynchronous on the chain's stream.  in/out must be 16-byte aligned, stride a multiple
 * of 8 samples; in and out may not overlap. */
int msdr_chain_update_device(msdr_chain *chain, const int16_t *d_in, int16_t *d_out, uint32_t n_blocks, size_t stride);

/* Same for the channel sub-range [ch0, ch0+nch) only: d_in/d_out hold nch rows (row r = channel ch0 + r).
 * Lets a caller stream channel shards through the device independently (msdr_chain_update does exactly that). */
int msdr_chain_update_range_device(msdr_chain *chain, uint32_t ch0, uint32_t nch, const int16_t *d_in, int16_t *d_out, uint32_t n_blocks,
                                   size_t stride);

/* Channels channels[0..n) only, in list order: row i of d_in / d_out is channel channels[i].  Same buffer, alignment, stride and
 * state rules as msdr_chain_update_range_device; results, outputs and state equal those of range updates of the same channels.
 * `channels` is a host array in any order.  MSDR_ERR_ARGUMENT, before anything is enqueued, for a channel >= the chain's
 * channel count, a channel listed twice, or channels == NULL with n > 0; n == 0 launches nothing.  int16 input: the
 * front-end state (msdr_chain_enable_frontend) is left alone (ADC codes: msdr_chain_update_adc_list_device).  Runs on the
 * time-folded kernel while the list's channel groups fit one per SM, else on the row-block kernel, never on the chain kernel
 * v4; scattered channels gather their state, so a list can run below a range of the same size (rates: DESIGN.md §6).  The
 * row plan of each distinct list is cached like that of a range (INTEGRATION.md §3h). */
int msdr_chain_update_list_device(msdr_chain *chain, const uint32_t *channels, uint32_t n, const int16_t *d_in, int16_t *d_out,
                                  uint32_t n_blocks, size_t stride);
/* The same on host buffers of n rows, through the 3-slot copy / kernel / copy pipeline of msdr_chain_update (the list is cut
 * into chunks of host_chunk_channels entries like the chain is there). */
int msdr_chain_update_list(msdr_chain *chain, const uint32_t *channels, uint32_t n, const int16_t *in, int16_t *out, uint32_t n_blocks,
                           size_t stride);

/* Device time of the last update in milliseconds (CUDA events), the analogue of the reference's
 * micros()-around-demodulation() load figure (Minimal-SDR.ino:533,774; :415-432). Synchronises. */
int msdr_chain_last_update_ms(msdr_chain *chain, float *ms);
/* AudioProcessorUsage() / AudioProcessorUsageMax() / AudioProcessorUsageMaxReset() of the Teensy core as the sketch uses them
 * (Minimal-SDR.ino:424-426: load as a percentage of the block period AUDIO_BLOCK_SAMPLES / pdb_freq_actual): device time of an
 * update divided by the real-time duration of the blocks it processed at `sample_rate_hz`, for the last update and as a
 * running maximum.  The first call switches the "timing" option on (updates before it are not counted); reading the figures
 * waits for the last update to finish. */
int msdr_chain_processor_usage(msdr_chain *chain, double sample_rate_hz, float *last_percent, float *max_percent);
int msdr_chain_processor_usage_max_reset(msdr_chain *chain);
/* Number of kernels launched by this chain since creation (bench.py reports it as gpu_launches). */
uint64_t msdr_chain_launch_count(const msdr_chain *chain);
/* How often the row plan of the tensor-core kernel (channels sorted by tap table, Toeplitz operands) was rebuilt: once per
 * change of a table binding, a table's contents or the updated channel range - never per update of an unchanged configuration. */
uint64_t msdr_chain_plan_build_count(const msdr_chain *chain);
/* Which fused kernel (and which of its shapes) the last update launched; bench.py names it in `roofline.kernel`. */
const char *msdr_chain_last_kernel(const msdr_chain *chain);

int msdr_chain_get_state(msdr_chain *chain, uint32_t ch, msdr_channel_state *out);
int msdr_chain_set_state(msdr_chain *chain, uint32_t ch, const msdr_channel_state *in);

/* ---- snapshots: checkpoint / resume / migration / re-sharding of channel ranges ----
 * A snapshot of channels [ch0, ch0+nch) holds everything they carry: their FIR tables (renumbered densely), modes and ANR switches, the
 * FIR history, both biquad objects, the SYNCAM PLL, and the front-end and LMS state when the chain has them.  The format is versioned and
 * little-endian, every section starts on a 256-byte boundary (DESIGN.md 7); state sections are plain strided copies of the chain's arrays.
 * msdr_chain_restore(chain, ch0, buf, bytes, first, n) gives chain channels [ch0, ch0+n) the state of snapshot channels [first, first+n)
 * (restoring a whole snapshot into the range it came from gives back exactly the chain that was saved), into any chain on any device
 * whose flags equal the snapshot's and whose max_taps covers the tables used.  A different FIR history length (max_taps) keeps the last
 * min(H, H') samples, like msdr_chain_set_state.  Restore is all or nothing: MSDR_ERR_ARGUMENT for a bad magic, a truncated buffer, bad
 * offsets, ranges outside the snapshot or the chain, other flags, a table longer than max_taps or other AGC parameters than the chain's
 * front end; MSDR_ERR_UNSUPPORTED for another format version; MSDR_ERR_NOMEM when the range would need more than MSDR_MAX_FIR_SETS live
 * tables (tables only the range used give their slots back first).  A refused restore changes nothing.
 *   - front end: a snapshot with one enables it on a chain without one (its AGC parameters; other channels start as after
 *     msdr_chain_enable_frontend); a chain with one and a snapshot without gives the restored channels the initial front-end state.
 *   - ANR: a snapshot of a chain that ever switched ANR on allocates the LMS arrays; one without gives restored channels the initial state.
 *   - a restore is one configuration change: the next update over a range builds at most one row plan.
 * The host calls return when the buffer is written / may be freed; pinned buffers (msdr_host_alloc) move at PCIe rate.  The device
 * calls take a buffer on the chain's device and are asynchronous on the chain's stream, ordered after every earlier update; keep d_buf
 * alive until the stream has passed.  restore_device reads header, tables and meta with one small synchronous copy, and trusts the
 * state sections (a host restore also checks the front-end agc_idx and ANR in_idx of every restored channel). */
size_t msdr_chain_snapshot_bytes(const msdr_chain *chain, uint32_t nch);
int msdr_chain_snapshot(msdr_chain *chain, uint32_t ch0, uint32_t nch, void *buf, size_t bytes);          /* host buffer, returns when written */
int msdr_chain_snapshot_device(msdr_chain *chain, uint32_t ch0, uint32_t nch, void *d_buf, size_t bytes); /* device buffer on the chain's device, asynchronous on its stream */
int msdr_chain_restore(msdr_chain *chain, uint32_t ch0, const void *buf, size_t bytes, uint32_t first, uint32_t n);
int msdr_chain_restore_device(msdr_chain *chain, uint32_t ch0, const void *d_buf, size_t bytes, uint32_t first, uint32_t n);
/* host-only, no device needed: validates a snapshot header (host copy of at least its first 256 bytes).  flags = the chain flags of the
 * snapshot, plus MSDR_SNAPSHOT_FRONTEND / MSDR_SNAPSHOT_ANR for the sections it has; max_taps_needed = the longest table it holds. */
#define MSDR_SNAPSHOT_FRONTEND (1u << 16)
#define MSDR_SNAPSHOT_ANR (1u << 17)
int msdr_snapshot_info(const void *header, size_t bytes, uint32_t *n_channels, uint32_t *max_taps_needed, uint32_t *flags);

/* Options.  "variant" selects the shape of the fused kernel for studies and cross-checks (all shapes are bit-exact, DESIGN.md 6):
 *   0    default, by channel count: the time-folded kernel (msdr_chain_v6.cu) up to one 32-channel group block per SM; tensor-core
 *        FIR producers (tcgen05 kind::i8) + pinned biquad chains (msdr_chain_v4.cu: feed-forward helper warps up to 148 channel
 *        groups, two chain sets per SM beyond) up to one wave of those (9472 channels on 148 SMs); the row-block kernel
 *        (msdr_chain_v5.cu, whole tiles, or half tiles for the 256-tap window) from there
 *   16384  never the time-folded kernel;  65536  the time-folded kernel for any channel count;  +2 there: feed-forward products as DFMA
 *   8192   never the row-block kernel;    4096   the row-block kernel for any channel count;    32768  its half-tile form for any window
 *          (+1, +2, +4, +8, +12 there: the stage's products as IMAD.WIDE instead of IMAD.HI (the half-tile form: the other way round) /
 *          DFMA feed-forward / chained DFMA / all DFMA / split 16 x 16 bit)
 *   128  helper-warp shape even beyond 148 groups;  2048: post-warp shape (whole stages in the chain warps);
 *   256  classic shape (neither helper nor post warps)
 *   512  never run two chain sets per SM
 *   +16 / +32: ablation (skip the FIR / the biquad arithmetic; results are wrong, timing only)
 * "timing" (CUDA events around each update), "host_chunk_channels", "host_chunk_blocks" (msdr_chain_update pipelining).
 * "spare_sms" = n: the chain kernel for few channels launches n fewer CTAs than there are SMs (never fewer than it has channel groups
 * to pin), leaving those SMs to a kernel on another stream, e.g. the front end of the next block batch (msdr_frontend_set_option "sms").
 * Environment, developer aids: MSDR_VARIANT (default variant of new chains), MSDR_PROF (per-role cycle counters on stderr). */
int msdr_chain_set_option(msdr_chain *chain, const char *key, int value);

/* pinned host memory for update() */
void *msdr_host_alloc(size_t bytes);
void msdr_host_free(void *p);

/* ---- stage-level batched operators (one reference primitive each; HOST buffers) ------------------
 * Used by the AudioStream façade (include/msdr/Audio.h) and by the per-stage parity tests. `rows`
 * independent streams of `n` samples each, row-major with the given stride. */

/* fs/4 mix, Minimal-SDR.ino:546-558.  n % 4 == 0. */
int msdr_op_mix_fs4(int device, const int16_t *in, int16_t *outI, int16_t *outQ, uint32_t rows, uint32_t n, size_t stride);

/* arm_fir_fast_q15 (arm_fir_fast_q15.c:60-329) over `rows` streams sharing one tap table.  history: int16
 * [rows][numTaps-1] in/out (NULL = zero history, not written back) — the first numTaps-1 entries of pState. */
int msdr_op_fir_fast_q15(int device, uint16_t numTaps, const int16_t *coeffs, int16_t *history,
                         const int16_t *in, int16_t *out, uint32_t rows, uint32_t n, size_t stride);

/* demodulation switch, Minimal-SDR.ino:589-628.  kind: 0 LSB, 1 USB, 2 AM/CW f32, 3 AM/CW/SYNCAM q31. */
int msdr_op_demod(int device, int kind, const int16_t *I, const int16_t *Q, int16_t *out, uint32_t rows, uint32_t n, size_t stride);

/* AudioFilterBiquad::update (filter_biquad.cpp:33-82) over `rows` streams, in place, n % 2 == 0.
 * definition: int32 [rows][32] in/out, filter_biquad.h:152 layout. */
int msdr_op_biquad(int device, int32_t *definition, int16_t *data, uint32_t rows, uint32_t n, size_t stride);

/* AudioEffectFreqConv::update (freq_conv.cpp:30-116), in place on I and Q; oscI/oscQ: int16[n] tables
 * shared by all rows (the sketch's Osc_I_buffer_i / Osc_Q_buffer_i, freq_conv.h:33-34). */
int msdr_op_freq_conv(int device, int dir, int pass, int16_t *I, int16_t *Q, const int16_t *oscI, const int16_t *oscQ,
                      uint32_t rows, uint32_t n, size_t stride);

/* arm_sqrt_q31 (arm_sqrt_q31.c:50-138) element-wise; status[i] = 0 or -1 like arm_status (may be NULL). */
int msdr_op_sqrt_q31(int device, const int32_t *in, int32_t *out, int32_t *status, uint32_t n);

/* K3 study (DESIGN.md): mix + FIR pair + demodulation on the tensor cores (tcgen05 kind::i8, byte-split Toeplitz form), no
 * biquad, zero initial history.  n must be a multiple of 64.  kinds: per-row demod kind (as msdr_op_demod) or NULL for kind0. */
int msdr_op_fir_demod_tc(int device, uint16_t numTaps, const int16_t *cI, const int16_t *cQ, const uint8_t *kinds, int kind0, const int16_t *in,
                         int16_t *out, uint32_t rows, uint32_t n, size_t stride);
/* Device-resident timing of the same kernel on pseudo-random data: milliseconds per launch over `iters` launches. */
int msdr_study_fir_demod_tc_time(int device, uint16_t numTaps, uint32_t rows, uint32_t n, int kind0, int iters, float *ms_per_iter);
/* Exhaustive device check: the epilogue's branch-free float square root against sqrt.rn.f32 for every AM envelope argument
 * (integers 0 .. 2^31-1, arm_sqrt_f32 of Minimal-SDR.ino:606); *mismatches must come back 0. */
int msdr_study_sqrt_check(int device, uint64_t *mismatches);

/* ---- front-end conditioning (SURVEY 8f rank 1): what sits between the ADC and the receive chain in the sketch ---------------
 * raw unsigned ADC codes -> DC-blocking high-pass (AudioInputAnalog::update, input_adc.cpp:198-212) -> AudioAmplifier gain
 * (mixer.cpp:34-47,134-159) -> int16 IF samples for msdr_chain_update*; per block the sketch's AGC (Minimal-SDR.ino:445-515)
 * moves the amplifier gain for the blocks that follow (zero queue latency in a batch).  agc_start / agc_max / agc_on are the
 * sketch's AGC_start (0.25), AGC_Max (40) and AGC_on (.ino:94-100).  One object per batch of channels, state carried from
 * update to update.  Known reference defect reproduced as "value dropped": every 26th block maximum is stored outside
 * agc_buffer (.ino:481-482). */
typedef struct msdr_frontend msdr_frontend;
typedef struct msdr_frontend_state {
  int32_t hpf_x1, hpf_y1;  /* input_adc.cpp:37-38 */
  int32_t multiplier;      /* AudioAmplifier::multiplier (mixer.h:80) */
  int32_t agc_idx;         /* .ino:451 */
  float agc_val;           /* .ino:104 */
  int16_t agc_buffer[25];  /* .ino:450 */
  int16_t reserved;
} msdr_frontend_state;
int msdr_frontend_create(msdr_frontend **out, int device, uint32_t n_channels, float agc_start, float agc_max, int agc_on);
void msdr_frontend_destroy(msdr_frontend *fe);
int msdr_frontend_set_stream(msdr_frontend *fe, void *cuda_stream);
int msdr_frontend_synchronize(msdr_frontend *fe);
const char *msdr_frontend_last_error(const msdr_frontend *fe);
/* AudioInputAnalog::init (input_adc.cpp:59-63): hpf_x1 = first reading << 14, hpf_y1 = 0 */
int msdr_frontend_preset(msdr_frontend *fe, uint32_t ch0, uint32_t nch, uint16_t first_reading);
/* host buffers [n_channels][stride] (synchronous) / device buffers (asynchronous on the object's stream; 16-byte aligned rows) */
int msdr_frontend_update(msdr_frontend *fe, const uint16_t *adc, int16_t *out, uint32_t n_blocks, size_t stride);
int msdr_frontend_update_device(msdr_frontend *fe, const uint16_t *d_adc, int16_t *d_out, uint32_t n_blocks, size_t stride);
int msdr_frontend_get_state(msdr_frontend *fe, uint32_t ch, msdr_frontend_state *out);
int msdr_frontend_set_state(msdr_frontend *fe, uint32_t ch, const msdr_frontend_state *in);
uint64_t msdr_frontend_launch_count(const msdr_frontend *fe);
/* "sms" = n > 0: run the conditioning kernel in about n CTAs of several warps (one per SM) instead of one small CTA per 32 channels
 * spread over the whole GPU, so that it can run BESIDE a receive chain that leaves SMs free (msdr_chain_set_option "spare_sms"):
 * conditioning of block batch k+1 on one stream while the chain works on batch k on another.  0 = spread (default). */
int msdr_frontend_set_option(msdr_frontend *fe, const char *key, int value);
/* AudioAmplifier::gain (mixer.h:75-79): clamp to +-32767, multiplier = (int32_t)(gain * 65536.0f) */
int32_t msdr_amp_gain_multiplier(float gain);

/* ---- receive chain from raw ADC codes: the front end above per channel of a chain, in front of it ------------------------------
 * adc1 -> amp_adc -> queue_adc -> demodulation() with AGC(p_adc) on every block (Minimal-SDR.ino:76-78,445-515) as one object.
 * Output, chain state and front-end state equal msdr_frontend_update followed by msdr_chain_update with the same parameters, however
 * a stream is cut into updates.  The FIR history holds conditioned IF samples in both input formats, so int16 and ADC updates may be
 * interleaved on one chain; an int16 update leaves the front-end state alone.  Buffer, alignment and stride rules are those of
 * msdr_chain_update / msdr_chain_update_device.  msdr_chain_last_kernel names the path: the front end fused into the converters of
 * the many-channel row-block kernels, or the front-end kernel over the range followed by the int16 path. */
/* (Re)initialise the per-channel front end of every channel of the chain, like msdr_frontend_create:
   hpf 0, agc_idx 25, agc_val = agc_start, multiplier = gain(agc_start). */
int msdr_chain_enable_frontend(msdr_chain *chain, float agc_start, float agc_max, int agc_on);
int msdr_chain_frontend_preset(msdr_chain *chain, uint32_t ch0, uint32_t nch, uint16_t first_reading); /* input_adc.cpp:59-63 */
/* The same for the channels channels[0..n) (host array, any order): MSDR_ERR_ARGUMENT for a channel >= the chain's channel count
 * or channels == NULL with n > 0, MSDR_ERR_NOT_INITIALISED before msdr_chain_enable_frontend; a refused call changes nothing.
 * One synchronising call for the whole list; its cost grows with n, not with the span of the listed channels. */
int msdr_chain_frontend_preset_list(msdr_chain *chain, const uint32_t *channels, uint32_t n, uint16_t first_reading);
/* MSDR_ERR_NOT_INITIALISED before msdr_chain_enable_frontend */
int msdr_chain_update_adc(msdr_chain *chain, const uint16_t *adc, int16_t *out, uint32_t n_blocks, size_t stride);  /* host buffers */
int msdr_chain_update_adc_device(msdr_chain *chain, const uint16_t *d_adc, int16_t *d_out, uint32_t n_blocks, size_t stride);
int msdr_chain_update_adc_range_device(msdr_chain *chain, uint32_t ch0, uint32_t nch, const uint16_t *d_adc, int16_t *d_out,
                                       uint32_t n_blocks, size_t stride);
/* Channel lists of ADC codes: row i of d_adc / d_out is chain channel channels[i] (host array, any order), asynchronous on the
 * chain's stream.  Output, chain state and front-end state equal those of msdr_chain_update_adc_range_device calls over the same
 * channels, however a stream is cut into calls; unlisted channels, their front end included, are not touched.  Refusals, before
 * anything is enqueued and changing nothing: MSDR_ERR_NOT_INITIALISED before msdr_chain_enable_frontend or while a channel has
 * no FIR bound; MSDR_ERR_ARGUMENT for a channel >= the chain's channel count, a channel listed twice, channels == NULL with
 * n > 0, or buffers, alignment and stride that msdr_chain_update_adc_range_device refuses.  n == 0 launches nothing.  The
 * front-end kernel conditions the listed rows with each listed channel's front-end state, then the kernel and the cached row
 * plan of msdr_chain_update_list_device for the same list run on them (msdr_chain_last_kernel: "msdr::fe::frontend_kernel
 * (front end), then ...; channel list"). */
int msdr_chain_update_adc_list_device(msdr_chain *chain, const uint32_t *channels, uint32_t n, const uint16_t *d_adc, int16_t *d_out,
                                      uint32_t n_blocks, size_t stride);
/* The same on host buffers of n rows, through the copy pipeline of msdr_chain_update_list. */
int msdr_chain_update_adc_list(msdr_chain *chain, const uint32_t *channels, uint32_t n, const uint16_t *adc, int16_t *out,
                               uint32_t n_blocks, size_t stride);
/* agc_idx outside [0, 25] is MSDR_ERR_ARGUMENT */
int msdr_chain_get_frontend_state(msdr_chain *chain, uint32_t ch, msdr_frontend_state *out);
int msdr_chain_set_frontend_state(msdr_chain *chain, uint32_t ch, const msdr_frontend_state *in);
/* AudioAmplifier::update / applyGain (mixer.cpp:34-47,134-159) in place on host rows: SSAT16((multipliers[row] * x) >> 16).
 * Multiplier 65536 leaves the data unchanged and 0 gives zeros (the reference transmits no block at all for 0). */
int msdr_op_amplifier(int device, const int32_t *multipliers, int16_t *data, uint32_t rows, uint32_t n, size_t stride);
/* AudioOutputAnalog's sample formatting (output_dac.cpp:143): 12-bit DAC code = ((int16 sample) + 32768) >> 4. */
int msdr_op_dac_codes(int device, const int16_t *in, uint16_t *out, uint32_t rows, uint32_t n, size_t stride);

/* ---- LMS automatic notch / noise reduction (SURVEY 8f rank 3): Minimal-SDR.ino:702-770 ------------------------------------------
 * The sketch runs it on p_dac between demodulation and queue_dac when ANR_on > 0 (1 = notch: output the LMS error, 2 = noise
 * reduction: output the prediction).  Stand-alone stateful operator on demodulated int16 audio [n_channels][stride], in place;
 * 64 taps, 512-entry delay line, float32 with the reference's double sub-expressions; bit-exact with the reference compiled
 * for the host.  Not fused into the receive chain kernel (whose biquads it would precede). */
typedef struct msdr_anr msdr_anr;
typedef struct msdr_anr_state {
  float d[512];   /* ANR_d, .ino:724 */
  float w[64];    /* ANR_w[0..63], .ino:725 */
  float lidx;     /* .ino:715 */
  float ngamma;   /* .ino:718 */
  int32_t in_idx; /* .ino:723 */
} msdr_anr_state;
int msdr_anr_create(msdr_anr **out, int device, uint32_t n_channels);
void msdr_anr_destroy(msdr_anr *anr);
int msdr_anr_set_stream(msdr_anr *anr, void *cuda_stream);
int msdr_anr_synchronize(msdr_anr *anr);
const char *msdr_anr_last_error(const msdr_anr *anr);
int msdr_anr_update(msdr_anr *anr, int mode, int16_t *data, uint32_t n_blocks, size_t stride);          /* host buffer, synchronous */
int msdr_anr_update_device(msdr_anr *anr, int mode, int16_t *d_data, uint32_t n_blocks, size_t stride);  /* device buffer, asynchronous */
int msdr_anr_get_state(msdr_anr *anr, uint32_t ch, msdr_anr_state *out);
int msdr_anr_set_state(msdr_anr *anr, uint32_t ch, const msdr_anr_state *in);
uint64_t msdr_anr_launch_count(const msdr_anr *anr);
/* The same inside a receive chain, where the sketch has it: between the demodulation switch and the biquads (ANR_on, .ino:99,702).
 * anr_on: 0 off, 1 notch, 2 noise reduction, per channel range.  Channels with ANR on (like channels in mode SYNCAM) are finished
 * beside the fused kernel on scratch copies; all other channels are untouched.  LMS state survives switching off and on. */
int msdr_chain_set_anr(msdr_chain *chain, uint32_t ch0, uint32_t nch, int anr_on);
int msdr_chain_get_anr_state(msdr_chain *chain, uint32_t ch, msdr_anr_state *out);
int msdr_chain_set_anr_state(msdr_chain *chain, uint32_t ch, const msdr_anr_state *in);

/* ---- synchronous-AM demodulator with PLL (SURVEY 8f rank 4): `case SYNCAM`, Minimal-SDR.ino:631-688 -------------------------------
 * Stand-alone stateful operator: the FIR-filtered I and Q streams [n_channels][stride] in, corr[0] narrowed to int16 out.
 * float32 with transcendental functions; parity with the reference compiled for a host is a tolerance (libm implementations
 * differ in the last ulp): <= 1e-5 relative RMS, tests/test_gpu_syncam.py.  A receive chain runs this operator for its channels
 * in mode SYNCAM (without MSDR_FLAG_AM_Q31) beside the fused kernel, on scratch copies of those channels (msdr_capi.cu). */
typedef struct msdr_syncam msdr_syncam;
int msdr_syncam_create(msdr_syncam **out, int device, uint32_t n_channels);
void msdr_syncam_destroy(msdr_syncam *sc);
int msdr_syncam_set_stream(msdr_syncam *sc, void *cuda_stream);
const char *msdr_syncam_last_error(const msdr_syncam *sc);
int msdr_syncam_update(msdr_syncam *sc, const int16_t *I, const int16_t *Q, int16_t *out, uint32_t n_blocks, size_t stride);
int msdr_syncam_update_device(msdr_syncam *sc, const int16_t *d_I, const int16_t *d_Q, int16_t *d_out, uint32_t n_blocks, size_t stride);
int msdr_syncam_get_state(msdr_syncam *sc, uint32_t ch, float *fil_out, float *omega2, float *phzerror);
int msdr_syncam_set_state(msdr_syncam *sc, uint32_t ch, float fil_out, float omega2, float phzerror);
int msdr_syncam_constants(float *omega_min, float *omega_max, float *g1, float *g2);
uint64_t msdr_syncam_launch_count(const msdr_syncam *sc);

const char *msdr_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MSDR_H */
