// msdr/Audio.h — C++ façade over the C ABI (msdr.h) with the reference's object API, batched over channels.
//
// The reference is an Arduino/Teensy sketch whose receive path is written against the Teensy Audio library:
// AudioStream objects joined by AudioConnection, `update()` once per 128-sample block, queues that couple the
// interrupt-driven graph to the foreground `demodulation()` (Minimal-SDR.ino:66-81, 518-775).  This header keeps those
// names and call shapes so the sketch's DSP code ports line by line, but every object carries a BATCH of independent
// channels and all arithmetic runs in the CUDA kernels behind msdr.h:
//
//   reference (one channel)                         here (n channels)
//   ------------------------------------------      -----------------------------------------------------------
//   audio_block_t { int16_t data[128]; }            audio_block_t { int16_t *data; }  = [channels][128], pinned host memory
//   AudioStream / AudioConnection / update_all()    same names; update_all() runs objects in construction order
//   AudioRecordQueue::begin/available/readBuffer/   same (53-deep ring, record_queue.h:33-55; drops when full,
//     freeBuffer, AudioPlayQueue::available/          record_queue.cpp:88-90)  /  same (32-deep, play_queue.h:33-50)
//     getBuffer/playBuffer
//   AudioFilterBiquad::setCoefficients/setLowpass…  same signatures (filter_biquad.h:43-149); update() = msdr_op_biquad, or a
//                                                   no-op pass-through when the object is bound to a Receiver (fused kernel)
//   AudioEffectFreqConv::direction/passthrough      same (freq_conv.h:36-56); update() = msdr_op_freq_conv
//   AudioFilterFIR::begin(coeffs, n)/end()          same (the Teensy Audio library's filter_fir.h, which the reference lists at
//                                                   src/Audio/Audio.h:96 but does not vendor); update() = msdr_op_fir_fast_q15
//   AudioProcessorUsageMax()/…MaxReset()            same (Minimal-SDR.ino:424-426); fed by the Receivers' device time per block
//   arm_fir_init_q15 + arm_fir_fast_q15 (x2),       Receiver::init_FIR / tune / demodulation(): ONE fused launch for the whole
//     mix loop, demod switch in demodulation()        batch, including the two biquad objects that follow queue_dac
//
// Errors keep the reference's conventions: missing input or bad stage => silently nothing (filter_biquad.cpp:41,86),
// arm_status codes from FIR init; CUDA failures are reported through last_status()/msdr_last_error().
// Not thread-safe; one host thread drives a Receiver (the reference has one foreground loop and one audio IRQ).
#ifndef MSDR_AUDIO_H
#define MSDR_AUDIO_H

#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../msdr.h"

namespace msdr {

#ifndef AUDIO_BLOCK_SAMPLES
#define AUDIO_BLOCK_SAMPLES MSDR_BLOCK_SAMPLES
#endif
#ifndef AUDIO_SAMPLE_RATE_EXACT
#define AUDIO_SAMPLE_RATE_EXACT 44117.64706 /* Teensy core constant the Audio library hard-wires */
#endif

enum { SYNCAM = MSDR_MODE_SYNCAM, AM = MSDR_MODE_AM, LSB = MSDR_MODE_LSB, USB = MSDR_MODE_USB, CW = MSDR_MODE_CW }; // stations.h:4

// One AudioStream block for the whole batch: data[c * AUDIO_BLOCK_SAMPLES + n].
struct audio_block_t {
  int16_t *data = nullptr;
  uint32_t channels = 0;
  uint16_t ref_count = 0;
  uint16_t memory_pool_index = 0;
};

class AudioConnection;

// Block pool: AudioMemory(n) of the reference, sized in batch blocks.
class AudioPool {
public:
  static AudioPool &instance() { static AudioPool p; return p; }
  void configure(uint32_t channels, unsigned blocks)
  {
    release_all();
    channels_ = channels;
    slab_ = static_cast<int16_t *>(msdr_host_alloc(sizeof(int16_t) * (size_t)blocks * channels * AUDIO_BLOCK_SAMPLES));
    blocks_.resize(slab_ ? blocks : 0);
    for (unsigned i = 0; i < blocks_.size(); ++i) {
      blocks_[i].data = slab_ + (size_t)i * channels * AUDIO_BLOCK_SAMPLES;
      blocks_[i].channels = channels;
      blocks_[i].ref_count = 0;
      blocks_[i].memory_pool_index = (uint16_t)i;
    }
    used_max_ = 0;
  }
  audio_block_t *allocate()
  {
    unsigned used = 0;
    audio_block_t *found = nullptr;
    for (auto &b : blocks_) {
      if (b.ref_count == 0 && !found) { found = &b; }
      if (b.ref_count) ++used;
    }
    if (!found) return nullptr; // reference: allocation failure => caller silently drops (freq_conv.cpp:64)
    found->ref_count = 1;
    if (used + 1 > used_max_) used_max_ = used + 1;
    return found;
  }
  static void release(audio_block_t *b) { if (b && b->ref_count) --b->ref_count; }
  uint32_t channels() const { return channels_; }
  unsigned usage_max() const { return used_max_; }
  ~AudioPool() { release_all(); }
private:
  void release_all() { if (slab_) msdr_host_free(slab_); slab_ = nullptr; blocks_.clear(); }
  std::vector<audio_block_t> blocks_;
  int16_t *slab_ = nullptr;
  uint32_t channels_ = 0;
  unsigned used_max_ = 0;
};
inline void AudioMemory(uint32_t channels, unsigned blocks) { AudioPool::instance().configure(channels, blocks); }
inline unsigned AudioMemoryUsageMax() { return AudioPool::instance().usage_max(); }
inline void AudioNoInterrupts() {} // updates are already serialised with setters (one host thread, one stream)
inline void AudioInterrupts() {}

// AudioStream: contract inferred from the reference's use (filter_biquad.cpp:39-81, freq_conv.cpp:37-113, mixer.cpp:141-156).
class AudioStream {
public:
  AudioStream(unsigned char ninput, audio_block_t **iqueue) : num_inputs(ninput), inputQueue(iqueue)
  {
    for (unsigned i = 0; i < num_inputs; ++i) inputQueue[i] = nullptr;
    registry().push_back(this);
  }
  virtual ~AudioStream()
  {
    auto &r = registry();
    for (size_t i = 0; i < r.size(); ++i)
      if (r[i] == this) { r.erase(r.begin() + (long)i); break; }
  }
  virtual void update(void) = 0;
  // one audio interrupt: every object in construction order (the Teensy core's update_all)
  static void update_all()
  {
    for (AudioStream *s : registry()) s->update();
  }
protected:
  static audio_block_t *allocate(void) { return AudioPool::instance().allocate(); }
  static void release(audio_block_t *block) { AudioPool::release(block); }
  audio_block_t *receiveReadOnly(unsigned int index = 0)
  {
    if (index >= num_inputs) return nullptr;
    audio_block_t *b = inputQueue[index];
    inputQueue[index] = nullptr;
    return b;
  }
  audio_block_t *receiveWritable(unsigned int index = 0)
  {
    audio_block_t *b = receiveReadOnly(index);
    if (b && b->ref_count > 1) { // shared: copy on write
      audio_block_t *c = allocate();
      if (c) memcpy(c->data, b->data, sizeof(int16_t) * (size_t)b->channels * AUDIO_BLOCK_SAMPLES);
      release(b);
      b = c;
    }
    return b;
  }
  void transmit(audio_block_t *block, unsigned char index = 0);
  unsigned char num_inputs;
  audio_block_t **inputQueue;
private:
  friend class AudioConnection;
  struct Dest { unsigned char src_index; AudioStream *dst; unsigned char dst_index; };
  std::vector<Dest> destinations;
  static std::vector<AudioStream *> &registry() { static std::vector<AudioStream *> r; return r; }
};

class AudioConnection {
public:
  AudioConnection(AudioStream &source, AudioStream &destination) { connect(source, 0, destination, 0); }
  AudioConnection(AudioStream &source, unsigned char sourceOutput, AudioStream &destination, unsigned char destinationInput)
  {
    connect(source, sourceOutput, destination, destinationInput);
  }
private:
  static void connect(AudioStream &s, unsigned char so, AudioStream &d, unsigned char di) { s.destinations.push_back({so, &d, di}); }
};

inline void AudioStream::transmit(audio_block_t *block, unsigned char index)
{
  for (const Dest &c : destinations) {
    if (c.src_index != index || c.dst_index >= c.dst->num_inputs) continue;
    if (c.dst->inputQueue[c.dst_index] == nullptr) {
      c.dst->inputQueue[c.dst_index] = block;
      block->ref_count++;
    }
  }
}

// ---- AudioRecordQueue (record_queue.{h,cpp}) ----------------------------------------------------------------------
class AudioRecordQueue : public AudioStream {
public:
  AudioRecordQueue(void) : AudioStream(1, inputQueueArray), userblock(nullptr), head(0), tail(0), enabled(0) {}
  void begin(void) { clear(); enabled = 1; }
  int available(void) { return head >= tail ? (int)(head - tail) : (int)(53 + head - tail); }
  void clear(void)
  {
    if (userblock) { release(userblock); userblock = nullptr; }
    uint32_t t = tail;
    while (t != head) { if (++t >= 53) t = 0; release(queue[t]); }
    tail = t;
  }
  int16_t *readBuffer(void)
  {
    if (userblock) return nullptr;
    uint32_t t = tail;
    if (t == head) return nullptr;
    if (++t >= 53) t = 0;
    userblock = queue[t];
    tail = t;
    return userblock->data;
  }
  void freeBuffer(void) { if (!userblock) return; release(userblock); userblock = nullptr; }
  void end(void) { enabled = 0; }
  virtual void update(void)
  {
    audio_block_t *block = receiveReadOnly();
    if (!block) return;
    if (!enabled) { release(block); return; }
    uint32_t h = head + 1;
    if (h >= 53) h = 0;
    if (h == tail) release(block); // ring full: newest block dropped silently (record_queue.cpp:88-90)
    else { queue[h] = block; head = h; }
  }
private:
  audio_block_t *inputQueueArray[1];
  audio_block_t *queue[53];
  audio_block_t *userblock;
  uint32_t head, tail, enabled;
};

// ---- AudioPlayQueue (play_queue.{h,cpp}) --------------------------------------------------------------------------
class AudioPlayQueue : public AudioStream {
public:
  AudioPlayQueue(void) : AudioStream(0, nullptr), userblock(nullptr), head(0), tail(0) {}
  bool available(void)
  {
    if (userblock) return true;
    userblock = allocate();
    return userblock != nullptr;
  }
  int16_t *getBuffer(void)
  {
    if (userblock) return userblock->data;
    userblock = allocate();
    return userblock ? userblock->data : nullptr;
  }
  // the reference spins while the ring is full (play_queue.cpp:56); a host harness has no concurrent consumer, so a
  // full ring drains one block through the graph first
  void playBuffer(void)
  {
    if (!userblock) return;
    uint32_t h = head + 1;
    if (h >= 32) h = 0;
    if (h == tail) AudioStream::update_all();
    queue[h] = userblock;
    head = h;
    userblock = nullptr;
  }
  virtual void update(void)
  {
    uint32_t t = tail;
    if (t == head) return;
    if (++t >= 32) t = 0;
    audio_block_t *block = queue[t];
    tail = t;
    transmit(block);
    release(block);
  }
private:
  audio_block_t *queue[32];
  audio_block_t *userblock;
  uint32_t head, tail;
};

// ---- a sink that keeps the last block (stands in for AudioOutputAnalog, which is Teensy hardware) ------------------
class AudioCapture : public AudioStream {
public:
  AudioCapture(void) : AudioStream(1, inputQueueArray) {}
  virtual void update(void)
  {
    audio_block_t *b = receiveReadOnly();
    if (!b) return;
    last.assign(b->data, b->data + (size_t)b->channels * AUDIO_BLOCK_SAMPLES);
    ++blocks;
    release(b);
  }
  std::vector<int16_t> last;
  unsigned blocks = 0;
private:
  audio_block_t *inputQueueArray[1];
};

class Receiver;

// ---- AudioFilterBiquad (filter_biquad.{h,cpp}) --------------------------------------------------------------------
class AudioFilterBiquad : public AudioStream {
public:
  AudioFilterBiquad(void) : AudioStream(1, inputQueueArray) { memset(definition, 0, sizeof(definition)); }
  virtual void update(void);
  void setCoefficients(uint32_t stage, const int *coefficients);
  void setCoefficients(uint32_t stage, const double *coefficients)
  {
    int coef[5];
    for (int i = 0; i < 5; ++i) coef[i] = (int)(coefficients[i] * 1073741824.0);
    setCoefficients(stage, coef);
  }
  // http://www.musicdsp.org/files/Audio-EQ-Cookbook.txt, as filter_biquad.h:56-149
  void setLowpass(uint32_t stage, float frequency, float q = 0.7071f)
  {
    double w0, alpha, cosW0, scale; prep(frequency, q, w0, alpha, cosW0, scale);
    int coef[5] = {(int)(((1.0 - cosW0) / 2.0) * scale), (int)((1.0 - cosW0) * scale), 0, (int)((-2.0 * cosW0) * scale), (int)((1.0 - alpha) * scale)};
    coef[2] = coef[0];
    setCoefficients(stage, coef);
  }
  void setHighpass(uint32_t stage, float frequency, float q = 0.7071f)
  {
    double w0, alpha, cosW0, scale; prep(frequency, q, w0, alpha, cosW0, scale);
    int coef[5] = {(int)(((1.0 + cosW0) / 2.0) * scale), (int)(-(1.0 + cosW0) * scale), 0, (int)((-2.0 * cosW0) * scale), (int)((1.0 - alpha) * scale)};
    coef[2] = coef[0];
    setCoefficients(stage, coef);
  }
  void setBandpass(uint32_t stage, float frequency, float q = 1.0f)
  {
    double w0, alpha, cosW0, scale; prep(frequency, q, w0, alpha, cosW0, scale);
    int coef[5] = {(int)(alpha * scale), 0, (int)((-alpha) * scale), (int)((-2.0 * cosW0) * scale), (int)((1.0 - alpha) * scale)};
    setCoefficients(stage, coef);
  }
  void setNotch(uint32_t stage, float frequency, float q = 1.0f)
  {
    double w0, alpha, cosW0, scale; prep(frequency, q, w0, alpha, cosW0, scale);
    int coef[5] = {(int)scale, (int)((-2.0 * cosW0) * scale), 0, (int)((-2.0 * cosW0) * scale), (int)((1.0 - alpha) * scale)};
    coef[2] = coef[0];
    setCoefficients(stage, coef);
  }
  void setLowShelf(uint32_t stage, float frequency, float gain, float slope = 1.0f)
  {
    double a, sinsq, aMinus, aPlus; shelf(frequency, gain, slope, a, sinsq, aMinus, aPlus);
    const double scale = 1073741824.0 / ((a + 1.0) + aMinus + sinsq);
    int coef[5] = {(int)(a * ((a + 1.0) - aMinus + sinsq) * scale), (int)(2.0 * a * ((a - 1.0) - aPlus) * scale),
                   (int)(a * ((a + 1.0) - aMinus - sinsq) * scale), (int)(-2.0 * ((a - 1.0) + aPlus) * scale), (int)(((a + 1.0) + aMinus - sinsq) * scale)};
    setCoefficients(stage, coef);
  }
  void setHighShelf(uint32_t stage, float frequency, float gain, float slope = 1.0f)
  {
    double a, sinsq, aMinus, aPlus; shelf(frequency, gain, slope, a, sinsq, aMinus, aPlus);
    const double scale = 1073741824.0 / ((a + 1.0) - aMinus + sinsq);
    int coef[5] = {(int)(a * ((a + 1.0) + aMinus + sinsq) * scale), (int)(-2.0 * a * ((a - 1.0) + aPlus) * scale),
                   (int)(a * ((a + 1.0) + aMinus - sinsq) * scale), (int)(2.0 * ((a - 1.0) - aPlus) * scale), (int)(((a + 1.0) - aMinus - sinsq) * scale)};
    setCoefficients(stage, coef);
  }
  int last_status() const { return status_; }
private:
  friend class Receiver;
  static void prep(float frequency, float q, double &w0, double &alpha, double &cosW0, double &scale)
  {
    w0 = frequency * (2 * 3.141592654 / AUDIO_SAMPLE_RATE_EXACT);
    alpha = sin(w0) / ((double)q * 2.0);
    cosW0 = cos(w0);
    scale = 1073741824.0 / (1.0 + alpha);
  }
  static void shelf(float frequency, float gain, float slope, double &a, double &sinsq, double &aMinus, double &aPlus)
  {
    a = pow(10.0, gain / 40.0);
    const double w0 = frequency * (2 * 3.141592654 / AUDIO_SAMPLE_RATE_EXACT);
    const double sinW0 = sin(w0), cosW0 = cos(w0);
    sinsq = sinW0 * sqrt((pow(a, 2.0) + 1.0) * (1.0 / slope - 1.0) + 2.0 * a);
    aMinus = (a - 1.0) * cosW0;
    aPlus = (a + 1.0) * cosW0;
  }
  int32_t definition[32];          // one cascade shared by every channel (stand-alone use), filter_biquad.h:152 layout
  std::vector<int32_t> per_channel; // [channels][32] working copy carrying each channel's history
  audio_block_t *inputQueueArray[1];
  Receiver *bound_ = nullptr;      // when set: the fused kernel runs this cascade, update() only forwards the block
  int object_ = 0;
  int status_ = 0;
};

// ---- AudioEffectFreqConv (freq_conv.{h,cpp}); the oscillator tables are members instead of undefined externs ---------
class AudioEffectFreqConv : public AudioStream {
public:
  AudioEffectFreqConv() : AudioStream(2, inputQueueArray), dir(0), pass(1)
  {
    for (int i = 0; i < AUDIO_BLOCK_SAMPLES; ++i) { // fs/4 default: cos -> Osc_Q, sin -> Osc_I
      static const int16_t c4[4] = {32767, 0, -32767, 0}, s4[4] = {0, 32767, 0, -32767};
      Osc_Q_buffer_i[i] = c4[i & 3];
      Osc_I_buffer_i[i] = s4[i & 3];
    }
  }
  void direction(bool d) { dir = d; }
  void passthrough(bool p) { pass = p; }
  int16_t Osc_Q_buffer_i[AUDIO_BLOCK_SAMPLES];
  int16_t Osc_I_buffer_i[AUDIO_BLOCK_SAMPLES];
  int device = 0;
  virtual void update(void)
  {
    audio_block_t *blockI = receiveWritable(0), *blockQ = receiveWritable(1);
    if (!blockI) { if (blockQ) release(blockQ); return; }
    if (!blockQ) { release(blockI); return; }
    if (pass) // pass == 0 forwards unchanged (freq_conv.cpp:49-56)
      msdr_op_freq_conv(device, dir, 1, blockI->data, blockQ->data, Osc_I_buffer_i, Osc_Q_buffer_i, blockI->channels, AUDIO_BLOCK_SAMPLES,
                        AUDIO_BLOCK_SAMPLES);
    transmit(blockI, 0);
    transmit(blockQ, 1);
    release(blockI);
    release(blockQ);
  }
private:
  audio_block_t *inputQueueArray[2];
  bool dir, pass;
};

// ---- AudioFilterFIR: the Teensy Audio library's FIR object (filter_fir.h; listed at src/Audio/Audio.h:96, not vendored by the
// reference).  Call shape from the library's documentation: begin(coefficients, count) binds a q15 table (borrowed pointer,
// like arm_fir_init_q15.c:103) and zeroes the delay line; FIR_PASSTHRU forwards blocks unchanged; end() or a failed init (odd
// count, arm_fir_init_q15.c:93-96; more than FIR_MAX_COEFFS) leaves the object without coefficients and it then consumes its
// input and transmits nothing.  update() is arm_fir_fast_q15 (arm_fir_fast_q15.c:60-329) on every channel of the batch block.
#ifndef FIR_MAX_COEFFS
#define FIR_MAX_COEFFS 200
#endif
#define FIR_PASSTHRU ((const short *)1)
class AudioFilterFIR : public AudioStream {
public:
  AudioFilterFIR(void) : AudioStream(1, inputQueueArray), coeff_p(nullptr), n_coeffs(0) {}
  void begin(const short *cp, int n)
  {
    coeff_p = cp;
    n_coeffs = n;
    history.clear(); // arm_fir_init_q15 zeroes pState
    if (coeff_p && coeff_p != FIR_PASSTHRU && (n > FIR_MAX_COEFFS || n < 2 || (n & 1))) coeff_p = nullptr;
  }
  void end(void) { coeff_p = nullptr; }
  int device = 0;
  int last_status() const { return status_; }
  virtual void update(void)
  {
    audio_block_t *block = receiveReadOnly();
    if (!block) return;
    if (!coeff_p) { release(block); return; }
    if (coeff_p == FIR_PASSTHRU) { transmit(block); release(block); return; }
    audio_block_t *b_new = allocate();
    if (b_new) {
      const size_t hn = (size_t)block->channels * (size_t)(n_coeffs - 1);
      if (history.size() != hn) history.assign(hn, 0);
      status_ = msdr_op_fir_fast_q15(device, (uint16_t)n_coeffs, coeff_p, history.data(), block->data, b_new->data, block->channels,
                                     AUDIO_BLOCK_SAMPLES, AUDIO_BLOCK_SAMPLES);
      transmit(b_new);
      release(b_new);
    }
    release(block);
  }
private:
  const short *coeff_p;
  int n_coeffs;
  std::vector<int16_t> history; // [channels][n_coeffs - 1]: the head of each channel's pState (arm_fir_fast_q15.c:296-327)
  audio_block_t *inputQueueArray[1];
  int status_ = 0;
};

// ---- AudioAmplifier (mixer.{h,cpp}): the sketch's amp_adc / amp_dac ---------------------------------------------------------
class AudioAmplifier : public AudioStream {
public:
  AudioAmplifier(void) : AudioStream(1, inputQueueArray), multiplier(65536) {}
  void gain(float n) { multiplier = msdr_amp_gain_multiplier(n); } // mixer.h:75-79
  int device = 0;
  virtual void update(void)
  {
    if (multiplier == 0) { // zero gain: discard the input, transmit nothing (mixer.cpp:139-142)
      audio_block_t *b = receiveReadOnly(0);
      if (b) release(b);
      return;
    }
    audio_block_t *block = multiplier == 65536 ? receiveReadOnly(0) : receiveWritable(0);
    if (!block) return;
    if (multiplier != 65536) {
      std::vector<int32_t> m(block->channels, multiplier);
      msdr_op_amplifier(device, m.data(), block->data, block->channels, AUDIO_BLOCK_SAMPLES, AUDIO_BLOCK_SAMPLES);
    }
    transmit(block);
    release(block);
  }
private:
  int32_t multiplier;
  audio_block_t *inputQueueArray[1];
};

// ---- Frontend: adc1's DC-blocking filter + amp_adc + AGC() for a batch of channels in one object --------------------------
// (AudioInputAnalog is Teensy hardware; what it does to the samples, input_adc.cpp:198-212, and what the sketch does with
// them before demodulation(), .ino:76-78,445-515,534, is this.)  update() = one or more audio blocks of raw ADC codes.
class Frontend {
public:
  explicit Frontend(uint32_t channels, int device = 0, float AGC_start = 0.25f, float AGC_Max = 40.0f, int AGC_on = 1) : n(channels), fe(nullptr)
  {
    if (msdr_frontend_create(&fe, device, channels, AGC_start, AGC_Max, AGC_on) != MSDR_OK) fe = nullptr;
  }
  ~Frontend() { msdr_frontend_destroy(fe); }
  Frontend(const Frontend &) = delete;
  Frontend &operator=(const Frontend &) = delete;
  bool ok() const { return fe != nullptr; }
  int begin(uint16_t first_reading) { return msdr_frontend_preset(fe, 0, n, first_reading); } // AudioInputAnalog::init, input_adc.cpp:59-63
  int update(const uint16_t *codes, int16_t *p_adc, uint32_t n_blocks, size_t stride) { return msdr_frontend_update(fe, codes, p_adc, n_blocks, stride); }
  float AGC_val(uint32_t channel = 0) const
  {
    msdr_frontend_state st;
    return msdr_frontend_get_state(fe, channel, &st) == MSDR_OK ? st.agc_val : 0.0f;
  }
  msdr_frontend *handle() { return fe; }
private:
  uint32_t n;
  msdr_frontend *fe;
};

// ---- Receiver: the sketch's FIR instances + demodulation() for a batch of channels, fused with the two biquads --------
class Receiver {
public:
  Receiver(uint32_t n_channels, int device = 0, uint32_t max_taps = 0, uint32_t flags = 0) : n_(n_channels)
  {
    status_ = msdr_chain_create(&chain_, device, n_channels, max_taps, flags);
    live().push_back(this);
  }
  ~Receiver()
  {
    auto &r = live();
    for (size_t i = 0; i < r.size(); ++i)
      if (r[i] == this) { r.erase(r.begin() + (long)i); break; }
    msdr_chain_destroy(chain_);
  }
  static std::vector<Receiver *> &live() { static std::vector<Receiver *> r; return r; }
  Receiver(const Receiver &) = delete;
  Receiver &operator=(const Receiver &) = delete;
  bool ok() const { return chain_ != nullptr; }
  int last_status() const { return status_; }
  const char *last_error() const { return msdr_last_error(chain_); }
  msdr_chain *handle() { return chain_; }

  // AudioConnection patchCord2(queue_dac, biquad1_dac); patchCord4a(biquad1_dac, biquad2_dac)  (Minimal-SDR.ino:77,79):
  // the two objects that follow queue_dac are executed by the fused kernel
  void bind(AudioFilterBiquad &biquad1, AudioFilterBiquad &biquad2)
  {
    biquad1.bound_ = this; biquad1.object_ = 0;
    biquad2.bound_ = this; biquad2.object_ = 1;
    for (int obj = 0; obj < 2; ++obj) { // replay coefficients set before binding
      AudioFilterBiquad &b = obj ? biquad2 : biquad1;
      for (uint32_t s = 0; s < 4; ++s) {
        const int32_t *d = b.definition + 8 * s;
        if (s == 0 || (b.definition[8 * (s - 1) + 7] & 0x80000000)) {
          int coef[5] = {d[0], d[1], d[2], -d[3], -d[4]};
          if (s == 0 && !(d[0] | d[1] | d[2] | d[3] | d[4])) continue;
          status_ = msdr_biquad_set_coefficients(chain_, obj, 0, n_, s, coef);
        }
      }
    }
  }
  // global `mode` + init_FIR() (Minimal-SDR.ino:901-930) for a channel range; tables are the caller's (the sketch's constants)
  int set_mode(int mode, uint32_t ch0 = 0, uint32_t nch = ~0u) { return status_ = msdr_chain_set_mode(chain_, ch0, cnt(ch0, nch), mode); }
  // ANR_on of the sketch (.ino:99): 0 off, 1 LMS notch, 2 LMS noise reduction, between demodulation and the biquads
  int set_ANR(int ANR_on, uint32_t ch0 = 0, uint32_t nch = ~0u) { return status_ = msdr_chain_set_anr(chain_, ch0, cnt(ch0, nch), ANR_on); }
  int init_FIR(uint16_t numTaps, const int16_t *cI, const int16_t *cQ, uint32_t ch0 = 0, uint32_t nch = ~0u)
  {
    return status_ = msdr_fir_init_q15(chain_, ch0, cnt(ch0, nch), numTaps, cI, cQ);
  }
  // calc_demod_filter(): in-place rewrite of the bound table (Minimal-SDR.ino:221-223)
  int set_FIR_coefficients(const int16_t *cI, const int16_t *cQ, uint32_t ch0 = 0, uint32_t nch = ~0u)
  {
    return status_ = msdr_fir_set_coefficients(chain_, ch0, cnt(ch0, nch), cI, cQ);
  }
  // unsigned long demodulation(void) (Minimal-SDR.ino:518-775): one block from queue_adc to queue_dac, same gates
  // (:520-521); returns 1 when a block was processed.  The block reaching queue_dac already carries both biquads.
  unsigned long demodulation(AudioRecordQueue &queue_adc, AudioPlayQueue &queue_dac)
  {
    if (queue_dac.available() == false) return 0;
    if (queue_adc.available() < 1) return 0;
    int16_t *p_adc = queue_adc.readBuffer();
    int16_t *p_dac = queue_dac.getBuffer();
    status_ = msdr_chain_update(chain_, p_adc, p_dac, 1, AUDIO_BLOCK_SAMPLES);
    queue_adc.freeBuffer();
    queue_dac.playBuffer();
    return status_ == MSDR_OK ? 1 : 0;
  }
  // many blocks at once on caller buffers [channels][stride]
  int update(const int16_t *in, int16_t *out, uint32_t n_blocks, size_t stride) { return status_ = msdr_chain_update(chain_, in, out, n_blocks, stride); }
  // adc1 -> amp_adc -> queue_adc -> demodulation() with AGC(p_adc) on every block (Minimal-SDR.ino:76-78,445-515) in this one object:
  // begin_frontend() sets up every channel's DC block, amplifier and AGC (AGC_start, AGC_Max, AGC_on of .ino:94-100), update_adc()
  // takes raw uint16 ADC codes [channels][stride] and returns audio, AGC_val(ch) is the sketch's global of that channel
  int begin_frontend(float agc_start = 0.25f, float agc_max = 40.0f, int agc_on = 1)
  {
    return status_ = msdr_chain_enable_frontend(chain_, agc_start, agc_max, agc_on);
  }
  int update_adc(const uint16_t *codes, int16_t *out, uint32_t n_blocks, size_t stride)
  {
    return status_ = msdr_chain_update_adc(chain_, codes, out, n_blocks, stride);
  }
  float AGC_val(uint32_t ch)
  {
    msdr_frontend_state s{};
    status_ = msdr_chain_get_frontend_state(chain_, ch, &s);
    return s.agc_val;
  }
  // checkpoint / resume of a channel range (msdr_chain_snapshot / msdr_chain_restore): snapshot() fills `blob` with everything channels
  // [ch0, ch0+nch) carry, restore() gives channels [ch0, ch0+n) the state of snapshot channels [first, first+n) (n = ~0u: the rest)
  int snapshot(std::vector<uint8_t> &blob, uint32_t ch0 = 0, uint32_t nch = ~0u)
  {
    blob.resize(msdr_chain_snapshot_bytes(chain_, cnt(ch0, nch)));
    return status_ = msdr_chain_snapshot(chain_, ch0, cnt(ch0, nch), blob.data(), blob.size());
  }
  int restore(const std::vector<uint8_t> &blob, uint32_t ch0 = 0, uint32_t first = 0, uint32_t n = ~0u)
  {
    if (n == ~0u) {
      uint32_t total = 0;
      if ((status_ = msdr_snapshot_info(blob.data(), blob.size(), &total, nullptr, nullptr)) != MSDR_OK) return status_;
      n = total - first;
    }
    return status_ = msdr_chain_restore(chain_, ch0, blob.data(), blob.size(), first, n);
  }
  uint32_t channels() const { return n_; }
private:
  uint32_t cnt(uint32_t ch0, uint32_t nch) const { return nch == ~0u ? n_ - ch0 : nch; }
  msdr_chain *chain_ = nullptr;
  uint32_t n_;
  int status_;
};

// AudioProcessorUsageMax() / AudioProcessorUsageMaxReset() / AudioProcessorUsage() of the Teensy core, as the sketch prints them
// (Minimal-SDR.ino:424-426): processing time as a percentage of the block period.  Here: the largest figure over the live
// Receivers, each = device time of an update / real-time duration of its blocks at AudioProcessorUsageSampleRate() (the
// sketch's pdb_freq_actual; default AUDIO_SAMPLE_RATE_EXACT).  Counting starts with the first call.
inline double &AudioProcessorUsageSampleRate() { static double fs = AUDIO_SAMPLE_RATE_EXACT; return fs; }
inline float AudioProcessorUsage_(bool want_max)
{
  float best = 0.0f;
  for (Receiver *r : Receiver::live()) {
    float last = 0.0f, mx = 0.0f;
    if (r->ok() && msdr_chain_processor_usage(r->handle(), AudioProcessorUsageSampleRate(), &last, &mx) == MSDR_OK)
      best = std::fmax(best, want_max ? mx : last);
  }
  return best;
}
inline float AudioProcessorUsage() { return AudioProcessorUsage_(false); }
inline float AudioProcessorUsageMax() { return AudioProcessorUsage_(true); }
inline void AudioProcessorUsageMaxReset()
{
  for (Receiver *r : Receiver::live())
    if (r->ok()) msdr_chain_processor_usage_max_reset(r->handle());
}

inline void AudioFilterBiquad::setCoefficients(uint32_t stage, const int *coefficients)
{
  if (stage >= 4) return; // filter_biquad.cpp:86
  int32_t *dest = definition + (stage << 3);
  if (stage > 0) *(dest - 1) |= 0x80000000;
  dest[0] = coefficients[0]; dest[1] = coefficients[1]; dest[2] = coefficients[2];
  dest[3] = coefficients[3] * -1; dest[4] = coefficients[4] * -1;
  dest[7] &= 0x80000000;
  for (size_t c = 0; c * 32 < per_channel.size(); ++c) { // same edit on every channel's working copy: history kept
    int32_t *d = per_channel.data() + c * 32 + (stage << 3);
    if (stage > 0) *(d - 1) |= 0x80000000;
    memcpy(d, dest, 5 * sizeof(int32_t));
    d[7] &= 0x80000000;
  }
  if (bound_) status_ = msdr_biquad_set_coefficients(bound_->handle(), object_, 0, bound_->channels(), stage, coefficients);
}

inline void AudioFilterBiquad::update(void)
{
  audio_block_t *block = receiveWritable();
  if (!block) return;
  if (!bound_) {
    if (per_channel.size() != (size_t)block->channels * 32) {
      per_channel.resize((size_t)block->channels * 32);
      for (uint32_t c = 0; c < block->channels; ++c) memcpy(per_channel.data() + (size_t)c * 32, definition, sizeof(definition));
    }
    status_ = msdr_op_biquad(0, per_channel.data(), block->data, block->channels, AUDIO_BLOCK_SAMPLES, AUDIO_BLOCK_SAMPLES);
  }
  transmit(block);
  release(block);
}

} // namespace msdr
#endif // MSDR_AUDIO_H
