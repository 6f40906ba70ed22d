// adc_receiver.cpp — the sketch's receive path from the ADC on the façade as ONE object: Receiver::begin_frontend() puts the DC
// block, amp_adc and AGC() in front of demodulation() and the two biquads (Minimal-SDR.ino:76-81,445-515), update_adc() takes raw codes.
//   adc_receiver <channels> <blocks> <numTaps> <tables.bin> <codes.bin> <out.bin> <out_agc.bin>
// tables.bin: int16 cI[numTaps], cQ[numTaps] (every channel AM).  codes.bin: uint16 [channels][blocks*128].  The first three blocks go in
// one update each, the rest in one call.  out.bin: int16 audio; out_agc.bin: float AGC_val of every channel after the last block.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "msdr/Audio.h"
using namespace msdr;

AudioFilterBiquad biquad1_dac, biquad2_dac;

int main(int argc, char **argv)
{
  if (argc != 8) return 2;
  const uint32_t C = (uint32_t)atoi(argv[1]), NB = (uint32_t)atoi(argv[2]), T = (uint32_t)atoi(argv[3]);
  const size_t L = (size_t)NB * AUDIO_BLOCK_SAMPLES;
  std::vector<int16_t> taps(2 * (size_t)T), out((size_t)C * L);
  std::vector<uint16_t> codes((size_t)C * L);
  FILE *f = fopen(argv[4], "rb");
  if (!f || fread(taps.data(), 2, taps.size(), f) != taps.size()) return 2;
  fclose(f);
  f = fopen(argv[5], "rb");
  if (!f || fread(codes.data(), 2, codes.size(), f) != codes.size()) return 2;
  fclose(f);

  Receiver rx(C);
  if (!rx.ok()) { fprintf(stderr, "%s\n", rx.last_error()); return 3; }
  biquad1_dac.setLowpass(0, 3000.0f, 0.7071f);
  biquad2_dac.setNotch(0, 5514.7f, 15.0f);
  rx.bind(biquad1_dac, biquad2_dac);
  rx.set_mode(AM);
  rx.init_FIR((uint16_t)T, taps.data(), taps.data() + T);
  if (rx.begin_frontend(0.25f, 40.0f, 1) != MSDR_OK) { fprintf(stderr, "%s\n", rx.last_error()); return 3; }
  uint32_t b = 0;
  for (; b < NB && b < 3; ++b)
    if (rx.update_adc(codes.data() + (size_t)b * AUDIO_BLOCK_SAMPLES, out.data() + (size_t)b * AUDIO_BLOCK_SAMPLES, 1, L) != MSDR_OK) break;
  if (b == 3 && NB > 3) rx.update_adc(codes.data() + 3 * AUDIO_BLOCK_SAMPLES, out.data() + 3 * AUDIO_BLOCK_SAMPLES, NB - 3, L);
  if (rx.last_status() != MSDR_OK) { fprintf(stderr, "update_adc: %s\n", rx.last_error()); return 4; }
  std::vector<float> agc(C);
  for (uint32_t c = 0; c < C; ++c) agc[c] = rx.AGC_val(c);
  f = fopen(argv[6], "wb"); if (!f) return 2; fwrite(out.data(), 2, out.size(), f); fclose(f);
  f = fopen(argv[7], "wb"); if (!f) return 2; fwrite(agc.data(), 4, agc.size(), f); fclose(f);
  printf("adc_receiver: %u channels x %u blocks, last kernel: %s\n", C, NB, msdr_chain_last_kernel(rx.handle()));
  return 0;
}
