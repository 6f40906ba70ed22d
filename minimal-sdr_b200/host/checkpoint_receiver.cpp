// checkpoint_receiver.cpp — stop a stream, save the Receiver to a file, restore it into a new Receiver and carry on: the output equals
// that of one Receiver that never stopped (Receiver::snapshot / Receiver::restore on msdr_chain_snapshot / msdr_chain_restore).
//   checkpoint_receiver <channels> <blocks> <stop_block> <numTaps> <tables.bin> <in.bin> <checkpoint.bin> <out.bin>
// tables.bin: int16 cI[numTaps], cQ[numTaps].  in.bin: int16 IF samples [channels][blocks*128].  Channels alternate AM / USB / LSB / CW
// on the given table, ANR 2 on every eighth; blocks [0, stop_block) run on the first Receiver, which is then saved to checkpoint.bin and
// destroyed; a second Receiver, configured by nothing but the file, runs blocks [stop_block, blocks).  out.bin: int16 audio.
// stop_block 0: one Receiver runs every block and nothing is saved (the uninterrupted run to compare with).
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "msdr/Audio.h"
using namespace msdr;

AudioFilterBiquad biquad1_dac, biquad2_dac;

int main(int argc, char **argv)
{
  if (argc != 9) return 2;
  const uint32_t C = (uint32_t)atoi(argv[1]), NB = (uint32_t)atoi(argv[2]), stop = (uint32_t)atoi(argv[3]), T = (uint32_t)atoi(argv[4]);
  if (stop >= NB) return 2;
  const size_t L = (size_t)NB * AUDIO_BLOCK_SAMPLES;
  std::vector<int16_t> taps(2 * (size_t)T), in((size_t)C * L), out((size_t)C * L);
  FILE *f = fopen(argv[5], "rb");
  if (!f || fread(taps.data(), 2, taps.size(), f) != taps.size()) return 2;
  fclose(f);
  f = fopen(argv[6], "rb");
  if (!f || fread(in.data(), 2, in.size(), f) != in.size()) return 2;
  fclose(f);

  {
    Receiver rx(C);
    if (!rx.ok()) { fprintf(stderr, "%s\n", rx.last_error()); return 3; }
    biquad1_dac.setLowpass(0, 3000.0f, 0.7071f);
    biquad2_dac.setNotch(0, 5514.7f, 15.0f);
    rx.bind(biquad1_dac, biquad2_dac);
    rx.init_FIR((uint16_t)T, taps.data(), taps.data() + T);
    const int modes[4] = {AM, USB, LSB, CW};
    for (uint32_t c = 0; c < C; ++c) rx.set_mode(modes[c % 4], c, 1);
    for (uint32_t c = 0; c < C; c += 8) rx.set_ANR(2, c, 1);
    if (rx.update(in.data(), out.data(), stop ? stop : NB, L) != MSDR_OK) { fprintf(stderr, "update: %s\n", rx.last_error()); return 4; }
    if (stop == 0) {
      f = fopen(argv[8], "wb"); if (!f) return 2; fwrite(out.data(), 2, out.size(), f); fclose(f);
      printf("checkpoint_receiver: %u channels, %u blocks uninterrupted\n", C, NB);
      return 0;
    }
    std::vector<uint8_t> blob;
    if (rx.snapshot(blob) != MSDR_OK) { fprintf(stderr, "snapshot: %s\n", rx.last_error()); return 4; }
    f = fopen(argv[7], "wb");
    if (!f || fwrite(blob.data(), 1, blob.size(), f) != blob.size()) return 2;
    fclose(f);
  } // the first Receiver is gone

  f = fopen(argv[7], "rb");
  if (!f) return 2;
  fseek(f, 0, SEEK_END);
  std::vector<uint8_t> blob((size_t)ftell(f));
  fseek(f, 0, SEEK_SET);
  if (fread(blob.data(), 1, blob.size(), f) != blob.size()) return 2;
  fclose(f);
  Receiver rx2(C);
  if (!rx2.ok()) { fprintf(stderr, "%s\n", rx2.last_error()); return 3; }
  if (rx2.restore(blob) != MSDR_OK) { fprintf(stderr, "restore: %s\n", rx2.last_error()); return 4; }
  const size_t off = (size_t)stop * AUDIO_BLOCK_SAMPLES;
  if (rx2.update(in.data() + off, out.data() + off, NB - stop, L) != MSDR_OK) { fprintf(stderr, "update: %s\n", rx2.last_error()); return 4; }
  f = fopen(argv[8], "wb"); if (!f) return 2; fwrite(out.data(), 2, out.size(), f); fclose(f);
  printf("checkpoint_receiver: %u channels, %u + %u blocks, %zu-byte checkpoint\n", C, stop, NB - stop, blob.size());
  return 0;
}
