// msdr_chain_v6.cu — K1d: the fused receive chain for FEW channels with nothing leaving the SM: one persistent CTA owns a block of 32
// channels that share a tap table and walks it through time.
//
//   int16 IF samples -> [fs/4 mix folded into the byte planes] -> FIR pair as int8 Toeplitz GEMMs on tcgen05.mma (exact mod 2^32,
//   msdr_fir_tc.cu) -> >>15, SSAT16 -> SSB sum / AM envelope -> biquad object 1 -> biquad object 2 -> int16 audio
//
// Reference semantics: Minimal-SDR.ino:546-558 (mix), arm_fir_fast_q15.c:60-329 (FIR), Minimal-SDR.ino:589-628 (demod),
// filter_biquad.cpp:33-82 (biquad).
//
// 4096 channels are 128 warps of serial biquad recurrence, one per SM, and a tensor-core tile has 128 rows.  msdr_chain_v4.cu squares
// the two with FIR producers that fill 128-channel tiles for any SM's chains and hand them over through global memory (write-back,
// readiness counters, a load back through L2: ~10 % of the launch is fill and drain, the chains wait 9 % of their time).  Here the 128
// rows of a tile are TIME instead: row (q, c) = channel c of 16, time block q of 8, and the tile's output is 16 channels x 256
// consecutive samples.  The A operand needs no copies for that.  Its byte planes are kept as plain time series per 8-channel group,
//   plane[unit u of 16 window words][8-channel group hh][channel i][16 bytes],
// and the canonical no-swizzle K-major layout is pure address arithmetic: K-adjacent core matrices 256 B apart (the next unit),
// M-adjacent 8-row groups 128 B apart.  Row group 2 q + hh then starts at unit q, i.e. every time block reads the window that ends at
// its own 16 new words - the rows overlap in memory, each sample is converted once.  N = 32 (the first 32 columns of the same Toeplitz
// operand the other kernels use, read in place through the descriptor strides).
//
// A group block is two half blocks of 16 same-table channels (a tile each), each half with its own Toeplitz operand; the plan pairs a
// half with an envelope demodulator (a square root per sample) with an SSB half, so that every CTA carries the same load.
//
// 16 warps (13 used), roles by warp id (warp id % 4 = SM sub-partition):
//   7        load      cp.async (LDGSTS) of a tile's raw rows (16 rows x 512 B, gathered through the row map) into a 2-stage staging ring
//   14, 15   convert   (row, unit) tasks: raw int16 -> fs/4 sign fold -> four byte planes in one of three operand buffers; the window tail
//                      of the same half's previous tile is copied in front (16-byte copies), the carried history at sample 0
//   6        MMA       one elected lane: 2 branches x 4 byte-plane products x K/32 MMAs (M128 N32 K32) per tile; two tiles live in TMEM
//   0-3      epilogue  TMEM lane = (time block, channel); per 8-column pass: tcgen05.ld, recombine, >>15, SSAT16, demodulate -> scratch;
//                      then TMEM is handed back and the 64 bytes go into the span buffer (32 channels x 256 samples, two of them)
//   10       FF1       lane = channel: span buffer -> e[n] of object 1 (the input-side products of the stage) into a slot of ring 1
//   4        chain A   recurrence of object 1 over the slot, results in place over the consumed e[n] words
//   11       FF2       A's results -> e[n] of object 2 into a slot of ring 2
//   5        chain B   recurrence of object 2, in place
//   9        store     ring-2 slot -> `out`
// Chain A, chain B, FF1 and FF2 each have a sub-partition of their own; everything else is light (a CTA produces only what its own 32
// channels consume).  DRAM traffic is the algorithmic 2 B in + 2 B out per sample.  Loops over column passes and sample groups are kept
// rolled on purpose: the kernel is sensitive to its instruction-cache footprint (DESIGN.md 6, K1d).
#include <cstdlib>
#include "msdr_chain_v5_common.cuh"

namespace msdr {
namespace v6 {

using namespace tc;
using v5::kPad;
using v5::Prof;
using v5::lds128;
using v5::sts128;
using v5::demod_ssb_regs;
using v5::demod_regs;

constexpr int kWarps = 16;
constexpr int kThreads = kWarps * 32;
constexpr int kChainA = 4, kChainB = 5, kMmaWarp = 6, kLoadWarp = 7, kStoreWarp = 9, kFF1 = 10, kFF2 = 11, kConv0 = 14;
constexpr int kConvThreads = 64;
constexpr int G = 32;             // channels of a group block (one chain warp)
constexpr int HR = 16;            // channels of a tile
constexpr int NB = 32;            // GEMM N = samples of one time block
constexpr int QB = 8;             // time blocks of a tile
constexpr int SPAN = QB * NB;     // samples of a tile row set = 256
constexpr int SUB = 64;           // chain sub-tile, samples
constexpr int RS = 2;             // raw staging stages
constexpr int NSLOT_MAX = 12;      // both rings together (p.tc_ring, even); the barrier arrays are indexed per ring
constexpr int EW = SUB + 4;                                   // sub-tile slot: rows of 64 e[n] words; the packed int16 results overwrite the row's front
constexpr uint32_t kSlotBytes = G * EW * 4u;                  // 8704
constexpr uint32_t RAWP = SPAN * 2 + 16;                      // staging / span buffer row pitch in bytes (16 mod 128: conflict-free)
constexpr uint32_t kRawStageBytes = HR * RAWP;
constexpr uint32_t kSpanBufBytes = G * RAWP;
constexpr uint32_t kUnitBytes = 2 * 128;                      // one unit (16 window words) of one plane: 2 channel groups x 128 B
constexpr uint32_t kAccCols = 3 * NB;                         // TMEM columns of one branch of a tile
constexpr uint32_t kCtrlBytes = 1024;
constexpr uint32_t kScratchBytes = 4 * 2048;                 // epilogue: one demodulated tile part per warp, [column group][lane][16 B]
struct __align__(16) Ctrl {
  uint64_t raw_full[RS];          // load -> convert   : the stage's copies have landed (32 arrivals, cp.async.mbarrier.arrive.noinc)
  uint64_t raw_free[RS];          // convert -> load   : stage read (2 arrivals)
  uint64_t a_full[3];             // convert -> MMA    : operand buffer (tile number mod 3) complete (2 arrivals)
  uint64_t a_free[3];             // MMA -> convert    : the tile's MMAs are complete (tcgen05.commit)
  uint64_t tmem_full[2];          // MMA -> epilogue   : accumulators of tile buffer b complete (tcgen05.commit)
  uint64_t tmem_empty[2];         // epilogue -> MMA   : drained (4 arrivals)
  uint64_t b_full, b_free;        // convert <-> MMA   : Toeplitz operand of the group block's table
  uint64_t y_full[2];             // epilogue -> FF1   : span buffer complete (8 arrivals: 4 warps x 2 tiles)
  uint64_t y_free[2];             // FF1 -> epilogue
  // two rings of sub-tile slots: ring 1 FF1 -> chain A -> FF2, ring 2 FF2 -> chain B -> store (indices are per ring)
  uint64_t ld_full[NSLOT_MAX];    // FF1 -> chain A
  uint64_t ab_full[NSLOT_MAX];    // chain A -> FF2
  uint64_t m_full[NSLOT_MAX];     // FF2 -> chain B
  uint64_t st_full[NSLOT_MAX];    // chain B -> store
  uint64_t slot_free[NSLOT_MAX];  // FF2 -> FF1        : ring 1 slot read
  uint64_t free2[NSLOT_MAX];      // store -> FF2      : ring 2 slot stored
  uint32_t tmem_base;
  long long t_clk, t_ns; // developer profile: kernel entry
};
static_assert(sizeof(Ctrl) <= kCtrlBytes, "Ctrl must fit its smem slot");

__host__ __device__ inline uint32_t units_per_buf(uint32_t K) { return 2u * (K / 32u) + 7u; } // history 2 KS - 2, new 8, one read past the end (times zero taps)
__host__ __device__ inline uint32_t a_plane6(uint32_t K) { return units_per_buf(K) * kUnitBytes; }
__host__ __device__ inline uint32_t b_plane6(uint32_t K) { return (uint32_t)NB * K; }
size_t smem_bytes(uint32_t K, uint32_t nslot)
{
  return (size_t)kCtrlBytes + 12u * a_plane6(K) + 8u * b_plane6(K) + (size_t)RS * kRawStageBytes + 2u * kSpanBufBytes + kScratchBytes + (size_t)nslot * kSlotBytes + 1024u;
}

__device__ __forceinline__ void umma_i8_n32(uint32_t dcol, uint64_t da, uint64_t db, uint32_t a_signed, uint32_t b_signed, uint32_t acc)
{
  const uint32_t idesc = (2u << 4) | (a_signed << 7) | (b_signed << 10) | ((uint32_t)(NB >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
  asm volatile(
      "{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %4, 0;\n\telect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
      ::"r"(dcol), "l"(da), "l"(db), "r"(idesc), "r"(acc), "r"(0), "r"(0), "r"(0), "r"(0)
      : "memory");
}
// eight output columns of one branch: the three byte-plane accumulators (NB columns apart) -> the reference's accumulator mod 2^32.
// Every sub-partition's integer multiplier is the busiest pipe of this kernel (the chains' and the helpers' IMAD.HI), so the epilogue
// stays off it: byte permutes and a three-input add (PRMT, PRMT, IADD3) instead of the two IMAD the compiler makes of shift-and-add.
__device__ __forceinline__ uint32_t shl16_alu(uint32_t v) { uint32_t r; asm("prmt.b32 %0, %1, 0, 0x1044;" : "=r"(r) : "r"(v)); return r; }
__device__ __forceinline__ uint32_t shl8_alu(uint32_t v) { uint32_t r; asm("prmt.b32 %0, %1, 0, 0x2104;" : "=r"(r) : "r"(v)); return r; }
__device__ __forceinline__ void drain8(uint32_t taddr, uint32_t (&acc)[8])
{
  uint32_t a0[8], a1[8], a2[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(a0[0]), "=r"(a0[1]), "=r"(a0[2]), "=r"(a0[3]), "=r"(a0[4]), "=r"(a0[5]), "=r"(a0[6]), "=r"(a0[7]) : "r"(taddr));
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(a1[0]), "=r"(a1[1]), "=r"(a1[2]), "=r"(a1[3]), "=r"(a1[4]), "=r"(a1[5]), "=r"(a1[6]), "=r"(a1[7]) : "r"(taddr + (uint32_t)NB));
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(a2[0]), "=r"(a2[1]), "=r"(a2[2]), "=r"(a2[3]), "=r"(a2[4]), "=r"(a2[5]), "=r"(a2[6]), "=r"(a2[7]) : "r"(taddr + 2u * (uint32_t)NB));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
#ifdef MSDR_V6_EPI_IMAD
  for (int j = 0; j < 8; ++j) acc[j] = (a0[j] << 16) + (a1[j] << 8) + a2[j];
#else
  for (int j = 0; j < 8; ++j) acc[j] = shl16_alu(a0[j]) + shl8_alu(a1[j]) + a2[j];
#endif
}
// SSB kinds on the packed words p = I | Q << 16 (Minimal-SDR.ino:591-604: the int16 sum wraps, no saturation), off the multiplier:
//   t = p ^ xm;  upper half of t + (t << 16) + xc  = I + Q (USB: xm = xc = 0)  or  I + ~Q + 1 = I - Q (LSB: xm = 0xFFFF0000, xc = 0x10000)
__device__ __forceinline__ void demod_ssb_alu(const uint32_t (&iq)[32], uint32_t xm, uint32_t xc, uint32_t (&out)[16])
{
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const uint32_t u0 = iq[2 * j] ^ xm, u1 = iq[2 * j + 1] ^ xm;
    const uint32_t t0 = u0 + shl16_alu(u0) + xc, t1 = u1 + shl16_alu(u1) + xc;
    out[j] = __byte_perm(t0, t1, 0x7632);
  }
}
// 16 window words (32 samples) of row rr -> unit `unit` of the four byte planes of one operand buffer (odd words negated: fs/4 mix,
// Minimal-SDR.ino:550,555; a unit starts on an even word)
__device__ __forceinline__ void convert_unit(uint32_t abuf, uint32_t a_plane, uint32_t unit, uint32_t rr, const uint4 (&v)[4])
{
  uint32_t el[4], eh[4], ol[4], oh[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint32_t a = v[j].x, b = neg16x2(v[j].y), c = v[j].z, d = neg16x2(v[j].w);
    el[j] = __byte_perm(__byte_perm(a, b, 0x0040), __byte_perm(c, d, 0x0040), 0x5410);
    eh[j] = __byte_perm(__byte_perm(a, b, 0x0051), __byte_perm(c, d, 0x0051), 0x5410);
    ol[j] = __byte_perm(__byte_perm(a, b, 0x0062), __byte_perm(c, d, 0x0062), 0x5410);
    oh[j] = __byte_perm(__byte_perm(a, b, 0x0073), __byte_perm(c, d, 0x0073), 0x5410);
  }
  const uint32_t off = abuf + unit * kUnitBytes + (rr >> 3) * 128u + (rr & 7u) * 16u;
  sts128(off + 0 * a_plane, make_uint4(eh[0], eh[1], eh[2], eh[3]));
  sts128(off + 1 * a_plane, make_uint4(el[0], el[1], el[2], el[3]));
  sts128(off + 2 * a_plane, make_uint4(oh[0], oh[1], oh[2], oh[3]));
  sts128(off + 3 * a_plane, make_uint4(ol[0], ol[1], ol[2], ol[3]));
}

// The three input-side products of a stage (msdr_chain_common.cuh: BqFF) as IMAD.HI on values carried as x << 16.  The chain kernel
// keeps them on the FP64 pipe (exact DFMA.RM) because its helpers share a crowded sub-partition; here the helpers' sub-partitions
// have the integer multiplier nearly to themselves and the fixed-latency pipe needs no scoreboard per product group: 196 against
// 188 Gsamples/s at C3 (variant bit 1 selects the DFMA form).
struct BqFFI {
  int b0, b1, b2;
  int x1, x2; // << 16
};
__device__ __forceinline__ int ff_step(BqFFI &f, int xs)
{
  int t0, t1, t2;
  asm("mul.hi.s32 %0, %1, %2;" : "=r"(t0) : "r"(f.b0), "r"(xs));
  asm("mul.hi.s32 %0, %1, %2;" : "=r"(t1) : "r"(f.b1), "r"(f.x1));
  asm("mul.hi.s32 %0, %1, %2;" : "=r"(t2) : "r"(f.b2), "r"(f.x2));
  f.x2 = f.x1; f.x1 = xs;
  return t0 + t1 + t2;
}
__device__ __forceinline__ void bq_load_ff(BqFFI &f, const int32_t *__restrict__ bq, uint32_t Cpad, int obj, uint32_t ch)
{
  const int32_t *b = bq + (size_t)(obj * 4 * 8) * Cpad + ch;
  f.b0 = __ldcg(b + 0 * (size_t)Cpad); f.b1 = __ldcg(b + 1 * (size_t)Cpad); f.b2 = __ldcg(b + 2 * (size_t)Cpad);
  const uint32_t w5 = (uint32_t)__ldcg(b + 5 * (size_t)Cpad); // (x[n-1] << 16) | (x[n-2] & 0xffff), filter_biquad.cpp:66-69
  f.x1 = (int)(w5 & 0xFFFF0000u);
  f.x2 = (int)(w5 << 16);
}
__device__ __forceinline__ void bq_store_ff(const BqFFI &f, int32_t *__restrict__ bq, uint32_t Cpad, int obj, uint32_t ch)
{
  bq[(size_t)(obj * 4 * 8 + 5) * Cpad + ch] = (int32_t)(((uint32_t)f.x1 & 0xFFFF0000u) | ((uint32_t)f.x2 >> 16));
}

// kList: launch row r is chain channel p.chlist[r] (chan_of); int16 input only
template <class FFT, bool kList = false>
__global__ void __launch_bounds__(kThreads, 1) chain_kernel(const ChainParams p)
{
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023u) & ~(uintptr_t)1023u);
  const uint32_t K = p.tc_K, KS = K / 32, KH = 2 * KS - 2, NH = p.tc_ring / 2; // slots per ring
  const uint32_t a_plane = a_plane6(K), b_plane = b_plane6(K);
  Ctrl *pc = reinterpret_cast<Ctrl *>(smem);
  uint8_t *sA = smem + kCtrlBytes;            // [tile number mod 3][plane][unit][2][8][16]
  uint8_t *sB = sA + 12 * a_plane;            // [half][plane][k unit][4 column groups][8][16]
  unsigned char *sRaw = sB + 8 * b_plane;
  unsigned char *sYb = sRaw + RS * kRawStageBytes;
  unsigned char *sScr = sYb + 2 * kSpanBufBytes;
  unsigned char *sSlot = sScr + kScratchBytes;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    if (p.prof) { pc->t_clk = clock64(); asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(pc->t_ns)); }
    for (int i = 0; i < RS; ++i) { mbar_init(&pc->raw_full[i], 32); mbar_init(&pc->raw_free[i], 2); }
    for (int i = 0; i < 3; ++i) { mbar_init(&pc->a_full[i], 2); mbar_init(&pc->a_free[i], 1); }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&pc->tmem_full[b], 1); mbar_init(&pc->tmem_empty[b], 4);
      mbar_init(&pc->y_full[b], 8); mbar_init(&pc->y_free[b], 1);
    }
    mbar_init(&pc->b_full, 2);
    mbar_init(&pc->b_free, 1);
    for (int s = 0; s < NSLOT_MAX; ++s) {
      mbar_init(&pc->ld_full[s], 1); mbar_init(&pc->ab_full[s], 1); mbar_init(&pc->m_full[s], 1); mbar_init(&pc->st_full[s], 1); mbar_init(&pc->slot_free[s], 1); mbar_init(&pc->free2[s], 1);
    }
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc_512(&pc->tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = pc->tmem_base;

  uint32_t ablate; // in a register: re-read from the constant bank once per sub-tile it cost the chains a cache miss each time
  asm volatile("mov.u32 %0, %1;" : "=r"(ablate) : "r"(p.ablate));
  const uint32_t nspan = (p.L + SPAN - 1) / SPAN; // L is a multiple of 128: the last span may be half empty
  const uint32_t nsub = p.L / SUB;
  const uint32_t n_gb = p.n_items;
  const int Hs = (int)p.H;
  const uint32_t stride16 = (uint32_t)(p.stride >> 3);

  if (warp == kLoadWarp) {
    // ================================================================== raw rows: global -> staging ring, one tile (16 rows x 512 B) per stage
    // lane -> rows r0 + 4 i, 16-byte chunks c + 8 j: a warp instruction copies four rows of 128 bytes
    Prof prof(p.prof, 5);
    uint32_t tseq = 0;
    const int r0 = lane >> 3, c = lane & 7;
    const uint4 *in16 = reinterpret_cast<const uint4 *>(p.in);
    for (uint32_t gb = blockIdx.x; gb < n_gb; gb += gridDim.x) {
      const uint32_t *rmap = p.tc_rowmap + (size_t)gb * G;
      uint32_t rows[8]; // [half][i]
#pragma unroll
      for (int i = 0; i < 8; ++i) rows[i] = __ldg(rmap + (i >> 2) * HR + r0 + 4 * (i & 3));
      for (uint32_t s = 0; s < nspan; ++s) {
#pragma unroll
        for (int h = 0; h < 2; ++h, ++tseq) {
          const uint32_t stage = tseq % RS;
          prof.start();
          mbar_wait(&pc->raw_free[stage], ((tseq / RS) & 1u) ^ 1u);
          prof.lap(0);
          const uint32_t dst0 = smem_u32(sRaw + stage * kRawStageBytes) + (uint32_t)r0 * RAWP + (uint32_t)c * 16u;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint32_t row = rows[h * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t col16 = s * (SPAN / 8) + (uint32_t)(c + 8 * j);
              const bool valid = row != kPad && col16 * 8u < p.L;
              const uint4 *src = in16 + ((size_t)(valid ? row : 0u) * stride16 + (valid ? col16 : 0u));
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst0 + (uint32_t)i * 4u * RAWP + (uint32_t)j * 128u), "l"(src), "r"(valid ? 16 : 0) : "memory");
            }
          }
          asm volatile("cp.async.mbarrier.arrive.noinc.shared.b64 [%0];" ::"r"(smem_u32(&pc->raw_full[stage])) : "memory");
          prof.lap(1);
        }
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    prof.flush();
  } else if (warp >= kConv0 && warp < kConv0 + 2) {
    // ================================================================== byte planes: staging ring -> operand buffers
    Prof prof(p.prof, 0);
    const uint32_t t = (uint32_t)(tid - kConv0 * 32), rr = t & 15u, u4 = t >> 4;
    uint32_t tseq = 0, sseq = 0, nblk = 0;
    for (uint32_t gb = blockIdx.x; gb < n_gb; gb += gridDim.x, ++nblk) {
      { // the first 32 columns of the Toeplitz operands of the two halves' tables; the previous block's MMAs must be done with the old ones
        const uint4 rb = __ldg(&p.tc_rb[gb]);
        mbar_wait(&pc->b_free, (nblk & 1u) ^ 1u);
        const uint32_t per_plane = (K / 16u) * 32u; // 16-byte chunks
        for (uint32_t i = t; i < 8u * per_plane; i += kConvThreads) {
          const uint32_t hp = i / per_plane, rem = i - hp * per_plane, ku = rem >> 5, cc = rem & 31u; // hp = half * 4 + plane
          const unsigned char *src = p.tc_bmat + (size_t)(hp < 4u ? rb.x : rb.y) * 4u * N * K;
          const uint4 v = __ldg(reinterpret_cast<const uint4 *>(src + (size_t)(hp & 3u) * N * K + (size_t)ku * (N / 8) * 128u + cc * 16u));
          *reinterpret_cast<uint4 *>(sB + hp * b_plane + ku * 512u + cc * 16u) = v;
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&pc->b_full);
      }
      const uint32_t row2[2] = {__ldg(p.tc_rowmap + (size_t)gb * G + rr), __ldg(p.tc_rowmap + (size_t)gb * G + HR + rr)};
      uint32_t hch2[kList ? 2 : 1]; // a list's history rows
      if constexpr (kList)
        for (int h = 0; h < 2; ++h) hch2[h] = row2[h] != kPad ? v5::chan_of<true>(p, row2[h]) : 0u;
      for (uint32_t s = 0; s < nspan; ++s, ++sseq) {
#pragma unroll
        for (int h = 0; h < 2; ++h, ++tseq) {
          const uint32_t stage = tseq % RS, ab = tseq % 3u;
          const uint32_t abuf = smem_u32(sA + ab * 4u * a_plane);
          prof.start();
          mbar_wait(&pc->raw_full[stage], (tseq / RS) & 1u);
          prof.lap(0);
          mbar_wait(&pc->a_free[ab], ((tseq / 3u) & 1u) ^ 1u);
          prof.lap(1);
          if (!(ablate & 1u)) {
            const uint32_t a = smem_u32(sRaw + stage * kRawStageBytes) + rr * RAWP;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              const uint32_t uu = u4 + 4u * (uint32_t)k;
              uint4 v[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) v[j] = lds128(a + uu * 64u + 16u * (uint32_t)j);
              convert_unit(abuf, a_plane, KH + uu, rr, v);
            }
            if (s == 0) { // in front of sample 0: the carried history, or zeros beyond the taps' reach
              const uint32_t row = row2[h];
              for (uint32_t x = u4; x < KH; x += 4) {
                uint4 v[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  const int smp = ((int)x - (int)KH) * 32 + 8 * j;
                  const size_t hc = kList ? (size_t)hch2[kList ? h : 0] : (size_t)p.ch0 + row;
                  v[j] = (row != kPad && smp >= -Hs) ? __ldg(reinterpret_cast<const uint4 *>(p.hist + hc * p.H + (Hs + smp))) : make_uint4(0, 0, 0, 0);
                }
                convert_unit(abuf, a_plane, x, rr, v);
              }
            } else { // the window tail of the previous span of this half: its last KH units are this span's first
              const uint32_t prev = smem_u32(sA + ((tseq + 1u) % 3u) * 4u * a_plane); // tile tseq - 2: the same half, one span earlier
              const uint32_t per_plane = KH * (kUnitBytes / 16u);
              for (uint32_t i = t; i < 4u * per_plane; i += kConvThreads) {
                const uint32_t pl = i / per_plane, rem = i % per_plane;
                sts128(abuf + pl * a_plane + rem * 16u, lds128(prev + pl * a_plane + QB * kUnitBytes + rem * 16u));
              }
            }
          }
          fence_proxy_async_smem(); // generic-proxy smem writes -> visible to the tensor core (async proxy)
          named_bar_sync(3, kConvThreads); // the tail copy of the next span reads what every converter thread wrote here
          if (lane == 0) { mbar_arrive(&pc->a_full[ab]); mbar_arrive(&pc->raw_free[stage]); }
          prof.lap(2);
        }
      }
      // carry the last H raw samples of the block's rows: hist <- tail of (hist || in[0..L)).  The old history was read at this block's
      // first span, by these threads; nobody else reads or writes the rows' history.
      if (t < (uint32_t)G) {
        const uint32_t row = __ldg(p.tc_rowmap + (size_t)gb * G + t);
        if (row != kPad) {
          const uint32_t hq = p.H >> 3; // uint4 per history row (<= 33)
          uint4 *hrow = reinterpret_cast<uint4 *>(p.hist + v5::hist_ch<kList>(p, row) * p.H);
          const uint4 *irow = reinterpret_cast<const uint4 *>(p.in + (size_t)row * p.stride);
          if (p.L >= p.H) {
            const uint4 *src = irow + ((p.L - p.H) >> 3);
            for (uint32_t i0 = 0; i0 < hq; i0 += 4) { // four loads in flight
              uint4 v[4];
#pragma unroll
              for (int k = 0; k < 4; ++k) if (i0 + k < hq) v[k] = __ldg(src + i0 + k);
#pragma unroll
              for (int k = 0; k < 4; ++k) if (i0 + k < hq) hrow[i0 + k] = v[k];
            }
          } else { // a short update: part of the old history survives (moved down in increasing order, never onto unread entries)
            const uint32_t lq = p.L >> 3, keep = hq - lq;
            for (uint32_t i = 0; i < keep; ++i) hrow[i] = __ldcg(hrow + i + lq);
            for (uint32_t i = keep; i < hq; ++i) hrow[i] = __ldg(irow + (i - keep));
          }
        }
      }
    }
    prof.flush();
  } else if (warp == kMmaWarp) {
    // ================================================================== tensor core
    Prof prof(p.prof, 1);
    // the descriptors differ only in their start-address field (16-byte units): one base each, offsets are added
    const uint64_t descA0 = make_desc(smem_u32(sA), kUnitBytes, 128); // K-adjacent core matrices: the next unit; M-adjacent: the next 8-row group
    const uint64_t descB0 = make_desc(smem_u32(sB), 512, 128);
    uint32_t tseq = 0, sseq = 0, nblk = 0;
    for (uint32_t gb = blockIdx.x; gb < n_gb; gb += gridDim.x, ++nblk) {
      mbar_wait(&pc->b_full, nblk & 1u);
      for (uint32_t s = 0; s < nspan; ++s, ++sseq) {
#pragma unroll
        for (int h = 0; h < 2; ++h, ++tseq) {
          const uint32_t ab = tseq % 3u, tb = tseq & 1u;
          prof.start();
          mbar_wait(&pc->a_full[ab], (tseq / 3u) & 1u);
          prof.lap(0);
          mbar_wait(&pc->tmem_empty[tb], ((tseq >> 1) & 1u) ^ 1u);
          prof.lap(1);
          tc_fence_after();
          if (!(ablate & 1u)) {
            for (uint32_t ks = 0; ks < KS; ++ks) {
              const uint64_t aoff = (uint64_t)((ab * 4u * a_plane + ks * 2u * kUnitBytes) >> 4), boff = (uint64_t)(((uint32_t)h * 4u * b_plane + ks * 2u * 512u) >> 4);
              const uint32_t acc = ks > 0;
#pragma unroll
              for (uint32_t br = 0; br < 2; ++br) {
                const uint64_t a_hi = descA0 + aoff + (uint64_t)((2u * br * a_plane) >> 4), a_lo = a_hi + (uint64_t)(a_plane >> 4); // hi planes signed, lo planes unsigned
                const uint64_t b_hi = descB0 + boff + (uint64_t)((2u * br * b_plane) >> 4), b_lo = b_hi + (uint64_t)(b_plane >> 4);
                const uint32_t d0 = tmem + tb * 2u * kAccCols + br * kAccCols;
                umma_i8_n32(d0, a_hi, b_hi, 1, 1, acc);
                umma_i8_n32(d0 + NB, a_hi, b_lo, 1, 0, acc);
                umma_i8_n32(d0 + NB, a_lo, b_hi, 0, 1, 1);
                umma_i8_n32(d0 + 2 * NB, a_lo, b_lo, 0, 0, acc);
              }
            }
          }
          umma_commit(&pc->tmem_full[tb]);
          umma_commit(&pc->a_free[ab]);
          prof.lap(2);
        }
      }
      umma_commit(&pc->b_free);
    }
    __syncwarp();
    prof.flush();
  } else if (warp < 4) {
    // ================================================================== epilogue: TMEM -> demodulated int16 in the span buffer
    // lane l of warp w holds TMEM lane 32 w + l = row group 4 w + l / 8 = (time block 2 w + l / 16, channel l % 16 of the tile)
    Prof prof(p.prof, 2);
    const uint32_t rr = (uint32_t)lane & 15u, q = 2u * (uint32_t)warp + ((uint32_t)lane >> 4);
    const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
    uint32_t tseq = 0, sseq = 0;
    for (uint32_t gb = blockIdx.x; gb < n_gb; gb += gridDim.x) {
      int kind2[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const uint32_t row = __ldg(p.tc_rowmap + (size_t)gb * G + h * HR + rr);
        kind2[h] = row != kPad ? demod_kind_of((int)p.mode[v5::chan_of<kList>(p, row)], p.am_q31) : 0;
      }
      // The loops below are deliberately NOT unrolled over tiles and column groups: the kernel's roles together stream far more
      // straight-line code than the instruction caches hold, and SMs with a longer path to the next cache level fell 7 % behind
      // (deterministic per SM).  Eight columns per pass through a 2 KB scratch part of this warp keep the epilogue's hot code small.
      const uint32_t scr = smem_u32(sScr) + (uint32_t)warp * 2048u + (uint32_t)lane * 16u;
      for (uint32_t s = 0; s < nspan; ++s, ++sseq) {
#pragma unroll 1
        for (int h = 0; h < 2; ++h, ++tseq) {
          const uint32_t tb = tseq & 1u, yb = sseq & 1u;
          const int kind = h ? kind2[1] : kind2[0];
          prof.start();
          mbar_wait(&pc->tmem_full[tb], (tseq >> 1) & 1u);
          prof.lap(0);
          tc_fence_after();
          const uint32_t ta = lane_addr + tb * 2u * kAccCols;
#pragma unroll 1
          for (int b = 0; b < 4; ++b) {
            uint32_t iq[8], o[4];
            if (!(ablate & (1u | 8u))) {
              uint32_t ai[8], aq[8];
              drain8(ta + (uint32_t)(8 * b), ai);
              drain8(ta + kAccCols + (uint32_t)(8 * b), aq);
#pragma unroll
              for (int j = 0; j < 8; ++j) iq[j] = pack_sat_iq((int)ai[j] >> 15, (int)aq[j] >> 15);
            } else {
#pragma unroll
              for (int j = 0; j < 8; ++j) iq[j] = 0u;
            }
            if (ablate & 4u) {
#pragma unroll
              for (int j = 0; j < 4; ++j) o[j] = iq[2 * j] ^ iq[2 * j + 1];
            } else if (kind <= 1) { // SSB kinds on the packed words p = I | Q << 16 (demod_ssb_alu)
              const uint32_t xm = kind ? 0u : 0xFFFF0000u, xc = kind ? 0u : 0x10000u;
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint32_t u0 = iq[2 * j] ^ xm, u1 = iq[2 * j + 1] ^ xm;
#ifdef MSDR_V6_EPI_IMAD
                o[j] = __byte_perm(u0 * 65537u + xc, u1 * 65537u + xc, 0x7632);
#else
                o[j] = __byte_perm(u0 + shl16_alu(u0) + xc, u1 + shl16_alu(u1) + xc, 0x7632);
#endif
              }
            } else { // envelope kinds: eight square roots in flight
              int y[8];
              if (kind == 2) {
#pragma unroll
                for (int j = 0; j < 8; ++j) y[j] = demod_inline<2>((int)(short)(iq[j] & 0xFFFFu), (int)iq[j] >> 16, 0);
              } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) y[j] = demod_inline<3>((int)(short)(iq[j] & 0xFFFFu), (int)iq[j] >> 16, 0);
              }
#pragma unroll
              for (int j = 0; j < 4; ++j) o[j] = ((uint32_t)y[2 * j] & 0xFFFFu) | ((uint32_t)y[2 * j + 1] << 16);
            }
            sts128(scr + (uint32_t)b * 512u, make_uint4(o[0], o[1], o[2], o[3]));
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&pc->tmem_empty[tb]);
          prof.lap(1);
          mbar_wait(&pc->y_free[yb], ((sseq >> 1) & 1u) ^ 1u);
          prof.lap(2);
          const uint32_t ya = smem_u32(sYb + yb * kSpanBufBytes) + ((uint32_t)h * HR + rr) * RAWP + q * 64u;
#pragma unroll
          for (int j = 0; j < 4; ++j) sts128(ya + 16u * j, lds128(scr + (uint32_t)j * 512u)); // this thread's own words
          __syncwarp();
          if (lane == 0) mbar_arrive(&pc->y_full[yb]);
          prof.lap(3);
        }
      }
    }
    prof.flush();
    named_bar_sync(2, 128); // every epilogue warp has read its last accumulators
    if (warp == 0) {
      tc_fence_before();
      tmem_dealloc_512(tmem);
    }
  } else if (warp == kChainA || warp == kChainB || warp == kFF1 || warp == kFF2) {
    // ================================================================== chain side: lane = channel of the group block
    // slot = rows [32][EW] of 32-bit words: feed-forward sums (or x << 16 for generic cascades), overwritten in place by the stage's packed
    // int16 results (front 128 bytes of the row)
    const bool is_chain = warp == kChainA || warp == kChainB;
    const int obj = (warp == kChainA || warp == kFF1) ? 0 : 1;
    Prof prof(p.prof, warp == kChainA ? 3 : warp == kChainB ? 4 : warp == kFF1 ? 7 : 8);
    uint32_t slot = 0, use = 1, sseq = 0; // ring position as running counters (slot, its use count: the mbarrier phase is its parity): the slot count is a run-time value, a division per sub-tile sat on the chains' path
    for (uint32_t gb = blockIdx.x; gb < n_gb; gb += gridDim.x) {
      const uint32_t row = __ldg(p.tc_rowmap + (size_t)gb * G + lane);
      const bool active = row != kPad;
      const uint32_t ch = kList ? (active ? v5::chan_of<true>(p, row) : 0u) : p.ch0 + (active ? row : 0u);
      // is every lane's object a single stage?  (generic cascades run whole stages in the chain warps, state in global)
      int nst = 1;
      if (active) {
        for (int k = 0; k < 3 && (nst == k + 1); ++k)
          if ((uint32_t)__ldcg(p.bq + (size_t)((obj * 4 + k) * 8 + 7) * p.Cpad + ch) & 0x80000000u) nst = k + 2;
      }
      const bool fast = __all_sync(0xffffffffu, nst == 1);
      if (is_chain) {
        const bool isA = warp == kChainA;
        BqRec rec{};
        uint32_t fl = 0u;
        if (fast && active) bq_load_rec(rec, fl, p.bq, p.Cpad, obj, ch);
        prof.start();
        for (uint32_t k = 0; k < nsub; ++k, slot = (slot + 1 == NH ? 0 : slot + 1), use += (slot == 0)) {
          prof.lap(2);
          mbar_wait(isA ? &pc->ld_full[slot] : &pc->m_full[slot], (use & 1u) ^ 1u);
          prof.lap(0);
          // in place: the eight results of a pass (16 bytes) go where the row's e[n] words have already been read (32 bytes per pass)
          const uint32_t ea = smem_u32(sSlot + (isA ? slot : NH + slot) * kSlotBytes) + (uint32_t)lane * (EW * 4u), ya = ea;
          if (!(ablate & 2u) && active) {
            if (fast) {
              uint4 n0 = lds128(ea), n1 = lds128(ea + 16u);
#pragma unroll 1
              for (int qq = 0; qq < SUB / 8; ++qq) {
                const uint4 e0 = n0, e1 = n1;
                if (qq + 1 < SUB / 8) { n0 = lds128(ea + 32u * (uint32_t)(qq + 1)); n1 = lds128(ea + 32u * (uint32_t)(qq + 1) + 16u); }
                const int y0 = rec_step(rec, (int)e0.x), y1 = rec_step(rec, (int)e0.y), y2 = rec_step(rec, (int)e0.z), y3 = rec_step(rec, (int)e0.w);
                const int y4 = rec_step(rec, (int)e1.x), y5 = rec_step(rec, (int)e1.y), y6 = rec_step(rec, (int)e1.z), y7 = rec_step(rec, (int)e1.w);
                sts128(ya + 16u * (uint32_t)qq, make_uint4(__byte_perm((uint32_t)y0, (uint32_t)y1, 0x7632), __byte_perm((uint32_t)y2, (uint32_t)y3, 0x7632),
                                                           __byte_perm((uint32_t)y4, (uint32_t)y5, 0x7632), __byte_perm((uint32_t)y6, (uint32_t)y7, 0x7632)));
              }
            } else { // generic cascade, stage-major like the reference (filter_biquad.cpp:44-79): E holds x << 16, filtered in place
              uint32_t *er = reinterpret_cast<uint32_t *>(sSlot + (isA ? slot : NH + slot) * kSlotBytes) + (uint32_t)lane * EW;
              uint32_t *yr = er; // packed in place, word n after words 2 n and 2 n + 1 were read
              for (int j = 0; j < nst; ++j) {
                BqStage gs;
                uint32_t gf;
                bq_load_stage(gs, gf, p.bq, p.Cpad, obj, j, ch);
                for (int n = 0; n < SUB; ++n) er[n] = (uint32_t)bq_step(gs, (int)er[n]);
                bq_store_stage(gs, gf, p.bq, p.Cpad, obj, j, ch);
              }
              for (int n = 0; n < SUB / 2; ++n) yr[n] = __byte_perm(er[2 * n], er[2 * n + 1], 0x7632);
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(isA ? &pc->ab_full[slot] : &pc->st_full[slot]);
          prof.lap(1);
        }
        if (fast && active) bq_store_rec(rec, fl, p.bq, p.Cpad, obj, ch);
        if (p.prof && lane == 0 && !isA) { // kernel entry -> chain B done, in SM cycles and in nanoseconds
          long long ns;
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
          long long *b = p.prof + (size_t)blockIdx.x * 64 + 40;
          b[0] = clock64() - pc->t_clk; b[1] = ns - pc->t_ns;
          uint32_t smid;
          asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
          b[2] = (long long)smid; b[3] = pc->t_ns;
        }
      } else {
        // feed-forward helpers.  FF1: span buffer -> e1 (object 1);  FF2: y1 (Y rows of the slot) -> e2 (object 2)
        const bool isF1 = warp == kFF1;
        FFT ff{};
        if (fast && active) bq_load_ff(ff, p.bq, p.Cpad, obj, ch);
        bool sym = false;
        sym = __all_sync(0xffffffffu, !(fast && active) || ff.b0 == ff.b2) && !(ablate & 16u);
        for (uint32_t s = 0; s < nspan; ++s, ++sseq) {
          const uint32_t yb = sseq & 1u;
          if (isF1) {
            prof.start();
            mbar_wait(&pc->y_full[yb], (sseq >> 1) & 1u);
            prof.lap(3);
          }
          const uint32_t nk = min(4u, nsub - 4u * s);
          for (uint32_t k = 0; k < nk; ++k, slot = (slot + 1 == NH ? 0 : slot + 1), use += (slot == 0)) {
            // FF1 fills a slot of ring 1; FF2 reads chain A's results from that slot's rows (their front halves) and fills a slot of ring 2
            const uint32_t ea = smem_u32(sSlot + (isF1 ? slot : NH + slot) * kSlotBytes) + (uint32_t)lane * (EW * 4u);
            prof.start();
            uint32_t src;
            if (isF1) {
              mbar_wait(&pc->slot_free[slot], use & 1u);
              src = smem_u32(sYb + yb * kSpanBufBytes) + (uint32_t)lane * RAWP + k * (SUB * 2u);
            } else {
              mbar_wait(&pc->ab_full[slot], (use & 1u) ^ 1u);
              mbar_wait(&pc->free2[slot], use & 1u);
              src = smem_u32(sSlot + slot * kSlotBytes) + (uint32_t)lane * (EW * 4u);
            }
            prof.lap(0);
            uint4 nx = lds128(src);
            // (loops over the eight-sample groups are not unrolled: see the epilogue's note on instruction-cache footprint)
            if (active && fast && sym) {
              // symmetric numerator (b0 == b2, every low-pass / notch section): hi(b2 x[n-2]) is the product hi(b0 x[n-2]) formed two
              // samples ago - two multiplies per sample instead of three
              if constexpr (sizeof(FFT) == sizeof(BqFFI)) {
                int q1, r1, r2, x1 = ff.x1, x2 = ff.x2;
                asm("mul.hi.s32 %0, %1, %2;" : "=r"(q1) : "r"(ff.b1), "r"(x1));
                asm("mul.hi.s32 %0, %1, %2;" : "=r"(r1) : "r"(ff.b0), "r"(x1));
                asm("mul.hi.s32 %0, %1, %2;" : "=r"(r2) : "r"(ff.b0), "r"(x2));
#pragma unroll 1
                for (int j = 0; j < SUB / 8; ++j) {
                  const uint32_t w[4] = {nx.x, nx.y, nx.z, nx.w};
                  if (j + 1 < SUB / 8) nx = lds128(src + 16u * (uint32_t)(j + 1));
                  uint32_t e[8];
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const int xs = (i & 1) ? (int)(w[i >> 1] & 0xFFFF0000u) : (int)(w[i >> 1] << 16);
                    int p0;
                    asm("mul.hi.s32 %0, %1, %2;" : "=r"(p0) : "r"(ff.b0), "r"(xs));
                    e[i] = (uint32_t)(p0 + q1 + r2);
                    r2 = r1; r1 = p0;
                    asm("mul.hi.s32 %0, %1, %2;" : "=r"(q1) : "r"(ff.b1), "r"(xs));
                  }
                  x2 = (int)(w[3] << 16); x1 = (int)(w[3] & 0xFFFF0000u);
                  sts128(ea + 32u * (uint32_t)j, make_uint4(e[0], e[1], e[2], e[3]));
                  sts128(ea + 32u * (uint32_t)j + 16u, make_uint4(e[4], e[5], e[6], e[7]));
                }
                ff.x1 = x1; ff.x2 = x2;
              } else { // the same with the products as exact DFMA.RM (msdr_chain_common.cuh: BqFF)
                int q1 = __double2loint(__fma_rd(ff.b1, ff.x1, ff.m1)), r1 = __double2loint(__fma_rd(ff.b0, ff.x1, ff.m0)), r2 = __double2loint(__fma_rd(ff.b0, ff.x2, ff.m0));
                double x1 = ff.x1, x2 = ff.x2;
#pragma unroll 1
                for (int j = 0; j < SUB / 8; ++j) {
                  const uint32_t w[4] = {nx.x, nx.y, nx.z, nx.w};
                  if (j + 1 < SUB / 8) nx = lds128(src + 16u * (uint32_t)(j + 1));
                  uint32_t e[8];
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const double xD = bq_d_from_int((i & 1) ? (int)w[i >> 1] >> 16 : (int)(short)(w[i >> 1] & 0xFFFFu));
                    const int p0 = __double2loint(__fma_rd(ff.b0, xD, ff.m0));
                    e[i] = (uint32_t)(p0 + q1 + r2);
                    r2 = r1; r1 = p0;
                    q1 = __double2loint(__fma_rd(ff.b1, xD, ff.m1));
                    if (i == 6) x2 = xD;
                    if (i == 7) x1 = xD;
                  }
                  sts128(ea + 32u * (uint32_t)j, make_uint4(e[0], e[1], e[2], e[3]));
                  sts128(ea + 32u * (uint32_t)j + 16u, make_uint4(e[4], e[5], e[6], e[7]));
                }
                ff.x1 = x1; ff.x2 = x2;
              }
            } else if (active && fast) {
#pragma unroll 1
              for (int j = 0; j < SUB / 8; ++j) {
                const uint32_t w[4] = {nx.x, nx.y, nx.z, nx.w};
                if (j + 1 < SUB / 8) nx = lds128(src + 16u * (uint32_t)(j + 1));
                uint32_t e[8];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  if constexpr (sizeof(FFT) == sizeof(BqFFI)) {
                    e[2 * i] = (uint32_t)ff_step(ff, (int)(w[i] << 16));
                    e[2 * i + 1] = (uint32_t)ff_step(ff, (int)(w[i] & 0xFFFF0000u));
                  } else {
                    e[2 * i] = (uint32_t)ff_step(ff, (int)(short)(w[i] & 0xFFFFu));
                    e[2 * i + 1] = (uint32_t)ff_step(ff, (int)w[i] >> 16);
                  }
                }
                sts128(ea + 32u * (uint32_t)j, make_uint4(e[0], e[1], e[2], e[3]));
                sts128(ea + 32u * (uint32_t)j + 16u, make_uint4(e[4], e[5], e[6], e[7]));
              }
            } else if (active) { // generic cascade: hand x << 16 through
#pragma unroll 1
              for (int j = 0; j < SUB / 8; ++j) {
                const uint32_t w[4] = {nx.x, nx.y, nx.z, nx.w};
                if (j + 1 < SUB / 8) nx = lds128(src + 16u * (uint32_t)(j + 1));
                sts128(ea + 32u * (uint32_t)j, make_uint4(w[0] << 16, w[0] & 0xFFFF0000u, w[1] << 16, w[1] & 0xFFFF0000u));
                sts128(ea + 32u * (uint32_t)j + 16u, make_uint4(w[2] << 16, w[2] & 0xFFFF0000u, w[3] << 16, w[3] & 0xFFFF0000u));
              }
            }
            __syncwarp();
            if (lane == 0) {
              mbar_arrive(isF1 ? &pc->ld_full[slot] : &pc->m_full[slot]);
              if (!isF1) mbar_arrive(&pc->slot_free[slot]); // ring 1's slot has been read
            }
            prof.lap(1);
          }
          if (isF1) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&pc->y_free[yb]);
          }
        }
        if (fast && active) bq_store_ff(ff, p.bq, p.Cpad, obj, ch);
      }
    }
    prof.flush();
  } else if (warp == kStoreWarp) {
    // ================================================================== final audio: Y rows of the slot -> `out`, 4 rows of 128 bytes per warp instruction
    Prof prof(p.prof, 6);
    const int r0 = lane >> 3, c = lane & 7;
    uint4 *out16 = reinterpret_cast<uint4 *>(p.out);
    uint32_t slot = 0, use = 1;
    for (uint32_t gb = blockIdx.x; gb < n_gb; gb += gridDim.x) {
      const uint32_t *rmap = p.tc_rowmap + (size_t)gb * G;
      uint32_t rows[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) rows[i] = __ldg(rmap + r0 + 4 * i);
      for (uint32_t k = 0; k < nsub; ++k, slot = (slot + 1 == NH ? 0 : slot + 1), use += (slot == 0)) {
        prof.start();
        mbar_wait(&pc->st_full[slot], (use & 1u) ^ 1u);
        prof.lap(0);
        const uint32_t sa = smem_u32(sSlot + (NH + slot) * kSlotBytes) + (uint32_t)r0 * (EW * 4u) + (uint32_t)c * 16u; // ring 2; the int16 results are the front 128 bytes of a row
        const uint32_t col16 = k * (SUB / 8) + (uint32_t)c;
        uint4 v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = lds128(sa + (uint32_t)i * 4u * (EW * 4u));
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (rows[i] != kPad) out16[(size_t)rows[i] * stride16 + col16] = v[i];
        __syncwarp();
        if (lane == 0) mbar_arrive(&pc->free2[slot]);
        prof.lap(1);
      }
    }
    prof.flush();
  }
}

} // namespace v6

// number of sub-tile slots (both rings: 8, 10 or 12) that fit next to the operand buffers of window K; 0 = this window is too long for the kernel
uint32_t chain_v6_config(uint32_t K, int smem_max)
{
  if (K % 32u || K / 32u < 2u) return 0;
  for (uint32_t n = v6::NSLOT_MAX; n >= 8u; n -= 2u) // an even count: two rings of at least four slots
    if (v6::smem_bytes(K, n) <= (size_t)smem_max) return n;
  return 0;
}
uint32_t chain_v6_group_rows() { return v6::G; }

cudaError_t launch_chain_v6(const ChainParams &p_in, cudaStream_t stream, int variant, int sms, ChainLaunchInfo *info)
{
  using namespace v6;
  ChainParams p = p_in;
  p.ablate = ((uint32_t)variant >> 4) & 3u;
  if (const char *ev = getenv("MSDR_ABLATE")) p.ablate |= (uint32_t)atoi(ev) & ~3u; // study only: 4 = no demodulation, 8 = no TMEM drain (results are wrong)
  const size_t smem = smem_bytes(p.tc_K, p.tc_ring);
  auto kern = p.chlist ? chain_kernel<BqFFI, true> : (variant & 2) ? chain_kernel<BqFF> : chain_kernel<BqFFI>; // study knob: bit 1 = feed-forward products as DFMA instead of IMAD.HI
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const uint32_t grid = p.n_items < (uint32_t)sms ? p.n_items : (uint32_t)sms;
  if (info) { info->grid = (int)grid; info->block = kThreads; info->smem = smem; info->tile = SPAN; }
  kern<<<grid, kThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

} // namespace msdr
