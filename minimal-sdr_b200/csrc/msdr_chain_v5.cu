// msdr_chain_v5.cu — K1c: the fused receive chain for MANY channels, one persistent CTA per SM that owns whole row blocks.
//
//   int16 IF samples -> [fs/4 mix folded into the byte planes] -> FIR pair as int8 Toeplitz GEMMs on tcgen05.mma (exact mod 2^32,
//   msdr_fir_tc.cu) -> >>15, SSAT16 -> SSB sum / AM envelope -> biquad object 1 -> biquad object 2 -> int16 audio
//
// Reference semantics: Minimal-SDR.ino:546-558 (mix), arm_fir_fast_q15.c:60-329 (FIR), Minimal-SDR.ino:589-628 (demod),
// filter_biquad.cpp:33-82 (biquad).
//
// msdr_chain_v4.cu is built around FEW channels: its biquad chains are pinned to SMs and fed through global memory by FIR producers
// that run anywhere, because 4096 channels are only 128 warps of serial recurrence.  With tens of thousands of channels there is
// enough recurrence for every SM, so here nothing is decoupled: a CTA takes a row block (128 channels that share one tap table,
// msdr_capi.cu::build_tc_plan) and walks it through time, 64 samples per tile, every stage handing its tile to the next through
// shared memory.  The FIR -> biquad intermediate never leaves the SM, no counters are polled, DRAM traffic is the algorithmic
// 2 B in + 2 B out per sample.  23 warps, roles by warp id (warp id % 4 = SM sub-partition):
//
//   warp 21        load      cp.async (LDGSTS) of the tile's raw rows (128 rows x 128 B, gathered through the row map; history or
//                            zeros in front of sample 0) into a 2-stage staging ring; completion arrives on an mbarrier
//   warps 16-19    convert   thread = row: raw int16 -> fs/4 sign fold -> four byte planes in the ring of A operands (the window of a
//                            tile is the last K/32 ring entries, so every sample is converted exactly once per launch)
//   warp 20        MMA       one elected lane: 2 branches x 4 byte-plane products x K/32 MMAs (M128 N64 K32) per tile, tcgen05.commit
//   warps 0-7      epilogue  TMEM lane quadrant = warp id % 4 (hardware rule), two warps per quadrant take 32 of the 64 columns each:
//                            tcgen05.ld, recombine, >>15, SSAT16 -> packed (I, Q) in registers, hand TMEM back, demodulate, park the
//                            int16 rows in one of four tile slots
//   warps 8-11     biquad 1  lane = row: object 1 over the slot in place (state in registers for the whole row block)
//   warps 12-15    biquad 2  object 2 likewise
//   warp 22        store     slot -> `out`, 128 B per row and tile, coalesced
//
// Every sub-partition hosts two epilogue warps, one warp of each biquad object and one converter: the TMEM read port (64 B/clk per
// SM, 24 B per output sample for the six int32 accumulators), the integer multiplier (5 IMAD.HI per sample and stage) and the issue
// slots are all used evenly.
#include <cstdlib>
#include <type_traits>
#include "msdr_chain_v5_common.cuh"

namespace msdr {
namespace v5 {

using namespace tc;

constexpr int kWarps = 23;
constexpr int kThreads = kWarps * 32;
constexpr int kEpiWarps = 8, kBqA0 = 8, kBqB0 = 12, kConv0 = 16, kMmaWarp = 20, kLoadWarp = 21, kStoreWarp = 22;
constexpr int RS = 2;                  // raw staging stages
constexpr int NS = 4;                  // tile slots: epilogue | biquad 1 | biquad 2 | store
constexpr int YW = N / 2 + 4;          // slot row pitch in words (4 mod 32: conflict-free row-wise 128-bit accesses)
constexpr uint32_t RAWP = 2 * N + 16;  // raw staging row pitch in bytes
constexpr uint32_t kRawStageBytes = M * RAWP;
constexpr uint32_t kSlotBytes = M * YW * 4;
constexpr uint32_t kCtrlBytes = 1024;
struct __align__(16) Ctrl {
  uint64_t raw_full[RS];        // load -> convert    : the stage's copies have landed (32 arrivals, cp.async.mbarrier.arrive.noinc)
  uint64_t raw_free[RS];        // convert -> load    : stage read (4 arrivals)
  uint64_t a_full[RING_MAX];    // convert -> MMA     : pair converted (4 arrivals)
  uint64_t blk_free[RING_MAX];  // MMA -> convert     : pair no longer read (tcgen05.commit)
  uint64_t tmem_full[2];        // MMA -> epilogue    : accumulators of branch I / Q complete (tcgen05.commit)
  uint64_t tmem_empty[2];       // epilogue -> MMA    : accumulators of branch I / Q drained (8 arrivals)
  uint64_t b_full;              // convert -> MMA     : Toeplitz operand of the row block's table in place (4 arrivals)
  uint64_t b_free;              // MMA -> convert     : all MMAs of the previous row block complete (tcgen05.commit)
  uint64_t y_full[NS][4];       // epilogue -> biquad 1 (per 32-row quarter; 2 arrivals: both column halves)
  uint64_t ab_full[NS][4];      // biquad 1 -> biquad 2 (per quarter)
  uint64_t st_full[NS];         // biquad 2 -> store  (4 arrivals)
  uint64_t slot_free[NS];       // store -> epilogue  (8 waiters)
  uint32_t tmem_base;
};
static_assert(sizeof(Ctrl) <= kCtrlBytes, "Ctrl must fit its smem slot");

size_t smem_bytes(uint32_t K, uint32_t ring)
{
  return (size_t)kCtrlBytes + 4u * a_plane_bytes(ring) + 4u * N * K + (size_t)RS * kRawStageBytes + (size_t)NS * kSlotBytes + 1024u;
}

// BQ: BqStage = all five SMLAW products of a stage as IMAD.HI; BqStageH = the three input-side products as exact DFMA.RM on the
// FP64 pipe (msdr_device.cuh).  Alone in its sub-partition a warp steps equally fast either way (43 cycles, it is issue-bound);
// here two biquad warps, two epilogue warps and a converter share a sub-partition and the integer multiplier is the scarce pipe
// (IMAD.HI occupies it for 5 cycles), so the default moves three of the five products off it.
// kAdc: `p.in` holds raw ADC codes; the converters run the front end over them (FeRow, msdr_chain_v5_common.cuh)
// kList: launch row r is chain channel p.chlist[r] (chan_of); int16 input only
template <class BQ, bool kAdc, bool kList = false>
__global__ void __launch_bounds__(kThreads, 1) chain_kernel(const ChainParams p)
{
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023u) & ~(uintptr_t)1023u);
  const uint32_t K = p.tc_K, KS = K / 32, ring = p.tc_ring;
  const uint32_t a_plane = a_plane_bytes(ring), b_plane = N * K;
  Ctrl *pc = reinterpret_cast<Ctrl *>(smem);
  uint8_t *sA = smem + kCtrlBytes;
  uint8_t *sB = sA + 4 * a_plane;
  unsigned char *sRaw = sB + 4 * b_plane;
  unsigned char *sY = sRaw + RS * kRawStageBytes;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int i = 0; i < RS; ++i) { mbar_init(&pc->raw_full[i], 32); mbar_init(&pc->raw_free[i], 4); }
    for (int i = 0; i < RING_MAX; ++i) { mbar_init(&pc->a_full[i], 4); mbar_init(&pc->blk_free[i], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&pc->tmem_full[b], 1); mbar_init(&pc->tmem_empty[b], kEpiWarps); }
    mbar_init(&pc->b_full, 4);
    mbar_init(&pc->b_free, 1);
    for (int s = 0; s < NS; ++s) {
      for (int q = 0; q < 4; ++q) { mbar_init(&pc->y_full[s][q], 2); mbar_init(&pc->ab_full[s][q], 1); }
      mbar_init(&pc->st_full[s], 4);
      mbar_init(&pc->slot_free[s], 1);
    }
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc_512(&pc->tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = pc->tmem_base;

  const uint32_t NT = p.L / N;              // tiles per row block (L is a multiple of 128)
  const uint32_t npairs = NT + KS - 1;      // ring entries per row block: KS - 1 of history in front
  const uint32_t n_rb = p.n_items;
  const int Hs = (int)p.H;

  if (warp == kLoadWarp) {
    // ================================================================== raw rows: global -> staging ring
    // lane -> (row r0 + 4 i, 16-byte chunk c): a warp instruction copies four rows of 128 bytes.  The 32 row offsets of a lane live
    // in registers (in 16-byte units, so 2^20 rows x any stride fit 32 bits): the copy loop is an address add and a cp.async.
    Prof prof(p.prof, 5);
    uint32_t pseq = 0;
    const int r0 = lane >> 3, c = lane & 7;
    const uint32_t stride16 = (uint32_t)(p.stride >> 3);
    const uint4 *in16 = reinterpret_cast<const uint4 *>(p.in);
    for (uint32_t rb = blockIdx.x; rb < n_rb; rb += gridDim.x) {
      const uint32_t *rmap = p.tc_rowmap + (size_t)rb * M;
      uint32_t rows[M / 4];
#pragma unroll
      for (int i = 0; i < M / 4; ++i) rows[i] = __ldg(rmap + r0 + 4 * i);
      // a list: the same registers hold the rows' chain channels (their history rows) for the stages in front of sample 0, then
      // the launch rows again (a second set of offsets beside them spilled)
      if constexpr (kList) {
#pragma unroll
        for (int i = 0; i < M / 4; ++i) rows[i] = rows[i] != kPad ? chan_of<true>(p, rows[i]) : kPad;
      }
      for (int j = -(int)(KS - 1); j < (int)NT; ++j, ++pseq) {
        if constexpr (kList) {
          if (j == 0) {
#pragma unroll
            for (int i = 0; i < M / 4; ++i) rows[i] = __ldg(p.tc_rowmap + (size_t)rb * M + r0 + 4 * i);
          }
        }
        const uint32_t stage = pseq % RS;
        prof.start();
        mbar_wait(&pc->raw_free[stage], ((pseq / RS) & 1u) ^ 1u, kNsLoad);
        prof.lap(0);
        const uint32_t dst0 = smem_u32(sRaw + stage * kRawStageBytes) + (uint32_t)r0 * RAWP + (uint32_t)c * 16u;
        if (p.ablate & 1u) {
        } else if (j >= 0) {
          const uint32_t col16 = (uint32_t)j * (N / 8) + (uint32_t)c; // this lane's chunk of the tile, in 16-byte units
#pragma unroll
          for (int i = 0; i < M / 4; ++i) {
            const bool valid = rows[i] != kPad;
            const uint4 *src = in16 + ((size_t)(valid ? rows[i] : 0u) * stride16 + col16);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst0 + (uint32_t)i * 4u * RAWP), "l"(src), "r"(valid ? 16 : 0) : "memory");
          }
        } else { // in front of sample 0: the carried history, or zeros beyond the taps' reach
          const int s = j * N + 8 * c; // first sample of this lane's chunk (negative)
#pragma unroll
          for (int i = 0; i < M / 4; ++i) {
            const bool valid = rows[i] != kPad && s >= -Hs;
            const size_t hc = kList ? (size_t)rows[i] : (size_t)p.ch0 + rows[i];
            const int16_t *src = valid ? p.hist + hc * p.H + (Hs + s) : p.in; // never dereferenced when the size is 0
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst0 + (uint32_t)i * 4u * RAWP), "l"(src), "r"(valid ? 16 : 0) : "memory");
          }
        }
        asm volatile("cp.async.mbarrier.arrive.noinc.shared.b64 [%0];" ::"r"(smem_u32(&pc->raw_full[stage])) : "memory");
        prof.lap(1);
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    prof.flush();
  } else if (warp >= kConv0 && warp < kConv0 + 4) {
    // ================================================================== byte planes: staging ring -> ring of A operands
    Prof prof(p.prof, 0);
    const uint32_t r = (uint32_t)(tid - kConv0 * 32); // row
    uint32_t pseq = 0, nblk = 0;
    for (uint32_t rb = blockIdx.x; rb < n_rb; rb += gridDim.x, ++nblk) {
      { // Toeplitz operand of this row block's table; the previous row block's MMAs must be done with the old one
        const uint32_t set = __ldg(&p.tc_rb[rb].x);
        mbar_wait(&pc->b_free, (nblk & 1u) ^ 1u, kNsConv);
        const uint4 *src = reinterpret_cast<const uint4 *>(p.tc_bmat + (size_t)set * 4 * b_plane);
        uint4 *dst = reinterpret_cast<uint4 *>(sB);
        for (uint32_t i = r; i < 4 * b_plane / 16; i += M) dst[i] = __ldg(src + i);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&pc->b_full);
      }
      FeRow fr;
      if constexpr (kAdc) fe_row_begin(fr, p, __ldg(p.tc_rowmap + (size_t)rb * M + r));
      for (uint32_t u = 0; u < npairs; ++u, ++pseq) {
        const uint32_t stage = pseq % RS, pos = pseq % ring;
        prof.start();
        mbar_wait(&pc->raw_full[stage], (pseq / RS) & 1u, kNsConv);
        prof.lap(0);
        mbar_wait(&pc->blk_free[pos], ((pseq / ring) & 1u) ^ 1u, kNsConv);
        prof.lap(1);
        if (!(p.ablate & 1u)) {
          const uint32_t a = smem_u32(sRaw + stage * kRawStageBytes) + r * RAWP;
          if constexpr (kAdc) {
            if (u >= KS - 1) { // codes of samples 64 j .. 64 j + 63, j = u - (KS - 1); in front of sample 0 the history is conditioned already
              const uint32_t t0 = (u - (KS - 1)) * N;
              if (t0 == 0) fe_row_shift_hist(fr, p);
              fe_row_run<N / 8>(fr, p, a, t0);
            }
          }
          uint4 v0[4], v1[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) { v0[j] = lds128(a + 16u * j); v1[j] = lds128(a + 64u + 16u * j); }
          convert_store(sA, a_plane, pos, 0, r, v0);
          convert_store(sA, a_plane, pos, 1, r, v1);
        }
        fence_proxy_async_smem(); // generic-proxy smem writes -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) { mbar_arrive(&pc->a_full[pos]); mbar_arrive(&pc->raw_free[stage]); }
        prof.lap(2);
      }
      if constexpr (kAdc) {
        fe_row_end(fr); // the history was written as the samples were conditioned
      } else { // carry the last H raw samples of this thread's row: hist <- tail of (hist || in[0..L)).  The old history was this row
        // block's first staging entries, which this thread converted long ago; nobody else reads or writes the row's history.
        const uint32_t row = __ldg(p.tc_rowmap + (size_t)rb * M + r);
        if (row != kPad) {
          const uint32_t hq = p.H >> 3; // uint4 per history row (<= 33)
          uint4 *hrow = reinterpret_cast<uint4 *>(p.hist + hist_ch<kList>(p, row) * p.H);
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
    IssueCtx ictx;
    issue_init(ictx, sA, a_plane, sB, b_plane);
    uint32_t qbase = 0, tseq = 0, nblk = 0;
    for (uint32_t rb = blockIdx.x; rb < n_rb; rb += gridDim.x, ++nblk) {
      mbar_wait(&pc->b_full, nblk & 1u);
      for (uint32_t t = 0; t < NT; ++t, ++tseq) {
        const uint32_t qt = qbase + t + KS - 1; // newest pair of this tile's window
        prof.start();
        mbar_wait(&pc->a_full[qt % ring], (qt / ring) & 1u, 32);
        prof.lap(0);
        // the two branches have their own accumulators and their own hand-off: the epilogue drains I while Q is being issued, and
        // the next tile's I products start as soon as I is drained
#pragma unroll
        for (uint32_t br = 0; br < 2; ++br) {
          mbar_wait(&pc->tmem_empty[br], (tseq & 1u) ^ 1u, 32);
          if (br == 0) prof.lap(1);
          tc_fence_after();
          if (!(p.ablate & 1u)) issue_branch(ictx, tmem, qt, KS, ring, br);
          umma_commit(&pc->tmem_full[br]);
        }
        umma_commit(&pc->blk_free[(qt - (KS - 1)) % ring]); // the oldest pair of the window is not read again
        prof.lap(2);
      }
      for (uint32_t s = 1; s < KS; ++s) umma_commit(&pc->blk_free[(qbase + npairs - KS + s) % ring]);
      umma_commit(&pc->b_free);
      qbase += npairs;
    }
    __syncwarp();
    prof.flush();
  } else if (warp < kEpiWarps) {
    // ================================================================== epilogue: TMEM -> demodulated int16 rows in a tile slot
    Prof prof(p.prof, 2);
    const int qd = warp & 3, half = warp >> 2;
    const uint32_t trow = (uint32_t)(qd * 32 + lane);
    const uint32_t lane_addr = tmem + ((uint32_t)(qd * 32) << 16) + (uint32_t)(half * 32);
    uint32_t tseq = 0;
    for (uint32_t rb = blockIdx.x; rb < n_rb; rb += gridDim.x) {
      const uint32_t row = __ldg(p.tc_rowmap + (size_t)rb * M + trow);
      const int kind = row != kPad ? demod_kind_of((int)p.mode[chan_of<kList>(p, row)], p.am_q31) : 0;
      // Eight columns per pass, the passes not unrolled: unrolled, the epilogue streamed ~7-26 KB of straight-line code per tile and warp
      // through the instruction caches it shares with the biquad warps (ncu: instruction-cache hit rate 86 %, no_instruction 8 % of the
      // warp samples; msdr_chain_v6.cu gained 16 % from the same change).  The per-branch tensor-memory hand-off stays: the I pass parks
      // its saturated values as int16 pairs in this thread's own 64 bytes of the tile slot, the Q pass reads them back, demodulates and
      // writes the result over them.
      for (uint32_t t = 0; t < NT; ++t, ++tseq) {
        const uint32_t slot = tseq % NS;
        prof.start();
        mbar_wait(&pc->tmem_full[0], tseq & 1u, 48);
        prof.lap(0);
        tc_fence_after();
        mbar_wait(&pc->slot_free[slot], ((tseq / NS) & 1u) ^ 1u, kNsSlot);
        const uint32_t ya = smem_u32(sY + slot * kSlotBytes) + trow * (uint32_t)(YW * 4) + (uint32_t)(half * 64);
#pragma unroll 1
        for (int b = 0; b < 4; ++b) {
          uint32_t ai[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
          if (!(p.ablate & 1u)) drain8(lane_addr + (uint32_t)(8 * b), ai);
          uint32_t w[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) w[j] = pack_sat_iq((int)ai[2 * j] >> 15, (int)ai[2 * j + 1] >> 15); // I of samples 2 j | 2 j + 1
          sts128(ya + 16u * (uint32_t)b, make_uint4(w[0], w[1], w[2], w[3]));
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&pc->tmem_empty[0]); // the next tile's I products may start
        mbar_wait(&pc->tmem_full[1], tseq & 1u, 48);
        tc_fence_after();
        prof.lap(1);
#pragma unroll 1
        for (int b = 0; b < 4; ++b) {
          uint32_t aq[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
          if (!(p.ablate & 1u)) drain8(lane_addr + (uint32_t)(kAccPerBranch * N + 8 * b), aq);
          const uint4 iw = lds128(ya + 16u * (uint32_t)b);
          const uint32_t ip[4] = {iw.x, iw.y, iw.z, iw.w};
          uint32_t iq[8], o[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t qp = pack_sat_iq((int)aq[2 * j] >> 15, (int)aq[2 * j + 1] >> 15);
            iq[2 * j] = __byte_perm(ip[j], qp, 0x5410);     // I | Q << 16 of sample 2 j
            iq[2 * j + 1] = __byte_perm(ip[j], qp, 0x7632); // ... of sample 2 j + 1
          }
          if (kind <= 1) { // SSB kinds straight on the packed words (demod_ssb_regs)
            const uint32_t xm = kind ? 0u : 0xFFFF0000u, xc = kind ? 0u : 0x10000u;
#pragma unroll
            for (int j = 0; j < 4; ++j) o[j] = __byte_perm((iq[2 * j] ^ xm) * 65537u + xc, (iq[2 * j + 1] ^ xm) * 65537u + xc, 0x7632);
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
          sts128(ya + 16u * (uint32_t)b, make_uint4(o[0], o[1], o[2], o[3]));
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) { mbar_arrive(&pc->tmem_empty[1]); mbar_arrive(&pc->y_full[slot][qd]); }
        prof.lap(2);
      }
    }
    prof.flush();
    named_bar_sync(2, kEpiWarps * 32); // every epilogue warp has read its last accumulators
    if (warp == 0) {
      tc_fence_before();
      tmem_dealloc_512(tmem);
    }
  } else if (warp >= kBqA0 && warp < kBqB0 + 4) {
    // ================================================================== biquad objects: lane = row, state in registers
    const bool isA = warp < kBqB0;
    const int obj = isA ? 0 : 1, q = isA ? warp - kBqA0 : warp - kBqB0;
    Prof prof(q == 0 ? p.prof : nullptr, isA ? 3 : 4);
    const uint32_t trow = (uint32_t)(q * 32 + lane);
    uint32_t tseq = 0;
    for (uint32_t rb = blockIdx.x; rb < n_rb; rb += gridDim.x) {
      const uint32_t row = __ldg(p.tc_rowmap + (size_t)rb * M + trow);
      const bool active = row != kPad;
      const uint32_t ch = kList ? (active ? chan_of<true>(p, row) : 0u) : p.ch0 + (active ? row : 0u);
      // cascade structure of this lane's object: stages run while bit31 of word 7 says another follows (filter_biquad.cpp:75,79)
      int nst = 1;
      BQ st[1];
      uint32_t fl = 0u;
      if (active) {
        for (int k = 0; k < 3 && (nst == k + 1); ++k)
          if ((uint32_t)__ldcg(p.bq + (size_t)((obj * 4 + k) * 8 + 7) * p.Cpad + ch) & 0x80000000u) nst = k + 2;
      }
      const bool fast = __all_sync(0xffffffffu, nst == 1);
      if (fast && active) bq_load_stage(st[0], fl, p.bq, p.Cpad, obj, 0, ch);
      // symmetric numerators (b0 == b2) in every lane: the four-product form of the stage (msdr_device.cuh: BqStageWS)
      bool sym = false;
      using SYM = typename BqSymOf<BQ>::type;
      constexpr bool kHasSym = !std::is_same<SYM, void>::value;
      typename std::conditional<kHasSym, SYM, BqStageWS>::type ss[1];
      if constexpr (kHasSym) {
        sym = fast && !(p.ablate & 4u) && __all_sync(0xffffffffu, !active || st[0].b0 == st[0].b2);
        if (sym && active) {
          static_cast<BqStage &>(ss[0]) = static_cast<const BqStage &>(st[0]);
          ss[0].p1 = __mulhi(st[0].b0, st[0].x1);
          ss[0].p2 = __mulhi(st[0].b0, st[0].x2);
        }
      }
      for (uint32_t t = 0; t < NT; ++t, ++tseq) {
        const uint32_t slot = tseq % NS, phs = (tseq / NS) & 1u;
        prof.start();
        mbar_wait(isA ? &pc->y_full[slot][q] : &pc->ab_full[slot][q], phs, kNsBq);
        prof.lap(0);
        const uint32_t ya = smem_u32(sY + slot * kSlotBytes) + trow * (uint32_t)(YW * 4);
        if (!(p.ablate & 2u) && active) {
          if (sym) bq_tile(ss, ya);
          else if (fast) bq_tile(st, ya);
          else { // generic cascade: stage-major over the tile like the reference (filter_biquad.cpp:44-79); state in global
            for (int j = 0; j < nst; ++j) {
              BQ gs[1];
              uint32_t gf;
              bq_load_stage(gs[0], gf, p.bq, p.Cpad, obj, j, ch);
              bq_tile(gs, ya);
              bq_store_stage(gs[0], gf, p.bq, p.Cpad, obj, j, ch);
            }
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(isA ? &pc->ab_full[slot][q] : &pc->st_full[slot]);
        prof.lap(1);
      }
      if constexpr (kHasSym) {
        if (sym && active) static_cast<BqStage &>(st[0]) = static_cast<const BqStage &>(ss[0]);
      }
      if (fast && active) bq_store_stage(st[0], fl, p.bq, p.Cpad, obj, 0, ch);
    }
    prof.flush();
  } else if (warp == kStoreWarp) {
    // ================================================================== final audio: slot -> `out` (row offsets in registers like the loader)
    Prof prof(p.prof, 6);
    const int r0 = lane >> 3, c = lane & 7;
    const uint32_t stride16 = (uint32_t)(p.stride >> 3);
    uint4 *out16 = reinterpret_cast<uint4 *>(p.out);
    uint32_t tseq = 0;
    for (uint32_t rb = blockIdx.x; rb < n_rb; rb += gridDim.x) {
      const uint32_t *rmap = p.tc_rowmap + (size_t)rb * M;
      uint32_t rows[M / 4];
#pragma unroll
      for (int i = 0; i < M / 4; ++i) rows[i] = __ldg(rmap + r0 + 4 * i);
      for (uint32_t t = 0; t < NT; ++t, ++tseq) {
        const uint32_t slot = tseq % NS, phs = (tseq / NS) & 1u;
        prof.start();
        mbar_wait(&pc->st_full[slot], phs, kNsStore);
        prof.lap(0);
        const uint32_t sa = smem_u32(sY + slot * kSlotBytes) + (uint32_t)r0 * (uint32_t)(YW * 4) + (uint32_t)c * 16u;
        const uint32_t col16 = t * (N / 8) + (uint32_t)c;
#pragma unroll
        for (int i0 = 0; i0 < M / 4; i0 += 4) {
          uint4 v[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) v[k] = lds128(sa + (uint32_t)(i0 + k) * 4u * (uint32_t)(YW * 4));
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (rows[i0 + k] != kPad) out16[(size_t)rows[i0 + k] * stride16 + col16] = v[k];
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&pc->slot_free[slot]);
        prof.lap(1);
      }
    }
    prof.flush();
  }
}

} // namespace v5

// deepest operand ring (at least one pair ahead of the window) that fits next to the staging ring and the tile slots; 0 = this
// window is too long for the row-block kernel (256 taps: the chain kernel of msdr_chain_v4.cu takes it)
uint32_t chain_v5_config(uint32_t K, int smem_max)
{
  if (K % 32u || K / 32u < 2u) return 0;
  for (uint32_t ring = tc::RING_MAX; ring >= K / 32u + 1u; --ring)
    if (v5::smem_bytes(K, ring) <= (size_t)smem_max) return ring;
  return 0;
}

cudaError_t launch_chain_v5(const ChainParams &p_in, cudaStream_t stream, int variant, int sms, ChainLaunchInfo *info)
{
  using namespace v5;
  ChainParams p = p_in;
  p.ablate = ((uint32_t)variant >> 4) & 3u;
  if (getenv("MSDR_NOSYM")) p.ablate |= 4u; // study: never the four-product stage for symmetric numerators
  const size_t smem = smem_bytes(p.tc_K, p.tc_ring);
  // default: the products as IMAD.HI (with the looped epilogue 352 against 339 Gsamples/s at C5 for the IMAD.WIDE form, which was 1.5 %
  // ahead before); study knobs: variant bit 0 = IMAD.WIDE for the four products off the recurrence, bit 1 = feed-forward products as DFMA
  auto kern = p.fe ? chain_kernel<BqStage, true> : p.chlist ? chain_kernel<BqStage, false, true>
                   : (variant & 12) == 12 ? chain_kernel<BqStageS, false> : (variant & 1) ? chain_kernel<BqStageW, false> : (variant & 2) ? chain_kernel<BqStageH, false>
                   : (variant & 4) ? chain_kernel<BqStageC, false> : (variant & 8) ? chain_kernel<BqStageE, false> : chain_kernel<BqStage, false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const uint32_t grid = p.n_items < (uint32_t)sms ? p.n_items : (uint32_t)sms;
  if (info) { info->grid = (int)grid; info->block = kThreads; info->smem = smem; info->tile = tc::N; }
  kern<<<grid, kThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

} // namespace msdr
