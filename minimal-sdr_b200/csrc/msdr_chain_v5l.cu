// msdr_chain_v5l.cu — K1c for LONG windows (256 taps: BASELINE config 4): the row-block kernel of msdr_chain_v5.cu with every hand-off
// between roles cut to HALF a tile (32 samples), because the 192-word window leaves no room for whole-tile buffers:
//
//   operand ring 7 pairs x 16 KB + Toeplitz operand 48 KB = 160 KB; left for staging and tile slots: 66 KB
//   msdr_chain_v5.cu wants 2 staging stages + 4 tile slots of 18 KB = 108 KB.  Here: 2 staging half-stages + 4 half-slots of 10 KB = 60 KB,
//   the same pipeline depth in half-size units (load | convert, epilogue | biquad 1 | biquad 2 | store).
//
// The units fall out of the structure: a K-block of the A operand is 32 samples, so a converter turns one staging half-stage into one
// K-block; the two epilogue warps of a TMEM lane quadrant already take the two 32-column halves of a tile, so each parks its own
// half-slot; the biquad warps run the half-slots in time order.  Same roles, same warps, same arithmetic and the same plan as
// msdr_chain_v5.cu; reference semantics as there (Minimal-SDR.ino:546-558,589-628, arm_fir_fast_q15.c:60-329, filter_biquad.cpp:33-82).
#include <type_traits>
#include "msdr_chain_v5_common.cuh"

namespace msdr {
namespace v5l {

using namespace tc;
using namespace v5;

constexpr int kWarps = 23;
constexpr int kThreads = kWarps * 32;
constexpr int kEpiWarps = 8, kBqA0 = 8, kBqB0 = 12, kConv0 = 16, kMmaWarp = 20, kLoadWarp = 21, kStoreWarp = 22;
constexpr int HU = N / 2;              // samples per hand-off unit (half a tile = one K-block of the A operand)
constexpr int RSH = 2;                 // raw staging half-stages
constexpr int NH = 4;                  // half-slots: epilogue | biquad 1 | biquad 2 | store
constexpr uint32_t HP = 2 * HU + 16;   // row pitch of a half-stage / half-slot in bytes (80: 20 words, conflict-free 128-bit rows)
constexpr uint32_t kHalfBytes = M * HP;
constexpr uint32_t kCtrlBytes = 1024;

struct __align__(16) Ctrl {
  uint64_t raw_full[RSH];       // load -> convert    : the half-stage's copies have landed (32 arrivals, cp.async.mbarrier.arrive.noinc)
  uint64_t raw_free[RSH];       // convert -> load    : half-stage read (4 arrivals)
  uint64_t a_full[RING_MAX];    // convert -> MMA     : pair converted (4 arrivals, after its second K-block)
  uint64_t blk_free[RING_MAX];  // MMA -> convert     : pair no longer read (tcgen05.commit)
  uint64_t tmem_full[2];        // MMA -> epilogue    : accumulators of branch I / Q complete (tcgen05.commit)
  uint64_t tmem_empty[2];       // epilogue -> MMA    : accumulators of branch I / Q drained (8 arrivals)
  uint64_t b_full;              // convert -> MMA     : Toeplitz operand of the row block's table in place (4 arrivals)
  uint64_t b_free;              // MMA -> convert     : all MMAs of the previous row block complete (tcgen05.commit)
  uint64_t y_full[NH][4];       // epilogue -> biquad 1 (per 32-row quarter; one epilogue warp owns a half-slot's quarter)
  uint64_t ab_full[NH][4];      // biquad 1 -> biquad 2 (per quarter)
  uint64_t st_full[NH];         // biquad 2 -> store  (4 arrivals)
  uint64_t slot_free[NH];       // store -> epilogue  (4 waiters)
  uint32_t tmem_base;
};
static_assert(sizeof(Ctrl) <= kCtrlBytes, "Ctrl must fit its smem slot");

size_t smem_bytes(uint32_t K, uint32_t ring)
{
  return (size_t)kCtrlBytes + 4u * a_plane_bytes(ring) + 4u * N * K + (size_t)(RSH + NH) * kHalfBytes + 1024u;
}

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
  unsigned char *sY = sRaw + RSH * kHalfBytes;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int i = 0; i < RSH; ++i) { mbar_init(&pc->raw_full[i], 32); mbar_init(&pc->raw_free[i], 4); }
    for (int i = 0; i < RING_MAX; ++i) { mbar_init(&pc->a_full[i], 4); mbar_init(&pc->blk_free[i], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&pc->tmem_full[b], 1); mbar_init(&pc->tmem_empty[b], kEpiWarps); }
    mbar_init(&pc->b_full, 4);
    mbar_init(&pc->b_free, 1);
    for (int s = 0; s < NH; ++s) {
      for (int q = 0; q < 4; ++q) { mbar_init(&pc->y_full[s][q], 1); mbar_init(&pc->ab_full[s][q], 1); }
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
  const uint32_t nhalf = 2 * npairs;        // staging half-stages per row block
  const uint32_t n_rb = p.n_items;
  const int Hs = (int)p.H;

  if (warp == kLoadWarp) {
    // ================================================================== raw rows: global -> staging half-stages
    // lane -> (row r0 + 8 i, 16-byte chunk c): a warp instruction copies eight rows of 64 bytes; the 16 row offsets of a lane in registers
    Prof prof(p.prof, 5);
    uint32_t hseq = 0;
    const int r0 = lane >> 2, c = lane & 3;
    const uint32_t stride16 = (uint32_t)(p.stride >> 3);
    const uint4 *in16 = reinterpret_cast<const uint4 *>(p.in);
    for (uint32_t rb = blockIdx.x; rb < n_rb; rb += gridDim.x) {
      const uint32_t *rmap = p.tc_rowmap + (size_t)rb * M;
      uint32_t rows[M / 8];
#pragma unroll
      for (int i = 0; i < M / 8; ++i) rows[i] = __ldg(rmap + r0 + 8 * i);
      // a list: the same registers hold the rows' chain channels (their history rows) for the stages in front of sample 0, then
      // the launch rows again (a second set of offsets beside them spilled)
      if constexpr (kList) {
#pragma unroll
        for (int i = 0; i < M / 8; ++i) rows[i] = rows[i] != kPad ? chan_of<true>(p, rows[i]) : kPad;
      }
      for (int hh = -2 * (int)(KS - 1); hh < 2 * (int)NT; ++hh, ++hseq) {
        if constexpr (kList) {
          if (hh == 0) {
#pragma unroll
            for (int i = 0; i < M / 8; ++i) rows[i] = __ldg(p.tc_rowmap + (size_t)rb * M + r0 + 8 * i);
          }
        }
        const uint32_t stage = hseq % RSH;
        prof.start();
        mbar_wait(&pc->raw_free[stage], ((hseq / RSH) & 1u) ^ 1u, kNsLoad);
        prof.lap(0);
        const uint32_t dst0 = smem_u32(sRaw + stage * kHalfBytes) + (uint32_t)r0 * HP + (uint32_t)c * 16u;
        if (p.ablate & 1u) {
        } else if (hh >= 0) {
          const uint32_t col16 = (uint32_t)hh * (HU / 8) + (uint32_t)c; // this lane's chunk of the half tile, in 16-byte units
#pragma unroll
          for (int i = 0; i < M / 8; ++i) {
            const bool valid = rows[i] != kPad;
            const uint4 *src = in16 + ((size_t)(valid ? rows[i] : 0u) * stride16 + col16);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst0 + (uint32_t)i * 8u * HP), "l"(src), "r"(valid ? 16 : 0) : "memory");
          }
        } else { // in front of sample 0: the carried history, or zeros beyond the taps' reach
          const int s = hh * HU + 8 * c; // first sample of this lane's chunk (negative)
#pragma unroll
          for (int i = 0; i < M / 8; ++i) {
            const bool valid = rows[i] != kPad && s >= -Hs;
            const size_t hc = kList ? (size_t)rows[i] : (size_t)p.ch0 + rows[i];
            const int16_t *src = valid ? p.hist + hc * p.H + (Hs + s) : p.in; // never dereferenced when the size is 0
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst0 + (uint32_t)i * 8u * HP), "l"(src), "r"(valid ? 16 : 0) : "memory");
          }
        }
        asm volatile("cp.async.mbarrier.arrive.noinc.shared.b64 [%0];" ::"r"(smem_u32(&pc->raw_full[stage])) : "memory");
        prof.lap(1);
      }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    prof.flush();
  } else if (warp >= kConv0 && warp < kConv0 + 4) {
    // ================================================================== byte planes: one half-stage -> one K-block of a ring entry
    Prof prof(p.prof, 0);
    const uint32_t r = (uint32_t)(tid - kConv0 * 32); // row
    uint32_t hseq = 0, pseq = 0, nblk = 0;
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
      for (uint32_t u = 0; u < nhalf; ++u, ++hseq) {
        const uint32_t stage = hseq % RSH, kb = u & 1u, pos = pseq % ring;
        prof.start();
        mbar_wait(&pc->raw_full[stage], (hseq / RSH) & 1u, kNsConv);
        prof.lap(0);
        if (kb == 0) mbar_wait(&pc->blk_free[pos], ((pseq / ring) & 1u) ^ 1u, kNsConv);
        prof.lap(1);
        if (!(p.ablate & 1u)) {
          const uint32_t a = smem_u32(sRaw + stage * kHalfBytes) + r * HP;
          if constexpr (kAdc) {
            if (u >= 2 * (KS - 1)) { // codes of samples 32 hh .. 32 hh + 31, hh = u - 2 (KS - 1); in front of sample 0 the history is conditioned already
              const uint32_t t0 = (u - 2 * (KS - 1)) * HU;
              if (t0 == 0) fe_row_shift_hist(fr, p);
              fe_row_run<HU / 8>(fr, p, a, t0);
            }
          }
          uint4 v[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) v[j] = lds128(a + 16u * j);
          convert_store(sA, a_plane, pos, kb, r, v);
        }
        fence_proxy_async_smem(); // generic-proxy smem writes -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&pc->raw_free[stage]);
          if (kb) mbar_arrive(&pc->a_full[pos]);
        }
        if (kb) ++pseq;
        prof.lap(2);
      }
      if constexpr (kAdc) {
        fe_row_end(fr); // the history was written as the samples were conditioned
      } else { // carry the last H raw samples of this thread's row: hist <- tail of (hist || in[0..L)), as in msdr_chain_v5.cu
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
    // ================================================================== tensor core (per-branch hand-off as in msdr_chain_v5.cu)
    Prof prof(p.prof, 1);
    IssueCtx ictx;
    issue_init(ictx, sA, a_plane, sB, b_plane);
    uint32_t qbase = 0, tseq = 0, nblk = 0;
    for (uint32_t rb = blockIdx.x; rb < n_rb; rb += gridDim.x, ++nblk) {
      mbar_wait(&pc->b_full, nblk & 1u, 64);
      for (uint32_t t = 0; t < NT; ++t, ++tseq) {
        const uint32_t qt = qbase + t + KS - 1; // newest pair of this tile's window
        prof.start();
        mbar_wait(&pc->a_full[qt % ring], (qt / ring) & 1u, 32);
        prof.lap(0);
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
    // ================================================================== epilogue: TMEM -> demodulated int16 rows in this warp's half-slot
    Prof prof(p.prof, 2);
    const int qd = warp & 3, half = warp >> 2;
    const uint32_t trow = (uint32_t)(qd * 32 + lane);
    const uint32_t lane_addr = tmem + ((uint32_t)(qd * 32) << 16) + (uint32_t)(half * 32);
    uint32_t tseq = 0;
    for (uint32_t rb = blockIdx.x; rb < n_rb; rb += gridDim.x) {
      const uint32_t row = __ldg(p.tc_rowmap + (size_t)rb * M + trow);
      const int kind = row != kPad ? demod_kind_of((int)p.mode[chan_of<kList>(p, row)], p.am_q31) : 0;
      for (uint32_t t = 0; t < NT; ++t, ++tseq) {
        const uint32_t useq = 2u * tseq + (uint32_t)half, slot = useq % NH; // this warp's half-slot of the tile
        uint32_t iq[32];
        prof.start();
        mbar_wait(&pc->tmem_full[0], tseq & 1u, 48);
        prof.lap(0);
        tc_fence_after();
        if (!(p.ablate & 1u)) {
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            uint32_t ai[8];
            drain8(lane_addr + (uint32_t)(8 * b), ai);
#pragma unroll
            for (int j = 0; j < 8; ++j) iq[8 * b + j] = (uint32_t)((int)ai[j] >> 15); // saturated together with Q below
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) iq[j] = 0u;
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&pc->tmem_empty[0]); // the next tile's I products may start
        mbar_wait(&pc->tmem_full[1], tseq & 1u, 48);
        tc_fence_after();
        if (!(p.ablate & 1u)) {
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            uint32_t aq[8];
            drain8(lane_addr + (uint32_t)(kAccPerBranch * N + 8 * b), aq);
#pragma unroll
            for (int j = 0; j < 8; ++j) iq[8 * b + j] = pack_sat_iq((int)iq[8 * b + j], (int)aq[j] >> 15);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&pc->tmem_empty[1]);
        prof.lap(1);
        uint32_t out[16];
        if (kind <= 1) demod_ssb_regs(iq, kind ? 0u : 0xFFFF0000u, kind ? 0u : 0x10000u, out);
        else if (kind == 2) demod_regs<2>(iq, 0, out);
        else demod_regs<3>(iq, 0, out);
        mbar_wait(&pc->slot_free[slot], ((useq / NH) & 1u) ^ 1u, kNsSlot);
        prof.lap(2);
        const uint32_t ya = smem_u32(sY + slot * kHalfBytes) + trow * HP;
#pragma unroll
        for (int j = 0; j < 4; ++j) sts128(ya + 16u * j, make_uint4(out[4 * j], out[4 * j + 1], out[4 * j + 2], out[4 * j + 3]));
        __syncwarp();
        if (lane == 0) mbar_arrive(&pc->y_full[slot][qd]);
        prof.lap(3);
      }
    }
    prof.flush();
    named_bar_sync(2, kEpiWarps * 32); // every epilogue warp has read its last accumulators
    if (warp == 0) {
      tc_fence_before();
      tmem_dealloc_512(tmem);
    }
  } else if (warp >= kBqA0 && warp < kBqB0 + 4) {
    // ================================================================== biquad objects: lane = row, state in registers, half-slots in time order
    const bool isA = warp < kBqB0;
    const int obj = isA ? 0 : 1, q = isA ? warp - kBqA0 : warp - kBqB0;
    Prof prof(q == 0 ? p.prof : nullptr, isA ? 3 : 4);
    const uint32_t trow = (uint32_t)(q * 32 + lane);
    uint32_t useq = 0;
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
        sym = fast && __all_sync(0xffffffffu, !active || st[0].b0 == st[0].b2);
        if (sym && active) {
          static_cast<BqStage &>(ss[0]) = static_cast<const BqStage &>(st[0]);
          ss[0].p1 = __mulhi(st[0].b0, st[0].x1);
          ss[0].p2 = __mulhi(st[0].b0, st[0].x2);
        }
      }
      for (uint32_t u = 0; u < 2 * NT; ++u, ++useq) {
        const uint32_t slot = useq % NH, phs = (useq / NH) & 1u;
        prof.start();
        mbar_wait(isA ? &pc->y_full[slot][q] : &pc->ab_full[slot][q], phs, kNsBq);
        prof.lap(0);
        const uint32_t ya = smem_u32(sY + slot * kHalfBytes) + trow * HP;
        if (!(p.ablate & 2u) && active) {
          if (sym) bq_tile<typename std::conditional<kHasSym, SYM, BqStageWS>::type, HU / 8>(ss, ya);
          else if (fast) bq_tile<BQ, HU / 8>(st, ya);
          else { // generic cascade: stage-major over the unit like the reference (filter_biquad.cpp:44-79); state in global
            for (int j = 0; j < nst; ++j) {
              BQ gs[1];
              uint32_t gf;
              bq_load_stage(gs[0], gf, p.bq, p.Cpad, obj, j, ch);
              bq_tile<BQ, HU / 8>(gs, ya);
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
    // ================================================================== final audio: half-slot -> `out`, 64 B per row and unit
    Prof prof(p.prof, 6);
    const int r0 = lane >> 2, c = lane & 3;
    const uint32_t stride16 = (uint32_t)(p.stride >> 3);
    uint4 *out16 = reinterpret_cast<uint4 *>(p.out);
    uint32_t useq = 0;
    for (uint32_t rb = blockIdx.x; rb < n_rb; rb += gridDim.x) {
      const uint32_t *rmap = p.tc_rowmap + (size_t)rb * M;
      uint32_t rows[M / 8];
#pragma unroll
      for (int i = 0; i < M / 8; ++i) rows[i] = __ldg(rmap + r0 + 8 * i);
      for (uint32_t u = 0; u < 2 * NT; ++u, ++useq) {
        const uint32_t slot = useq % NH, phs = (useq / NH) & 1u;
        prof.start();
        mbar_wait(&pc->st_full[slot], phs, kNsStore);
        prof.lap(0);
        const uint32_t sa = smem_u32(sY + slot * kHalfBytes) + (uint32_t)r0 * HP + (uint32_t)c * 16u;
        const uint32_t col16 = u * (HU / 8) + (uint32_t)c;
#pragma unroll
        for (int i0 = 0; i0 < M / 8; i0 += 4) {
          uint4 v[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) v[k] = lds128(sa + (uint32_t)(i0 + k) * 8u * HP);
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

} // namespace v5l

// deepest operand ring (at least one pair ahead of the window) that fits next to the half-size staging and slots; 0 = does not fit
uint32_t chain_v5l_config(uint32_t K, int smem_max)
{
  if (K % 32u || K / 32u < 2u) return 0;
  for (uint32_t ring = tc::RING_MAX; ring >= K / 32u + 1u; --ring)
    if (v5l::smem_bytes(K, ring) <= (size_t)smem_max) return ring;
  return 0;
}

cudaError_t launch_chain_v5l(const ChainParams &p_in, cudaStream_t stream, int variant, int sms, ChainLaunchInfo *info)
{
  using namespace v5l;
  ChainParams p = p_in;
  p.ablate = ((uint32_t)variant >> 4) & 3u;
  const size_t smem = smem_bytes(p.tc_K, p.tc_ring);
  // variant bit 0: all five products as IMAD.HI (cross-check)
  auto kern = p.fe ? chain_kernel<BqStageW, true> : p.chlist ? chain_kernel<BqStageW, false, true> : (variant & 1) ? chain_kernel<BqStage, false> : chain_kernel<BqStageW, false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const uint32_t grid = p.n_items < (uint32_t)sms ? p.n_items : (uint32_t)sms;
  if (info) { info->grid = (int)grid; info->block = kThreads; info->smem = smem; info->tile = tc::N; }
  kern<<<grid, kThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

} // namespace msdr
