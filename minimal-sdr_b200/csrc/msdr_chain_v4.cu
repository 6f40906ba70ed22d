// msdr_chain_v4.cu — K1 (tensor-core form): the fused receive chain with the FIR pair on tcgen05.mma kind::i8.
//
//   int16 IF samples -> [fs/4 mix folded into the byte planes] -> FIR pair as four int8 Toeplitz GEMMs per branch
//   (exact mod 2^32, msdr_fir_tc.cu) -> >>15, SSAT16 -> SSB sum / AM envelope -> biquad cascade -> int16 audio
//
// Reference semantics: Minimal-SDR.ino:546-558 (mix), arm_fir_fast_q15.c:60-329 (FIR), Minimal-SDR.ino:589-628 (demod),
// filter_biquad.cpp:33-82 (biquad).
//
// FIR work and biquad chains are decoupled — FIR work is produced by any SM, biquad chains are pinned to an SM for the whole
// launch and only ever wait for their own input — but the FIR producers are a tensor-core pipeline, which takes the FIR off
// the integer/FP64 issue slots the serial biquad recurrence needs.  One persistent CTA per SM, 16 warps, roles by warp id
// (warp id % 4 = SM sub-partition).  Default shape (POST; the others are listed at `Roles` below):
//
//   warps 0-3          epilogue  TMEM lane quadrant = warp id % 4 (hardware rule): thread = channel row.  tcgen05.ld, recombine
//                                the byte-plane products, >>15, SSAT16, park packed (I, Q) in one of two staging buffers, hand
//                                TMEM back to the MMA warp.  Nothing else: these warps are pinned next to the chain warps.
//   warps 10,11,14,15  post      warp i serves epilogue warp i: demodulate the parked rows, coalesced store of its 32 x 64 part
//                                of the tile to `out` (used as the intermediate buffer), count the rows into
//                                tile_cnt[group][unit] (threadfence + atomic = release).
//   warp 6             MMA       one thread issues 2 branches x 4 byte-plane products x K/32 MMAs (M128 N64 K32) per tile;
//                                tcgen05.commit -> mbarriers.
//   warps 7,12,13      convert   raw int16 (global / carried history) -> sign-folded byte planes in a ring of A operands, each
//                                window word converted once per work item, all loads of a ring entry in flight together.
//   warp 8             load      waits for tile_cnt (relaxed polls, one acquire fence for all units that are complete), then
//                                cp.async of 128-sample sub-tiles of the group's 32 rows into a 5-slot ring, two ahead.
//   warps 4, 5         chains    biquad object 1 / object 2 of channel group g = wave * grid + blockIdx (lane = channel, state
//                                in registers), a two-warp stage pipeline over the ring, in place in shared memory.
//   warp 9             store     final audio, slot -> `out`.
//
// A FIR work item = (row block of 128 channels sharing one tap table, span of 512 samples); items are claimed from a global
// counter in wave-major, then time-major order so that a chain's input is produced while it runs.  Rows are gathered through
// a row map (channels sorted by tap table inside each wave, msdr_capi.cu::build_tc_plan); readiness is counted per group and
// 128-sample unit, so a chain starts on a span after its first two tiles.
#include "msdr_chain_common.cuh"
#include "msdr_tc_common.cuh"

namespace msdr {
namespace v4 {

using namespace tc;

constexpr int SPAN = 512;          // samples per FIR work item
constexpr uint32_t kLead = 6;      // spans the FIR producers may run ahead of the chains (148 items in flight are ~5 spans by themselves)
constexpr int UNIT = 128;          // samples per readiness counter: a chain starts on a span after its first two tiles
// chain sub-tile ring: one slot being filtered by warp A, one by warp B, one draining to `out`, two landing.  With fewer
// slots the load of a sub-tile can only be issued when it is already needed and its latency (~2 k cycles) is paid per sub-tile.
constexpr int NSLOT = 5;
// sub-tile length p.sub = 128 samples (64 for windows K > 128, where the B operand needs the room); row pitch sub/2 + 4 words
// (4 mod 32: conflict-free row-wise LDS.128)
constexpr int kChainA = 4, kChainB = 5, kMmaWarp = 6, kStoreWarp = 9;
constexpr int kThreads = 16 * 32;
// Two shapes of the chain side (template parameter FF):
//   classic  load (warp 8) -> A -> B -> store: every warp runs whole biquad stages; 3 convert warps (7,12,13) and 4 post warps
//            (10,11,14,15) that demodulate and write back what the epilogue warps drained, so that the epilogue warps, which
//            the TMEM lane rule pins next to the chain warps, do as little as possible
//   DUAL     classic without post warps, but TWO chain sets per SM (load 12 -> A 10 -> B 11 -> store 13 is the second): for more
//            channel groups than SMs, where one chain pair per SM is the ceiling (~170 Gsamples/s); 3 convert warps (7,14,15)
//   FF       the three input-side products of a stage do not depend on its output, so they are taken off the chain warps:
//            raw loader (warp 8) -> FF1 (warp 10) -> A -> FF2 (warp 11) -> B -> store.  Warps 10/11 (sub-partitions 2, 3) hand the
//            chain warps the feed-forward sums e[n] as 32-bit words and A/B run only the two recurrence products per sample
//            (tools/microbench/lat.cu: 24 instead of 38 cycles per step isolated).  5 convert warps (7,12,13,14,15).  The default
//            up to one channel group per SM.
template <bool FF, bool POST, bool DUAL = false> struct Roles {
  static_assert(!(FF && POST) && !(DUAL && (FF || POST)), "shapes are exclusive: every warp has one role");
  static constexpr int NCONV = FF ? 5 : (POST || DUAL) ? 3 : 5;
  static constexpr int NPOST = POST ? 4 : 0;     // warps 10,11,14,15 take demodulation + write-back off the epilogue warps
  static constexpr int NSTAGE = POST ? 2 : 1;    // staging buffers between epilogue and post warps
  static constexpr int kLive = (4 + 1 + NCONV + NPOST) * 32;
  static constexpr int kLoadWarp = FF ? 10 : 8;  // FF helpers sit on different sub-partitions (2 and 3): each saturates an IMAD.HI pipe for a while
  static constexpr int kMidWarp = FF ? 11 : -1;
  static constexpr int kRawWarp = FF ? 8 : -1;   // FF: the raw rows are fetched by a warp of their own, FF1 only computes
  // converters wait on memory, not on issue slots: in the classic shape two of them sit next to the chain warps (12, 13)
  static __device__ __forceinline__ bool is_conv(int w)
  {
    return FF ? (w == 7 || w == 12 || w == 13 || w == 14 || w == 15) : DUAL ? (w == 7 || w == 14 || w == 15) : POST ? (w == 7 || w == 12 || w == 13) : (w == 7 || w == 10 || w == 11 || w == 14 || w == 15);
  }
  static __device__ __forceinline__ int conv_index(int w)
  {
    return FF ? (w == 7 ? 0 : w == 12 ? 1 : w == 13 ? 2 : w == 14 ? 3 : 4) : DUAL ? (w == 7 ? 0 : w == 14 ? 1 : 2) : POST ? (w == 7 ? 0 : w == 12 ? 1 : 2) : (w == 7 ? 0 : w == 10 ? 1 : w == 11 ? 2 : w == 14 ? 3 : 4);
  }
  // classic chain side: which chain set (0, or 1 in the DUAL shape) and which role (0 load, 1 A, 2 B, 3 store) a warp has
  static __device__ __forceinline__ void chain_role(int w, int &set, int &role)
  {
    set = role = -1;
    if (w == 8) { set = 0; role = 0; } else if (w == 4) { set = 0; role = 1; } else if (w == 5) { set = 0; role = 2; } else if (w == 9) { set = 0; role = 3; }
    if (DUAL) { // the second chain pair sits on sub-partitions 2 and 3, its I/O warps on 0 and 1
      if (w == 12) { set = 1; role = 0; } else if (w == 10) { set = 1; role = 1; } else if (w == 11) { set = 1; role = 2; } else if (w == 13) { set = 1; role = 3; }
    }
  }
  static __device__ __forceinline__ bool is_post(int w) { return POST && (w == 10 || w == 11 || w == 14 || w == 15); }
  static __device__ __forceinline__ int post_index(int w) { return w == 10 ? 2 : w == 11 ? 3 : w == 14 ? 0 : 1; } // post warp i serves epilogue warp i
};
constexpr int NSLOT_FF = 7, SUB_FF = 64; // load, FF1, A, FF2, B, store each hold a slot in steady state; one more decouples them
constexpr int EW = SUB_FF + 4, YW = SUB_FF / 2 + 4;                    // FF slot: e[n] rows (32-bit) and packed int16 rows, word pitches
constexpr uint32_t kSlotBytesFF = kGroup * (EW + YW) * 4u;
constexpr int NSLOT_MAX = 10; // FF: 7 slots; DUAL: 2 sets x 5
__host__ __device__ inline uint32_t slot_bytes(uint32_t sub) { return kGroup * (sub / 2 + 4) * 4u; }
constexpr uint32_t kCtrlBytes = 1536;


struct __align__(16) Ctrl {
  uint64_t a_full[RING_MAX];   // convert -> MMA   : pair converted (NCONV arrivals)
  uint64_t blk_free[RING_MAX]; // MMA -> convert   : pair no longer read (tcgen05.commit)
  uint64_t tmem_full;          // MMA -> epilogue  : accumulators complete (tcgen05.commit)
  uint64_t tmem_empty;         // epilogue -> MMA  : accumulators drained (4 arrivals)
  uint64_t staged_full[2][4];  // epilogue warp i -> post warp i : packed I/Q rows parked in staging buffer b (classic)
  uint64_t staged_free[2][4];  // post warp i -> epilogue warp i : staging buffer b written back
  uint64_t raw_full[NSLOT_MAX];  // raw loader -> FF1 (FF only): the sub-tile's cp.async copies have landed (32 arrivals)
  uint64_t ld_full[NSLOT_MAX];   // load -> chain A  : sub-tile in smem
  uint64_t ab_full[NSLOT_MAX];   // chain A -> B (classic) / chain A -> FF2 (FF) : object 1 done
  uint64_t m_full[NSLOT_MAX];    // FF2 -> chain B   : feed-forward sums of object 2 ready (FF only)
  uint64_t st_full[NSLOT_MAX];   // chain B -> store : object 2 done
  uint64_t slot_free[NSLOT_MAX]; // store -> load    : final audio written back, slot reusable
  uint32_t tmem_base;
  int item_rb[2], item_span[2]; // work item of the even / odd iteration (rb < 0: done)
  uint32_t rowmap[M];           // rows of the current item (written by the epilogue threads)
};
static_assert(sizeof(Ctrl) <= kCtrlBytes, "Ctrl must fit its smem slot");

uint32_t sub_for(uint32_t K) { return K > 128 ? 64 : 128; }
size_t smem_bytes(uint32_t K, uint32_t ring, bool ff, bool post, bool dual = false)
{
  const size_t slots = ff ? (size_t)NSLOT_FF * kSlotBytesFF : (size_t)(dual ? 2 : 1) * NSLOT * slot_bytes(sub_for(K));
  return (size_t)kCtrlBytes + 4u * a_plane_bytes(ring) + 4u * N * K + (post ? 2u : 1u) * kStagingBytes + slots + 1024u;
}

// developer profile (MSDR_PROF=1): per-CTA cycle totals, slot = role * 4 + counter
struct Prof {
  long long *base;
  long long acc[4];
  long long t;
  __device__ __forceinline__ Prof(long long *b, int role) : base(b ? b + (size_t)blockIdx.x * 64 + role * 4 : nullptr), acc{0, 0, 0, 0}, t(0) {}
  __device__ __forceinline__ void start() { if (base) t = clock64(); }
  __device__ __forceinline__ void lap(int i) { if (base) { const long long n = clock64(); acc[i] += n - t; t = n; } }
  __device__ __forceinline__ void flush() { if (base && (threadIdx.x & 31) == 0) for (int i = 0; i < 4; ++i) base[i] = acc[i]; }
};
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

__device__ __forceinline__ uint4 lds128(uint32_t a)
{
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t a, const uint4 &v)
{
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// one sub-tile of one chain row, in place in shared memory; nq (uint4 = 8 samples each) is even.  Two register sets alternate,
// so the next eight samples are on their way while the recurrence runs and no register moves sit in the loop.
template <class BQ>
__device__ __forceinline__ void chain_span(BQ (&st)[1], uint4 *row, int nq)
{
  const uint32_t a = smem_u32(row);
  uint4 v0 = lds128(a), v1;
#pragma unroll 1
  for (int q = 0; q < nq; q += 2) {
    v1 = lds128(a + 16u * (uint32_t)(q + 1));
    v0.x = bq_word<1>(st, v0.x);
    v0.y = bq_word<1>(st, v0.y);
    v0.z = bq_word<1>(st, v0.z);
    v0.w = bq_word<1>(st, v0.w);
    sts128(a + 16u * (uint32_t)q, v0);
    if (q + 2 < nq) v0 = lds128(a + 16u * (uint32_t)(q + 2));
    v1.x = bq_word<1>(st, v1.x);
    v1.y = bq_word<1>(st, v1.y);
    v1.z = bq_word<1>(st, v1.z);
    v1.w = bq_word<1>(st, v1.w);
    sts128(a + 16u * (uint32_t)(q + 1), v1);
  }
}

template <bool FF, bool POST, bool DUAL>
__global__ void __launch_bounds__(kThreads, 1) chain_kernel(const ChainParams p)
{
  using BQ = BqStage;
  using R = Roles<FF, POST, DUAL>;
  constexpr int NCONV = R::NCONV, kLive = R::kLive, kLoadWarp = R::kLoadWarp;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // the operand rings want 128-byte alignment; round the dynamic window up to 1 KB to be independent of the static layout
  unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023u) & ~(uintptr_t)1023u);
  const uint32_t K = p.tc_K, KS = K / 32, ring = p.tc_ring;
  const uint32_t a_plane = a_plane_bytes(ring), b_plane = N * K;
  Ctrl *pc = reinterpret_cast<Ctrl *>(smem);
  uint8_t *sA = smem + kCtrlBytes;
  uint8_t *sB = sA + 4 * a_plane;
  uint32_t *sOut = reinterpret_cast<uint32_t *>(sB + 4 * b_plane);
  unsigned char *bq_base = reinterpret_cast<unsigned char *>(sOut) + R::NSTAGE * kStagingBytes;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int i = 0; i < RING_MAX; ++i) { mbar_init(&pc->a_full[i], NCONV); mbar_init(&pc->blk_free[i], 1); }
    mbar_init(&pc->tmem_full, 1);
    mbar_init(&pc->tmem_empty, 4);
    for (int b = 0; b < 2; ++b)
      for (int i = 0; i < 4; ++i) { mbar_init(&pc->staged_full[b][i], 1); mbar_init(&pc->staged_free[b][i], 1); }
    for (int s = 0; s < NSLOT_MAX; ++s) {
      mbar_init(&pc->raw_full[s], 32);
      mbar_init(&pc->ld_full[s], 1); mbar_init(&pc->ab_full[s], 1); mbar_init(&pc->m_full[s], 1); mbar_init(&pc->st_full[s], 1); mbar_init(&pc->slot_free[s], 1);
    }
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc_512(&pc->tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = pc->tmem_base;
  const bool is_epi = warp < 4, is_mma = warp == kMmaWarp, is_conv = R::is_conv(warp), is_post = R::is_post(warp);

  if (is_epi || is_mma || is_conv || is_post) {
    // ================================================================== FIR + demod producers (tensor-core pipeline)
    Prof prof(p.prof, is_conv ? 0 : is_mma ? 1 : is_post ? 7 : 2);
    IssueCtx ictx;
    issue_init(ictx, sA, a_plane, sB, b_plane);
    uint32_t q = 0;     // pairs converted so far by this CTA (ring position q % ring, phase q / ring)
    uint32_t ntile = 0; // tiles processed so far by this CTA (TMEM hand-off phases)
    int cur_set = -1;
    uint32_t cur_wave = 0, wave_item0 = 0, wave_spans0 = 0; // claiming thread only
    const uint32_t n_tiles = p.L / N;
    for (uint32_t iter = 0;; ++iter) {
      if (is_mma && lane == 0) {
        const uint32_t it = (uint32_t)atomicAdd(&p.ctrl[0], 1);
        int rb = -1, span = 0;
        if (it < p.n_items) {
          for (;;) { // items are claimed in increasing order: walk the waves forward
            const uint32_t nrb = p.tc_wave_rb0[cur_wave + 1] - p.tc_wave_rb0[cur_wave];
            const uint32_t wgroups = min(p.W, p.NG - cur_wave * p.W); // chains of this wave
            if (it - wave_item0 < nrb * p.NT) {
              const uint32_t rem = it - wave_item0;
              span = (int)(rem / nrb);
              rb = (int)(p.tc_wave_rb0[cur_wave] + (rem - (uint32_t)span * nrb));
              // flow control: the demodulated intermediate lives in `out` and should still be in L2 when its chain reads it, so
              // the producers stay at most kLead spans ahead of the chains (p.ctrl[1] counts the spans the loaders have taken;
              // everything before a claimed item is being produced, so the chains always get to within one span of it)
              if ((uint32_t)span > kLead) {
                const int want = (int)(wave_spans0 + wgroups * ((uint32_t)span - kLead));
                const long long t0 = clock64();
                while (ld_relaxed_gpu(p.ctrl + 1) < want) {
                  __nanosleep(256);
                  if (clock64() - t0 > kWatchdogCycles) __trap();
                }
              }
              break;
            }
            wave_item0 += nrb * p.NT;
            wave_spans0 += wgroups * p.NT;
            ++cur_wave;
          }
        }
        pc->item_rb[iter & 1] = rb;
        pc->item_span[iter & 1] = span;
      }
      prof.start();
      named_bar_sync(1, kLive); // item visible; every producer role has finished the previous item
      prof.lap(3);
      const int rb = pc->item_rb[iter & 1];
      if (rb < 0) break;
      const uint32_t span = (uint32_t)pc->item_span[iter & 1];
      const uint32_t tb = span * (SPAN / N), te = min(tb + SPAN / N, n_tiles);
      const uint32_t qbase = q;
      const uint32_t npairs = (te - tb) + KS - 1;
      const uint4 rbi = __ldg(p.tc_rb + rb); // x: table id (the other words are 0)
      const uint32_t *rmap = p.tc_rowmap + (size_t)rb * M;

      if (is_conv) {
        const int ctid = R::conv_index(warp) * 32 + lane;
        if ((int)rbi.x != cur_set) { // (re)load the Toeplitz operand of this table; the pipeline is drained at item boundaries
          const uint4 *src = reinterpret_cast<const uint4 *>(p.tc_bmat + (size_t)rbi.x * 4 * b_plane);
          uint4 *dst = reinterpret_cast<uint4 *>(sB);
          for (uint32_t i = ctid; i < 4 * b_plane / 16; i += NCONV * 32) dst[i] = __ldg(src + i);
          cur_set = (int)rbi.x;
        }
        // this thread's conversion tasks: (row r, K-block kb) of every pair, 2 * M tasks over NCONV warps
        constexpr int NTASK = (2 * M + NCONV * 32 - 1) / (NCONV * 32);
        uint32_t trow[NTASK];
#pragma unroll
        for (int i = 0; i < NTASK; ++i) {
          const uint32_t task = ctid + i * NCONV * 32;
          trow[i] = task < 2 * M ? __ldg(rmap + task % M) : 0xFFFFFFFFu;
        }
        const int Hs = (int)p.H;
        auto load16 = [&](uint32_t row, long long s0, uint4 (&v)[4]) { // 32 samples from sample index s0 (may be negative: history)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const long long s = s0 + 8 * j;
            if (row == 0xFFFFFFFFu || s < -(long long)Hs) v[j] = make_uint4(0, 0, 0, 0); // padding row / beyond the taps' reach
            else if (s >= 0) v[j] = __ldg(reinterpret_cast<const uint4 *>(p.in + (size_t)row * p.stride + s));
            else v[j] = __ldcg(reinterpret_cast<const uint4 *>(p.hist + ((size_t)p.ch0 + row) * p.H + (Hs + s)));
          }
        };
        for (uint32_t u = 0; u < npairs; ++u, ++q) {
          const uint32_t pos = q % ring;
          prof.start();
          mbar_wait(&pc->blk_free[pos], ((q / ring) & 1u) ^ 1u);
          prof.lap(0);
          const long long w0 = ((long long)tb - (long long)(KS - 1) + (long long)u) * P; // first window word of the pair
          if (!(p.ablate & 1u)) {
            uint4 v[NTASK][4]; // all loads of the pair in flight together: one memory round trip per pair, not one per task
#pragma unroll
            for (int i = 0; i < NTASK; ++i) {
              const uint32_t task = ctid + i * NCONV * 32;
              if (task < 2 * M) load16(trow[i], 2 * (w0 + 16 * (long long)(task / M)), v[i]);
            }
#pragma unroll
            for (int i = 0; i < NTASK; ++i) {
              const uint32_t task = ctid + i * NCONV * 32;
              if (task < 2 * M) convert_store(sA, a_plane, pos, task / M, task % M, v[i]);
            }
          }
          fence_proxy_async_smem(); // generic-proxy smem writes -> visible to the tensor core (async proxy)
          __syncwarp();
          if (lane == 0) mbar_arrive(&pc->a_full[pos]);
          prof.lap(1);
        }
      } else if (is_mma) {
        q += npairs;
        { // warp-uniform: every lane waits, one elected lane issues (see umma_i8)
          uint32_t nt = ntile;
          for (uint32_t t = tb; t < te; ++t, ++nt) {
            const uint32_t qt = qbase + (t - tb) + KS - 1; // newest pair of this tile's window
            prof.start();
            mbar_wait(&pc->a_full[qt % ring], (qt / ring) & 1u);
            prof.lap(0);
            mbar_wait(&pc->tmem_empty, (nt & 1u) ^ 1u);
            prof.lap(1);
            tc_fence_after();
            if (!(p.ablate & 1u)) issue_tile(ictx, tmem, qt, KS, ring);
            umma_commit(&pc->tmem_full);
            umma_commit(&pc->blk_free[(qt - (KS - 1)) % ring]); // the oldest pair of the window is not read again
            prof.lap(2);
          }
          for (uint32_t s = 1; s < KS; ++s) umma_commit(&pc->blk_free[(qbase + npairs - KS + s) % ring]);
        }
        ntile += te - tb;
        __syncwarp();
      } else if (POST && is_epi) { // epilogue with post warps: drain only.  thread = channel row (TMEM lane)
        q += npairs;
        const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
        for (uint32_t t = tb; t < te; ++t, ++ntile) {
          const uint32_t buf = ntile & 1u, use = ntile >> 1;
          prof.start();
          mbar_wait(&pc->tmem_full, ntile & 1u);
          prof.lap(0);
          tc_fence_after();
          mbar_wait(&pc->staged_free[buf][warp], (use & 1u) ^ 1u); // the post warp has written this buffer back
          prof.lap(1);
          if (!(p.ablate & 1u)) drain_tile(lane_addr, sOut + buf * (kStagingBytes / 4) + (uint32_t)tid * OW);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            mbar_arrive(&pc->tmem_empty);           // the next tile's MMAs may start
            mbar_arrive(&pc->staged_full[buf][warp]);
          }
          prof.lap(2);
        }
      } else if (is_post) { // demodulation + write-back of the 32 rows epilogue warp `pw` parked
        q += npairs;
        const int pw = R::post_index(warp);
        const uint32_t prow = (uint32_t)(pw * 32 + lane);
        const uint32_t row = __ldg(rmap + prow);
        pc->rowmap[prow] = row;
        const int kind = row != 0xFFFFFFFFu ? demod_kind_of((int)p.mode[p.ch0 + row], p.am_q31) : 0;
        const uint32_t grp = row != 0xFFFFFFFFu ? row / kGroup : 0xFFFFFFFFu;
        const unsigned peers = __match_any_sync(0xffffffffu, grp); // lanes of this warp whose rows belong to the same channel group
        const bool leader = grp != 0xFFFFFFFFu && lane == __ffs(peers) - 1;
        const int npeers = __popc(peers);
        for (uint32_t t = tb; t < te; ++t, ++ntile) {
          const uint32_t buf = ntile & 1u, use = ntile >> 1;
          uint32_t *orow = sOut + buf * (kStagingBytes / 4) + prow * OW;
          const uint32_t *wrow = sOut + buf * (kStagingBytes / 4) + (uint32_t)(pw * 32) * OW;
          prof.start();
          mbar_wait(&pc->staged_full[buf][pw], use & 1u);
          prof.lap(0);
          if (!(p.ablate & 1u)) demod_row(orow, kind);
          __syncwarp();
          for (uint32_t i = lane; i < 32 * (N / 8) && !(p.ablate & 1u); i += 32) { // coalesced write-back: 32 rows x 128 bytes
            const uint32_t r = i / (N / 8), c = i % (N / 8);
            const uint32_t orow_g = pc->rowmap[pw * 32 + r];
            if (orow_g != 0xFFFFFFFFu)
              *reinterpret_cast<uint4 *>(p.out + (size_t)orow_g * p.stride + (size_t)t * N + c * 8) = *reinterpret_cast<const uint4 *>(wrow + r * OW + c * 4);
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&pc->staged_free[buf][pw]);
          prof.lap(1);
          if ((((t + 1) * N) % UNIT) == 0) { // publish: these rows have the unit in `out`
            __threadfence();
            __syncwarp();
            if (leader) atomicAdd(p.tile_cnt + (size_t)grp * p.NU + (t * N) / UNIT, npeers);
          }
          prof.lap(2);
        }
      } else { // epilogue without post warps: thread = channel row (TMEM lane).  The four warps only meet at the TMEM hand-off: every warp parks,
               // demodulates, writes back and publishes its own 32 rows.
        q += npairs;
        const uint32_t row = __ldg(rmap + tid);
        pc->rowmap[tid] = row;
        const int kind = row != 0xFFFFFFFFu ? demod_kind_of((int)p.mode[p.ch0 + row], p.am_q31) : 0;
        const uint32_t grp = row != 0xFFFFFFFFu ? row / kGroup : 0xFFFFFFFFu;
        const unsigned peers = __match_any_sync(0xffffffffu, grp); // lanes of this warp whose rows belong to the same channel group
        const bool leader = grp != 0xFFFFFFFFu && lane == __ffs(peers) - 1;
        const int npeers = __popc(peers);
        const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
        uint32_t *orow = sOut + (uint32_t)tid * OW;
        const uint32_t *wrow = sOut + (uint32_t)(warp * 32) * OW;
        for (uint32_t t = tb; t < te; ++t, ++ntile) {
          prof.start();
          mbar_wait(&pc->tmem_full, ntile & 1u);
          prof.lap(0);
          tc_fence_after();
          if (!(p.ablate & 1u)) drain_tile(lane_addr, orow);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&pc->tmem_empty); // the next tile's MMAs overlap the demodulation
          prof.lap(1);
          if (!(p.ablate & 1u)) demod_row(orow, kind);
          __syncwarp();
          for (uint32_t i = lane; i < 32 * (N / 8) && !(p.ablate & 1u); i += 32) { // coalesced write-back: 32 rows x 128 bytes
            const uint32_t r = i / (N / 8), c = i % (N / 8);
            const uint32_t orow_g = pc->rowmap[warp * 32 + r];
            if (orow_g != 0xFFFFFFFFu)
              *reinterpret_cast<uint4 *>(p.out + (size_t)orow_g * p.stride + (size_t)t * N + c * 8) = *reinterpret_cast<const uint4 *>(wrow + r * OW + c * 4);
          }
          if ((((t + 1) * N) % UNIT) == 0) { // publish: these rows have the unit in `out`
            __threadfence();
            __syncwarp();
            if (leader) atomicAdd(p.tile_cnt + (size_t)grp * p.NU + (t * N) / UNIT, npeers);
          }
          __syncwarp(); // the staging rows are rewritten by the next drain
          prof.lap(2);
        }
      }
    }
    if (warp == 0 || warp == kMmaWarp || warp == 7 || warp == 14) prof.flush();
    if (warp == 0) {
      tc_fence_before();
      tmem_dealloc_512(tmem);
    }
  }

  if constexpr (FF) {
    // ================================================================== FF chain side
    // slot = E rows [32][EW] (32-bit: feed-forward sums, or x << 16 for generic cascades) + Y rows [32][YW] (packed int16)
    const int nsub = (int)(p.L / SUB_FF); // L is a multiple of 128
    auto slotE = [&](int slot) { return reinterpret_cast<uint32_t *>(bq_base + (uint32_t)slot * kSlotBytesFF) + (uint32_t)lane * EW; };
    auto slotY = [&](int slot) { return reinterpret_cast<uint32_t *>(bq_base + (uint32_t)slot * kSlotBytesFF) + kGroup * EW + (uint32_t)lane * YW; };
    // is every lane's object a single stage?  (generic cascades run whole stages in the chain warps, state in global)
    auto object_fast = [&](int obj, uint32_t ch, bool active, int &nst) {
      nst = 1;
      if (active) {
        for (int k = 0; k < 3 && (nst == k + 1); ++k)
          if ((uint32_t)__ldcg(p.bq + (size_t)((obj * 4 + k) * 8 + 7) * p.Cpad + ch) & 0x80000000u) nst = k + 2;
      }
      return __all_sync(0xffffffffu, nst == 1);
    };
    if (warp == kChainA || warp == kChainB) {
      const bool isA = (warp == kChainA);
      const int obj = isA ? 0 : 1;
      Prof prof(p.prof, isA ? 3 : 4);
      uint32_t pos = 0;
      for (int g = (int)blockIdx.x; g < (int)p.NG; g += (int)p.W) {
        const uint32_t row = (uint32_t)(g * kGroup + lane), ch = p.ch0 + row;
        const bool active = row < p.C;
        int nst;
        const bool fast = object_fast(obj, ch, active, nst);
        BqRec rec{};
        uint32_t fl = 0u;
        if (fast && active) bq_load_rec(rec, fl, p.bq, p.Cpad, obj, ch);
        for (int k = 0; k < nsub; ++k, ++pos) {
          const int slot = (int)(pos % NSLOT_FF);
          const uint32_t phs = (pos / NSLOT_FF) & 1u;
          prof.start();
          mbar_wait(isA ? &pc->ld_full[slot] : &pc->m_full[slot], phs, 20);
          prof.lap(0);
          uint32_t *er = slotE(slot), *yr = slotY(slot);
          if (!(p.ablate & 2u) && active) {
            if (fast) {
              const uint32_t ea = smem_u32(er), ya = smem_u32(yr);
              uint4 n0 = lds128(ea), n1 = lds128(ea + 16u);
#pragma unroll 1
              for (int q = 0; q < SUB_FF / 8; ++q) {
                const uint4 e0 = n0, e1 = n1;
                if (q + 1 < SUB_FF / 8) { n0 = lds128(ea + 32u * (uint32_t)(q + 1)); n1 = lds128(ea + 32u * (uint32_t)(q + 1) + 16u); }
                const int y0 = rec_step(rec, (int)e0.x), y1 = rec_step(rec, (int)e0.y), y2 = rec_step(rec, (int)e0.z), y3 = rec_step(rec, (int)e0.w);
                const int y4 = rec_step(rec, (int)e1.x), y5 = rec_step(rec, (int)e1.y), y6 = rec_step(rec, (int)e1.z), y7 = rec_step(rec, (int)e1.w);
                sts128(ya + 16u * (uint32_t)q, make_uint4(__byte_perm((uint32_t)y0, (uint32_t)y1, 0x7632), __byte_perm((uint32_t)y2, (uint32_t)y3, 0x7632),
                                                           __byte_perm((uint32_t)y4, (uint32_t)y5, 0x7632), __byte_perm((uint32_t)y6, (uint32_t)y7, 0x7632)));
              }
            } else { // generic cascade, stage-major like the reference (filter_biquad.cpp:44-79): E holds x << 16, filtered in place
              for (int j = 0; j < nst; ++j) {
                BQ gs;
                uint32_t gf;
                bq_load_stage(gs, gf, p.bq, p.Cpad, obj, j, ch);
                for (int n = 0; n < SUB_FF; ++n) er[n] = (uint32_t)bq_step(gs, (int)er[n]);
                bq_store_stage(gs, gf, p.bq, p.Cpad, obj, j, ch);
              }
              for (int n = 0; n < SUB_FF / 2; ++n) yr[n] = __byte_perm(er[2 * n], er[2 * n + 1], 0x7632);
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(isA ? &pc->ab_full[slot] : &pc->st_full[slot]);
          prof.lap(1);
        }
        if (fast && active) bq_store_rec(rec, fl, p.bq, p.Cpad, obj, ch);
      }
      prof.flush();
    } else if (warp == kLoadWarp || warp == R::kMidWarp) {
      // feed-forward helpers, lane = channel row.  load+FF1: `out` -> e1 (object 1);  FF2: y1 (Y rows) -> e2 (object 2)
      const bool isLoad = (warp == kLoadWarp);
      const int obj = isLoad ? 0 : 1;
      Prof prof(p.prof, isLoad ? 5 : 7);
      uint32_t pos = 0;
      for (int g = (int)blockIdx.x; g < (int)p.NG; g += (int)p.W) {
        const uint32_t row = (uint32_t)(g * kGroup + lane), ch = p.ch0 + row;
        const bool active = row < p.C;
        const int nrows = min(kGroup, (int)p.C - g * kGroup);
        int nst;
        const bool fast = object_fast(obj, ch, active, nst);
        BqFF ff{};
        if (fast && active) bq_load_ff(ff, p.bq, p.Cpad, obj, ch);
        for (int k = 0; k < nsub; ++k, ++pos) {
          const int slot = (int)(pos % NSLOT_FF);
          const uint32_t phs = (pos / NSLOT_FF) & 1u;
          uint32_t *er = slotE(slot);
          uint4 v[SUB_FF / 8];
          prof.start();
          if (isLoad) {
            mbar_wait(&pc->raw_full[slot], phs, 32); // every lane's copies of this sub-tile have landed (raw loader, warp 8)
            prof.lap(0);
            prof.lap(1);
            const uint32_t *yr = slotY(slot);
            if (active) {
#pragma unroll
              for (int j = 0; j < SUB_FF / 8; ++j) v[j] = *reinterpret_cast<const uint4 *>(yr + 4 * j);
            }
          } else {
            mbar_wait(&pc->ab_full[slot], phs, 32);
            prof.lap(0);
            const uint32_t *yr = slotY(slot);
            if (active) {
#pragma unroll
              for (int j = 0; j < SUB_FF / 8; ++j) v[j] = *reinterpret_cast<const uint4 *>(yr + 4 * j);
            }
          }
          if (active && fast) { // branch-free straight-line code: the samples are independent, their DFMA latencies overlap
#pragma unroll
            for (int j = 0; j < SUB_FF / 8; ++j) {
              const uint32_t w[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
              uint32_t e[8];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                e[2 * i] = (uint32_t)ff_step(ff, (int)(short)(w[i] & 0xFFFFu));
                e[2 * i + 1] = (uint32_t)ff_step(ff, (int)w[i] >> 16);
              }
              *reinterpret_cast<uint4 *>(er + 8 * j) = make_uint4(e[0], e[1], e[2], e[3]);
              *reinterpret_cast<uint4 *>(er + 8 * j + 4) = make_uint4(e[4], e[5], e[6], e[7]);
            }
          } else if (active) { // generic cascade: hand x << 16 through
#pragma unroll
            for (int j = 0; j < SUB_FF / 8; ++j) {
              const uint32_t w[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
              *reinterpret_cast<uint4 *>(er + 8 * j) = make_uint4(w[0] << 16, w[0] & 0xFFFF0000u, w[1] << 16, w[1] & 0xFFFF0000u);
              *reinterpret_cast<uint4 *>(er + 8 * j + 4) = make_uint4(w[2] << 16, w[2] & 0xFFFF0000u, w[3] << 16, w[3] & 0xFFFF0000u);
            }
          }
          __syncwarp();
          if (lane == 0) {
            mbar_arrive(isLoad ? &pc->ld_full[slot] : &pc->m_full[slot]);
          }
          prof.lap(2);
        }
        if (fast && active) bq_store_ff(ff, p.bq, p.Cpad, obj, ch);
      }
      prof.flush();
    } else if (warp == R::kRawWarp) {
      // raw loader: the demodulated rows of sub-tile k go `out` -> Y rows of its slot with cp.async (no registers, coalesced: 4 rows
      // of 128 bytes per warp instruction), as far ahead of the feed-forward pass as the slot ring allows; the copies' completion
      // arrives on raw_full[slot] (cp.async.mbarrier.arrive.noinc, one arrival per lane)
      uint32_t pos = 0;
      for (int g = (int)blockIdx.x; g < (int)p.NG; g += (int)p.W) {
        const int nrows = min(kGroup, (int)p.C - g * kGroup);
        int ready = 0; // leading units known to be in `out` for every row of the group
        // all rows of the group have the unit of sub-tile k in `out`?  (blocking or a single poll)
        auto unit_ready = [&](int k, bool blocking) -> bool {
          const int need = (k * SUB_FF) / UNIT;
          while (ready <= need) {
            int ok = 1;
            if (lane == 0) {
              const long long t0 = clock64();
              while (ld_relaxed_gpu(p.tile_cnt + (size_t)g * p.NU + ready) < nrows) {
                if (!blocking) { ok = 0; break; }
                __nanosleep(64);
                if (clock64() - t0 > kWatchdogCycles) __trap();
              }
              if (ok) fence_acquire_gpu();
            }
            ok = __shfl_sync(0xffffffffu, ok, 0);
            if (!ok) return false;
            ++ready;
          }
          return true;
        };
        // load side: the raw rows of sub-tile kk go global -> Y rows of its slot with cp.async (no registers, coalesced: 4 rows of
        // 128 bytes per warp instruction), one sub-tile ahead of the feed-forward pass, so the ~1.3 k-cycle round trip is hidden
        const int cr0 = lane >> 3, cc = lane & 7;
        auto issue_rows = [&](int kk, uint32_t pp, bool blocking) -> bool {
          const int sl = (int)(pp % NSLOT_FF);
          if (!unit_ready(kk, blocking)) return false;
          if (blocking) mbar_wait(&pc->slot_free[sl], ((pp / NSLOT_FF) & 1u) ^ 1u);
          else if (!mbar_test_wait(&pc->slot_free[sl], ((pp / NSLOT_FF) & 1u) ^ 1u)) return false;
          const unsigned char *gsrc = reinterpret_cast<const unsigned char *>(p.out + ((size_t)g * kGroup + cr0) * p.stride + (size_t)kk * SUB_FF) + cc * 16;
          const uint32_t sdst = smem_u32(bq_base + (uint32_t)sl * kSlotBytesFF) + (uint32_t)(kGroup * EW + cr0 * YW) * 4u + cc * 16;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (cr0 + 4 * j < nrows)
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sdst + (uint32_t)j * 4u * YW * 4u), "l"(gsrc + (size_t)j * 4u * p.stride * 2u) : "memory");
          asm volatile("cp.async.commit_group;" ::: "memory");
          return true;
        };
        for (int k = 0; k < nsub; ++k, ++pos) {
          issue_rows(k, pos, true);
          asm volatile("cp.async.mbarrier.arrive.noinc.shared.b64 [%0];" ::"r"(smem_u32(&pc->raw_full[pos % NSLOT_FF])) : "memory");
          if (lane == 0 && ((((k + 1) * SUB_FF) % SPAN) == 0 || k + 1 == nsub)) atomicAdd(p.ctrl + 1, 1); // flow control: span taken
        }
        {
          // carry the last H raw samples: hist <- tail of (hist || in[0..L)).  Every unit of this group has been counted and
          // only a span's first window reaches back into the history, so nobody reads the old history any more.
          const uint32_t hq = p.H >> 3; // uint4 per history row (<= 33)
          for (int r = 0; r < nrows; ++r) {
            const size_t c = (size_t)g * kGroup + (size_t)r;
            uint4 *hrow = reinterpret_cast<uint4 *>(p.hist + ((size_t)p.ch0 + c) * p.H);
            const uint4 *irow = reinterpret_cast<const uint4 *>(p.in + c * p.stride);
            uint4 v0 = make_uint4(0, 0, 0, 0), v1 = v0;
            const uint32_t i0 = (uint32_t)lane, i1 = (uint32_t)lane + 32u;
            if (p.L >= p.H) {
              const uint4 *src = irow + ((p.L - p.H) >> 3);
              if (i0 < hq) v0 = src[i0];
              if (i1 < hq) v1 = src[i1];
            } else {
              const uint32_t lq = p.L >> 3, keep = hq - lq; // keep = old entries that survive
              if (i0 < hq) v0 = (i0 < keep) ? __ldcg(hrow + i0 + lq) : irow[i0 - keep];
              if (i1 < hq) v1 = (i1 < keep) ? __ldcg(hrow + i1 + lq) : irow[i1 - keep];
            }
            __syncwarp();
            if (i0 < hq) hrow[i0] = v0;
            if (i1 < hq) hrow[i1] = v1;
          }
        }
      }
      asm volatile("cp.async.wait_all;" ::: "memory");
    } else if (warp == kStoreWarp) {
      // final audio: Y rows -> `out`, 4 rows of 128 bytes per warp instruction
      Prof prof(p.prof, 6);
      const int r0 = lane >> 3, c = lane & 7;
      const size_t gstep = (size_t)4 * p.stride * 2u;
      uint32_t pos = 0;
      for (int g = (int)blockIdx.x; g < (int)p.NG; g += (int)p.W) {
        const int nrows = min(kGroup, (int)p.C - g * kGroup);
        unsigned char *gp0 = reinterpret_cast<unsigned char *>(p.out + ((size_t)g * kGroup + r0) * p.stride) + c * 16;
        for (int k = 0; k < nsub; ++k, ++pos) {
          const int slot = (int)(pos % NSLOT_FF);
          const uint32_t phs = (pos / NSLOT_FF) & 1u;
          const unsigned char *sp0 = bq_base + (uint32_t)slot * kSlotBytesFF + (uint32_t)(kGroup * EW + r0 * YW) * 4u + c * 16;
          unsigned char *gp = gp0 + (size_t)k * SUB_FF * 2u;
          prof.start();
          mbar_wait(&pc->st_full[slot], phs);
          prof.lap(0);
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (r0 + j * 4 < nrows) *reinterpret_cast<uint4 *>(gp + (size_t)j * gstep) = *reinterpret_cast<const uint4 *>(sp0 + (uint32_t)j * 4u * YW * 4u);
          __syncwarp();
          if (lane == 0) mbar_arrive(&pc->slot_free[slot]);
          prof.lap(1);
        }
      }
      prof.flush();
    }
    return;
  }
  int cset, crole;
  R::chain_role(warp, cset, crole);
  if (cset < 0) return;
  const int ci = cset * (int)gridDim.x + (int)blockIdx.x; // chain index: channel groups ci, ci + p.W, ... (p.W = chains per wave)
  const int sbase = cset * NSLOT;                          // this set's barriers and ring slots
  if (crole == 1 || crole == 2) {
    // ================================================================== biquad chain: warp A = object 1, warp B = object 2
    const bool isA = (crole == 1);
    const int obj = isA ? 0 : 1;
    const int SUB = (int)p.tc_sub, BW = SUB / 2 + 4;
    const uint32_t kSlotBytes = slot_bytes(p.tc_sub);
    const int nsub = (int)((p.L + SUB - 1) / SUB);
    Prof prof(cset == 0 ? p.prof : nullptr, isA ? 3 : 4);
    uint32_t pos = 0; // sub-tiles handled so far by this chain set (ring position; identical in all four chain-side warps)
    for (int g = ci; g < (int)p.NG; g += (int)p.W) {
      const uint32_t row = (uint32_t)(g * kGroup + lane), ch = p.ch0 + row;
      const bool active = row < p.C;

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

      for (int k = 0; k < nsub; ++k, ++pos) {
        const int slot = sbase + (int)(pos % NSLOT);
        const uint32_t phs = (pos / NSLOT) & 1u;
        prof.start();
        mbar_wait(isA ? &pc->ld_full[slot] : &pc->ab_full[slot], phs, 20);
        prof.lap(0);
        const int nq = (int)(min((uint32_t)SUB, p.L - (uint32_t)k * SUB) >> 3);
        uint4 *r0 = reinterpret_cast<uint4 *>(reinterpret_cast<uint32_t *>(bq_base + (uint32_t)slot * kSlotBytes) + (uint32_t)lane * BW);
        if (!(p.ablate & 2u)) {
          if (fast) {
            if (active) chain_span(st, r0, nq);
          } else { // generic cascade: stage-major over the sub-tile like the reference (filter_biquad.cpp:44-79); state in global
            const int nmax = __reduce_max_sync(0xffffffffu, active ? nst : 0);
            for (int j = 0; j < nmax; ++j) {
              if (active && j < nst) {
                BQ gs[1];
                uint32_t gf;
                bq_load_stage(gs[0], gf, p.bq, p.Cpad, obj, j, ch);
                chain_span(gs, r0, nq);
                bq_store_stage(gs[0], gf, p.bq, p.Cpad, obj, j, ch);
              }
            }
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(isA ? &pc->ab_full[slot] : &pc->st_full[slot]);
        prof.lap(1);
      }
      if (fast && active) bq_store_stage(st[0], fl, p.bq, p.Cpad, obj, 0, ch);
    }
    prof.flush();
  } else {
    // ================================================================== chain I/O: sub-tiles `out` -> smem ring -> `out`
    // Plain coalesced 16-byte accesses by two dedicated warps (32 per-row bulk copies per direction kept the SM's copy engine
    // busier than the biquad itself).  A warp instruction covers 32 >> lg rows of 1 << lg chunks; all addresses advance by
    // constants, so a sub-tile costs 32 << lg >> 5 loads and stores per lane and little else.
    const bool isLoad = (crole == 0);
    const int SUB = (int)p.tc_sub, BW = SUB / 2 + 4;
    const uint32_t kSlotBytes = slot_bytes(p.tc_sub);
    const int nsub = (int)((p.L + SUB - 1) / SUB); // L is a multiple of 128 and SUB is 64 or 128: sub-tiles are always full
    Prof prof(cset == 0 ? p.prof : nullptr, isLoad ? 5 : 6);
    const int lg = SUB == 128 ? 4 : 3;           // log2 of the 16-byte chunks per row
    const int rpi = 32 >> lg, nins = kGroup / rpi; // rows per warp instruction, instructions per sub-tile
    const int r0 = lane >> lg, c = lane & ((1 << lg) - 1);
    const size_t gstep = (size_t)rpi * p.stride * 2u;  // bytes between the rows of consecutive instructions
    const uint32_t sstep = (uint32_t)rpi * BW * 4u;
    uint32_t pos = 0;
    for (int g = ci; g < (int)p.NG; g += (int)p.W) {
      const int nrows = min(kGroup, (int)p.C - g * kGroup);
      unsigned char *gp0 = reinterpret_cast<unsigned char *>(p.out + ((size_t)g * kGroup + r0) * p.stride) + c * 16;
      int ready = 0; // leading units known to be in `out` for every row of the group
      // all rows of the group have the unit of sub-tile kk in `out`?  Blocking, or a single look.  Counters of later units that
      // are complete already are taken along, so that the acquire fence (an L1 invalidation, ~1.4 k cycles) is paid once for
      // all of them.
      auto unit_ready = [&](int kk, bool blocking) -> bool {
        const int need = (kk * SUB) / UNIT;
        if (ready > need) return true;
        int upto = ready; // first unit not known to be complete
        if (lane == 0) {
          const int *cnt = p.tile_cnt + (size_t)g * p.NU;
          const long long t0 = clock64();
          for (;;) {
            while (upto < (int)p.NU && upto <= need + 8 && ld_relaxed_gpu(cnt + upto) >= nrows) ++upto;
            if (upto > need || !blocking) break;
            __nanosleep(64);
            if (clock64() - t0 > kWatchdogCycles) __trap();
          }
          if (upto > ready) fence_acquire_gpu();
        }
        ready = __shfl_sync(0xffffffffu, upto, 0);
        return ready > need;
      };
      if (isLoad) {
        // global -> slot with cp.async (no registers), up to two sub-tiles ahead of the one handed to chain A, so the ~1.3 k-cycle
        // round trip to L2/HBM is off the chain's path
        constexpr int AHEAD = 2;
        auto issue = [&](int kk, uint32_t pp, bool blocking) -> bool {
          const int sl = sbase + (int)(pp % NSLOT);
          if (!unit_ready(kk, blocking)) return false;
          if (blocking) mbar_wait(&pc->slot_free[sl], ((pp / NSLOT) & 1u) ^ 1u);
          else if (!mbar_test_wait(&pc->slot_free[sl], ((pp / NSLOT) & 1u) ^ 1u)) return false;
          const unsigned char *gsrc = gp0 + (size_t)kk * SUB * 2u;
          const uint32_t sdst = smem_u32(bq_base + (uint32_t)sl * kSlotBytes) + (uint32_t)r0 * BW * 4u + c * 16;
          for (int j = 0; j < nins; ++j)
            if (r0 + j * rpi < nrows)
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sdst + (uint32_t)j * sstep), "l"(gsrc + (size_t)j * gstep) : "memory");
          asm volatile("cp.async.commit_group;" ::: "memory");
          return true;
        };
        int issued = 0; // sub-tiles requested so far
        for (int k = 0; k < nsub; ++k, ++pos) {
          const int slot = sbase + (int)(pos % NSLOT);
          prof.start();
          if (issued <= k) { issue(k, pos, true); issued = k + 1; }
          prof.lap(0);
          while (issued < nsub && issued <= k + AHEAD && issue(issued, pos + (uint32_t)(issued - k), false)) ++issued;
          prof.lap(1);
          // groups complete in order: wait until at most (issued - k - 1) newer ones are pending
          if (issued - k - 1 >= 2) asm volatile("cp.async.wait_group 2;" ::: "memory");
          else if (issued - k - 1 == 1) asm volatile("cp.async.wait_group 1;" ::: "memory");
          else asm volatile("cp.async.wait_group 0;" ::: "memory");
          __syncwarp(); // every lane's copies of this sub-tile have landed
          if (lane == 0) {
            mbar_arrive(&pc->ld_full[slot]);
            if ((((k + 1) * SUB) % SPAN) == 0 || k + 1 == nsub) atomicAdd(p.ctrl + 1, 1); // one more span taken (flow control)
          }
          prof.lap(2);
        }
      } else {
        for (int k = 0; k < nsub; ++k, ++pos) {
          const int slot = sbase + (int)(pos % NSLOT);
          const uint32_t phs = (pos / NSLOT) & 1u;
          unsigned char *sp0 = bq_base + (uint32_t)slot * kSlotBytes + (uint32_t)r0 * BW * 4u + c * 16;
          unsigned char *gp = gp0 + (size_t)k * SUB * 2u;
          prof.start();
          mbar_wait(&pc->st_full[slot], phs);
          prof.lap(0);
          for (int i0 = 0; i0 < nins; i0 += 8) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (r0 + (i0 + j) * rpi < nrows)
                *reinterpret_cast<uint4 *>(gp + (size_t)(i0 + j) * gstep) = *reinterpret_cast<const uint4 *>(sp0 + (uint32_t)(i0 + j) * sstep);
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&pc->slot_free[slot]);
          prof.lap(1);
        }
      }
      if (isLoad) {
        // carry the last H raw samples: hist <- tail of (hist || in[0..L)).  Every span of this group has been counted and
        // only a span's first window reaches back into the history, so nobody reads the old history any more.
        const uint32_t hq = p.H >> 3; // uint4 per history row (<= 33)
        for (int r = 0; r < nrows; ++r) {
          const size_t c = (size_t)g * kGroup + (size_t)r;
          uint4 *hrow = reinterpret_cast<uint4 *>(p.hist + ((size_t)p.ch0 + c) * p.H);
          const uint4 *irow = reinterpret_cast<const uint4 *>(p.in + c * p.stride);
          uint4 v0 = make_uint4(0, 0, 0, 0), v1 = v0;
          const uint32_t i0 = (uint32_t)lane, i1 = (uint32_t)lane + 32u;
          if (p.L >= p.H) {
            const uint4 *src = irow + ((p.L - p.H) >> 3);
            if (i0 < hq) v0 = src[i0];
            if (i1 < hq) v1 = src[i1];
          } else {
            const uint32_t lq = p.L >> 3, keep = hq - lq; // keep = old entries that survive
            if (i0 < hq) v0 = (i0 < keep) ? __ldcg(hrow + i0 + lq) : irow[i0 - keep];
            if (i1 < hq) v1 = (i1 < keep) ? __ldcg(hrow + i1 + lq) : irow[i1 - keep];
          }
          __syncwarp();
          if (i0 < hq) hrow[i0] = v0;
          if (i1 < hq) hrow[i1] = v1;
        }
      }
    }
    prof.flush();
  }
}

} // namespace v4

uint32_t chain_v4_span_samples() { return v4::SPAN; }
uint32_t chain_v4_unit_samples() { return v4::UNIT; }

// Shapes of the fused kernel for window K, each with the deepest operand ring (at least one pair ahead of the window) that fits:
//   shape 0  classic chain side + post warps (two staging buffers)     -- the default where shape 2 does not fit
//   shape 1  classic chain side, epilogue warps demodulate themselves  -- long windows (256 taps)
//   shape 2  FF chain side (feed-forward helper warps)                 -- the default up to one channel group per SM
//   shape 3  two chain sets per SM, no post warps                      -- more channel groups than SMs
// rings[s] = 0: shape s does not fit.  false = the tensor-core form does not apply at all.
bool chain_v4_config(uint32_t K, int smem_max, uint32_t rings[4])
{
  rings[0] = rings[1] = rings[2] = rings[3] = 0;
  if (K % 32u || K / 32u < 2u) return false;
  const uint32_t min_ring = K / 32u + 1u;
  for (int shape = 0; shape < 4; ++shape)
    for (uint32_t ring = tc::RING_MAX; ring >= min_ring; --ring)
      if (v4::smem_bytes(K, ring, shape == 2, shape == 0, shape == 3) <= (size_t)smem_max) { rings[shape] = ring; break; }
  return rings[0] || rings[1];
}

cudaError_t launch_chain_v4(const ChainParams &p_in, cudaStream_t stream, int variant, ChainLaunchInfo *info)
{
  using namespace v4;
  ChainParams p = p_in;
  p.ablate = ((uint32_t)variant >> 4) & 3u;
  p.tc_sub = sub_for(p.tc_K);
  const int shape = (int)p.tc_ff; // 0..3 as above
  const size_t smem = smem_bytes(p.tc_K, p.tc_ring, shape == 2, shape == 0, shape == 3);
  auto kern = shape == 2 ? chain_kernel<true, false, false> : shape == 0 ? chain_kernel<false, true, false>
            : shape == 3 ? chain_kernel<false, false, true> : chain_kernel<false, false, false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  uint32_t grid = shape == 3 ? p.W / 2 : p.W; // p.W = chains per wave; the DUAL shape runs two per CTA
  if (shape != 3 && p.spare_sms) { // leave SMs to a kernel on another stream; CTA b pins groups b, b + W, ...: every group below W needs its CTA
    const uint32_t need = p.NG < p.W ? p.NG : p.W;
    const uint32_t want = p.W > p.spare_sms ? p.W - p.spare_sms : 1u;
    grid = want > need ? want : need;
  }
  if (info) { info->grid = (int)grid; info->block = kThreads; info->smem = smem; info->tile = SPAN; }
  kern<<<grid, kThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

} // namespace msdr
