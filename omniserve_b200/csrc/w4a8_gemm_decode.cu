// W4A8 GEMM, decode-specialised (M <= 64) variant for sm_100a.  Same math, data path and operand formats as
// w4a8_gemm.cu (packed INT4 -> INT8 in registers -> tensor-memory A operand -> tcgen05.mma kind::i8, INT32 accumulators
// in TMEM, QServe dequant in the epilogue); what differs is everything that decides the LATENCY of a weight-streaming
// launch (round-2 measurements, profiles/r2_stream_probe.log):
//   * the bare load pipeline reaches the HBM roofline (6.6 TB/s) with four 8 KB stages per SM, yet the round-1 kernel
//     took 0.26 us per K-block per CTA no matter how few CTAs ran: its four unpack warps each touch EVERY K-block
//     (mbarrier wait -> ld.shared -> tcgen05.st -> wait::st -> arrive, ~500 cycles of dependent latency).  Here two
//     sets of four unpack warps alternate K-blocks, so two K-blocks are in that chain at any time;
//   * the CTA is small -- <= 99 KB shared memory, 256 tensor-memory columns, <= 80 registers x 384 threads -- so two
//     CTAs fit on an SM: two CTAs of this GEMM (independent pipelines) or this GEMM's CTA next to the CTA of the next
//     kernel of the decode chain, which programmatic dependent launch lets in early to prefetch ITS weights;
//   * split tiles: the K-slices of a tile are the CTAs of one cluster; each parks its INT32 partial in its own shared
//     memory, one barrier.cluster, every CTA sums ITS token columns from all peers over distributed shared memory and
//     stores fp16 -- exact, no L2 atomics, no "last CTA" (round 2: the L2 path below cost 4-6 us of dependent round trips per
//     GEMM).  Splits that are not an aligned 2/4/8-way split fall back to red.global.add.s32 straight from the TMEM
//     registers + arrival counter + finalisation by the last contributor.  Full tiles are stored as fp16 directly; the unpack
//     warps run the epilogue themselves (a decode CTA has 1-3 segments).
//
// Replaces the same reference kernels as w4a8_gemm.cu (per_chn/gemm_cuda.cu:308-657, per_group/gemm_cuda.cu:333-707).
#include "launch.h"
#include "moe_ops.h"
#include "ptx.cuh"
#include "w4a8_gemm.h"

#include <algorithm>
#include <mutex>
#include <stdlib.h>

namespace ob {
namespace dec {

constexpr int BM = 128;                  // weight rows per tile (UMMA M, TMEM lanes)
constexpr int BK = 128;                  // K bytes per K-block
constexpr int W_KB = BM * BK / 2;        // 8 KB packed per K-block
constexpr int S2_KB = 256;               // per-group: 128 B scales + 128 B zeros per K-block
constexpr int NUM_THREADS = 384;
constexpr int A_COLS = BK / 4;           // 32 TMEM columns per unpacked K-block
constexpr int TMEM_COLS = 256;
constexpr int ACC_COLS = 64;
// A pipeline STEP is KPS consecutive K-blocks of one segment: every ring (packed weights, activations, TMEM A slots)
// advances by steps, so the per-step handshakes (mbarrier waits / arrives, fences, commit) are paid once per KPS K-blocks.
#ifndef OB_DEC_KPS
#define OB_DEC_KPS 2
#endif
constexpr int KPS = OB_DEC_KPS;
#ifndef OB_DEC_CLUSTER_DEFAULT
#define OB_DEC_CLUSTER_DEFAULT true    // split-K inside a cluster over DSMEM (profiles/r2_cluster_splitk.log: 49.3 -> 43.7 us / layer)
#endif
constexpr int AB_STAGES = (TMEM_COLS - ACC_COLS) / (A_COLS * KPS);   // 3 steps: TMEM A ring == activation ring depth

template <int BN>
struct Cfg {
  static constexpr int W_STAGES = BN <= 32 ? 5 : 3;                  // steps of packed weights in flight
  static constexpr int W_STAGE = KPS * W_KB;
  static constexpr int B_STAGE = KPS * BN * BK;
  static constexpr int S2_STAGE = KPS * S2_KB;
  static constexpr int SMEM_B = 0;
  static constexpr int SMEM_W = SMEM_B + AB_STAGES * B_STAGE;
  static constexpr int SMEM_S2 = SMEM_W + W_STAGES * W_STAGE;
  static constexpr int SMEM_TOK = SMEM_S2 + W_STAGES * S2_STAGE;   // float sa[BN], ss[BN]
  static constexpr int SMEM_BAR = SMEM_TOK + BN * 8;
  static constexpr int NUM_BARS = 2 * W_STAGES + 3 * AB_STAGES + 2;
  static constexpr int SMEM_MISC = SMEM_BAR + NUM_BARS * 8;
  static constexpr int SMEM_TOTAL = SMEM_MISC + 64 + 1024;        // + alignment slack
  static_assert(SMEM_TOTAL <= 112 * 1024, "two CTAs per SM");
};

struct Params {
  const int8_t* s2_scales; const int8_t* s2_zeros;
  const __half* wscales; const __half* ascales; const __half* w_szs; const __half* a_ssums;
  __half* out;
  int32_t* ws;        // [grid][BN * 128] int32 partial tiles, zero between launches
  int32_t* counters;  // [grid]
  int M, N, K, ldc;
  int n_tiles, kb_per_tile, units_per_cta;
  int n_tiles_e;      // grouped mode: n-tiles per expert (n_tiles = groups * n_tiles_e)
  int cluster_s;      // > 1: the cluster_s CTAs of a cluster are the K-slices of ONE tile; split-K reduced over DSMEM
  long long* dbg_t;   // -DOB_DEC_TIMING builds only (tools/dec_waits.py): [grid][32] globaltimer stamps
};

// Grouped (mixture-of-experts) mode: the virtual tile index runs over (group, n-tile); a group is up to BN consecutive
// token rows routed to one expert (w4a8_moe_linear.py:83-94: x sorted by expert, `problem_sizes` rows per expert).
constexpr int MOE_MAX_GROUPS = 64;
struct MoeTab { int expert[MOE_MAX_GROUPS]; int row0[MOE_MAX_GROUPS]; int rows[MOE_MAX_GROUPS]; };
// Device-offset grouped mode: slot g is expert g; its rows come from the device table `offsets` [E+1] (moe_slot_rows), read
// only after griddepcontrol.wait, so the routing of the same decode step can produce it.
struct MoeDev { const int* offsets; int total_rows; };
struct NoMoe {};
template <bool MOE, bool DEV> struct MoeSel { using type = NoMoe; };
template <> struct MoeSel<true, false> { using type = MoeTab; };
template <> struct MoeSel<true, true> { using type = MoeDev; };
OB_DEVICE int moe_expert(const MoeTab& t, int g) { return t.expert[g]; }
OB_DEVICE int moe_expert(const MoeDev&, int g) { return g; }
OB_DEVICE void moe_slot(const MoeTab& t, int g, int& row0, int& rows) { row0 = t.row0[g]; rows = t.rows[g]; }
OB_DEVICE void moe_slot(const MoeDev& d, int g, int& row0, int& rows) {
  moe_slot_rows(d.offsets[g], d.offsets[g + 1], d.total_rows, &row0, &rows);
}

struct Seg { int tile, kb0, kb1; };

// This CTA's contiguous range of (tile, K-block) units, cut into per-tile segments.
struct SegIter {
  int KB, pos, end;
  OB_DEVICE void init(const Params& p) {
    KB = p.kb_per_tile;
    const long long tot = (long long)p.n_tiles * KB;
    const long long b = (long long)blockIdx.x * p.units_per_cta, e = b + p.units_per_cta;
    pos = (int)(b < tot ? b : tot);
    end = (int)(e < tot ? e : tot);
  }
  OB_DEVICE bool next(Seg& s) {
    if (pos >= end) return false;
    s.tile = pos / KB;
    s.kb0 = pos - s.tile * KB;
    const int room = KB - s.kb0, left = end - pos;
    s.kb1 = s.kb0 + (left < room ? left : room);
    pos += s.kb1 - s.kb0;
    return true;
  }
};

OB_DEVICE uint32_t vadd4(uint32_t a, uint32_t b) {   // bytewise (a + b) mod 256, `__vadd4` of per_group/gemm_cuda.cu:307
  const uint32_t s = (a & 0x7f7f7f7fu) + (b & 0x7f7f7f7fu);
  return s ^ ((a ^ b) & 0x80808080u);
}

#ifdef OB_DEC_TIMING
OB_DEVICE long long gtime() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define OB_GT(slot) do { if (p.dbg_t && lane == 0) p.dbg_t[blockIdx.x * 32 + (slot)] = gtime(); } while (0)
#else
#define OB_GT(slot) (void)0
#endif

OB_DEVICE void red_add_s32(int32_t* addr, int32_t v) {
  asm volatile("red.global.add.s32 [%0], %1;" ::"l"(addr), "r"(v) : "memory");
}
OB_DEVICE void bar_epi() { asm volatile("bar.sync 1, 256;" ::: "memory"); }   // the eight unpack / epilogue warps

// Cluster split-K: the S CTAs of a cluster hold the INT32 partial tiles of the same output tile in their own shared memory
// (layout [token column][128 rows]).  CTA `rank` owns BN / S token columns: thread (row = et & 127, h = et >> 7) reads the
// partials of its columns from all S CTAs over distributed shared memory -- BN / 2 independent 4-byte loads, issued back to
// back, 128 B per warp -- and returns the exact INT32 sums of columns rank * BN / S + h + 2 i in sum[i].
template <int BN, int S>
OB_DEVICE void cluster_reduce_cols(uint32_t stage_u32, uint32_t rank, int row, int h, int (&sum)[BN / 2]) {
  constexpr int COLS = BN / S;          // columns owned by a CTA
  constexpr int NI = COLS / 2;          // columns per thread
  static_assert(COLS >= 2 && (COLS % 2) == 0, "two column phases per CTA");
  int v[NI][S];
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const uint32_t local = stage_u32 + (uint32_t)(((rank * COLS + h + 2 * i) * BM + row) * 4);
#pragma unroll
    for (int pr = 0; pr < S; ++pr) v[i][pr] = ld_shared_cluster_s32(mapa_shared(local, (uint32_t)pr));
  }
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    int a = 0;
#pragma unroll
    for (int pr = 0; pr < S; ++pr) a += v[i][pr];
    sum[i] = a;
  }
}

template <int BN, bool PER_GROUP, bool MOE = false, bool DEV = false>
__global__ void __launch_bounds__(NUM_THREADS, 2)
w4a8_gemm_decode_kernel(const __grid_constant__ CUtensorMap act_map, const __grid_constant__ CUtensorMap w_map, const Params p,
                        const __grid_constant__ typename MoeSel<MOE, DEV>::type moe) {
  using C = Cfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sB = smem + C::SMEM_B;
  uint8_t* sW = smem + C::SMEM_W;
  uint8_t* sS2 = smem + C::SMEM_S2;
  float* sTok = reinterpret_cast<float*>(smem + C::SMEM_TOK);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::SMEM_BAR);
  uint64_t* w_full = bars;                         // packed weights (+ s2) of the step landed              (1 arrival + tx)
  uint64_t* w_empty = w_full + C::W_STAGES;        // the eight unpack warps read their K-blocks of the step (8)
  uint64_t* b_full = w_empty + C::W_STAGES;        // activation tiles of the step landed                 (1 + tx)
  uint64_t* a_full = b_full + AB_STAGES;           // the eight unpack warps filled the TMEM A slot        (8)
  uint64_t* ba_empty = a_full + AB_STAGES;         // MMAs that read activation stage s / A slot s retired (1, commit)
  uint64_t* acc_full = ba_empty + AB_STAGES;       // last MMA of the segment retired                      (1, commit)
  uint64_t* acc_empty = acc_full + 1;              // the eight epilogue warps drained the accumulator     (8)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + C::SMEM_MISC);
  int* sFlag = reinterpret_cast<int*>(smem + C::SMEM_MISC + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_trigger();
#ifdef OB_DEC_WAIT_FIRST
  pdl_wait();
#endif
  if (warp == 3) OB_GT(24);   // kernel entry

  if (warp == 0) {
    if (lane == 0) { tma_prefetch_desc(&act_map); tma_prefetch_desc(&w_map); }
    for (int i = lane; i < C::NUM_BARS; i += 32) {
      uint64_t* b = bars + i;
      const uint32_t cnt = ((b >= w_empty && b < b_full) || (b >= a_full && b < ba_empty) || b == acc_empty) ? 8u : 1u;
      mbar_init(b, cnt);
    }
    mbar_fence_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (warp == 3) OB_GT(25);   // prologue done (barriers, TMEM)

  if (warp == 0) {
    // ================================================================ weight producer: never waits for the previous
    // kernel (weights are constants), so under PDL it fills the ring while the predecessor is still draining
    if (lane == 0) {
      SegIter it; it.init(p);
      Seg sg;
      int stage = 0, phase = 0;
      while (it.next(sg)) {
        const int n_cnt = min(BM, p.N - sg.tile * BM);
        int w_tile = sg.tile;     // row-of-tiles coordinate in the packed weight tensor
        if constexpr (MOE) {
          const int g = sg.tile / p.n_tiles_e;
          w_tile = moe_expert(moe, g) * p.n_tiles_e + (sg.tile - g * p.n_tiles_e);   // experts are stacked along N
        }
        for (int kb = sg.kb0; kb < sg.kb1; kb += KPS) {
          const int cnt = min(KPS, sg.kb1 - kb);
          mbar_wait(&w_empty[stage], phase ^ 1);
          mbar_arrive_expect_tx(&w_full[stage], cnt * (W_KB + (PER_GROUP ? 2 * n_cnt : 0)));
          for (int j = 0; j < cnt; ++j) {
            tma_load_3d(sW + stage * C::W_STAGE + j * W_KB, &w_map, 0, (kb + j) * 4, w_tile * 4, &w_full[stage]);
            if (PER_GROUP) {
              uint8_t* d = sS2 + stage * C::S2_STAGE + j * S2_KB;
              bulk_g2s(d, p.s2_scales + (size_t)(kb + j) * p.N + sg.tile * BM, n_cnt, &w_full[stage]);
              bulk_g2s(d + 128, p.s2_zeros + (size_t)(kb + j) * p.N + sg.tile * BM, n_cnt, &w_full[stage]);
            }
          }
          if (++stage == C::W_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================================================================ activation producer (previous kernel's output)
    if (lane == 0) {
      pdl_wait();
      SegIter it; it.init(p);
      Seg sg;
      int stage = 0, phase = 0;
      while (it.next(sg)) {
        int row0 = 0;
        if constexpr (MOE) {
          int rows = 0;
          moe_slot(moe, sg.tile / p.n_tiles_e, row0, rows);
          if (rows == 0) row0 = 0;   // empty slot: the MMAs still drain the weight ring, nothing is stored
        }
        for (int kb = sg.kb0; kb < sg.kb1; kb += KPS) {
          const int cnt = min(KPS, sg.kb1 - kb);
          mbar_wait(&ba_empty[stage], phase ^ 1);
          mbar_arrive_expect_tx(&b_full[stage], cnt * BN * BK);
          for (int j = 0; j < cnt; ++j)
            tma_load_2d(sB + stage * C::B_STAGE + j * BN * BK, &act_map, (kb + j) * BK, row0, &b_full[stage]);
          if (++stage == AB_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 2) {
    // ================================================================ MMA issuer: one wait pair + one commit per step
    SegIter it; it.init(p);
    Seg sg;
    int st = 0, ph = 0, acc_phase = 0;
    constexpr uint32_t idesc = umma_idesc_i8(BM, BN, true, true);
    const uint64_t bdesc0 = umma_desc_kmajor_sw128(smem_u32(sB));
    const uint32_t a_tmem0 = tmem_base + ACC_COLS;
    while (it.next(sg)) {
      mbar_wait(acc_empty, acc_phase ^ 1);
      tc_fence_after();
      for (int kb = sg.kb0; kb < sg.kb1; kb += KPS) {
        const int cnt = min(KPS, sg.kb1 - kb);
        mbar_wait(&b_full[st], ph);
        mbar_wait(&a_full[st], ph);
        tc_fence_after();
        if (elect_one()) {
          uint64_t bdesc = bdesc0 + (uint64_t)((st * C::B_STAGE) >> 4);
          uint32_t a_tmem = a_tmem0 + st * (A_COLS * KPS);
          umma_i8_ts(tmem_base, a_tmem, bdesc, idesc, kb > sg.kb0 ? 1u : 0u);
          umma_i8_ts(tmem_base, a_tmem + 8, bdesc + 2, idesc, 1u);
          umma_i8_ts(tmem_base, a_tmem + 16, bdesc + 4, idesc, 1u);
          umma_i8_ts(tmem_base, a_tmem + 24, bdesc + 6, idesc, 1u);
          if (cnt > 1) {
            bdesc += (uint64_t)((BN * BK) >> 4);
            a_tmem += A_COLS;
            umma_i8_ts(tmem_base, a_tmem, bdesc, idesc, 1u);
            umma_i8_ts(tmem_base, a_tmem + 8, bdesc + 2, idesc, 1u);
            umma_i8_ts(tmem_base, a_tmem + 16, bdesc + 4, idesc, 1u);
            umma_i8_ts(tmem_base, a_tmem + 24, bdesc + 6, idesc, 1u);
          }
          umma_commit(&ba_empty[st]);
          if (kb + cnt >= sg.kb1) umma_commit(acc_full);
        }
        __syncwarp();
        if (++st == AB_STAGES) { st = 0; ph ^= 1; }
      }
      acc_phase ^= 1;
    }
  } else if (warp >= 4) {
    // ================================================================ unpack (set j converts K-block j of every step) + epilogue
    // Both sets take part in EVERY step (set 0: first K-block, set 1: second), so every ring is consumed strictly in
    // order by the same waiters -- a parity wait is never more than one phase ahead -- and the two K-blocks of a step are
    // converted concurrently.  A one-K-block step (odd tail of a segment) leaves set 1 with only the handshakes.
    const int set = (warp - 4) >> 2;
    const int q = warp & 3;                // TMEM lane quarter == n32 block inside the tile
    const int et = threadIdx.x - 128;      // 0..255
    SegIter it; it.init(p);
    Seg sg;
    const uint32_t sW_u32 = smem_u32(sW), sS2_u32 = smem_u32(sS2);
    const uint32_t t_q = tmem_base + ((uint32_t)(q * 32) << 16);
    int ws = 0, wph = 0, as = 0, aph = 0;
    int acc_phase = 0;
    bool waited = false;
    static_assert(KPS == 2, "one unpack set per K-block of a step");

    while (it.next(sg)) {
      for (int kb = sg.kb0; kb < sg.kb1; kb += KPS) {
        const bool mine = kb + set < sg.kb1;
        mbar_wait(&w_full[ws], wph);
        uint4 v[4];
        uint32_t ps = 0, pz = 0;
        if (mine) {
          const uint32_t wsm = sW_u32 + ws * C::W_STAGE + set * W_KB + q * 2048 + lane * 16;
#pragma unroll
          for (int a = 0; a < 4; ++a) v[a] = lds_v4(wsm + a * 512);
          if (PER_GROUP) {
            ps = lds_u32(sS2_u32 + ws * C::S2_STAGE + set * S2_KB + q * 32 + (lane >> 2) * 4);
            pz = lds_u32(sS2_u32 + ws * C::S2_STAGE + set * S2_KB + 128 + q * 32 + (lane >> 2) * 4);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&w_empty[ws]);     // this warp's part of the packed step is in registers
        if (++ws == C::W_STAGES) { ws = 0; wph ^= 1; }
        mbar_wait(&ba_empty[as], aph ^ 1);            // MMAs that read the slot's previous contents retired
        tc_fence_after();
        if (mine) {
          uint32_t sc[4], zr[4];
          if (PER_GROUP) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              sc[i] = (ps >> (8 * i)) & 0xFFu;
              zr[i] = ((pz >> (8 * i)) & 0xFFu) * 0x01010101u;
            }
          }
          const uint32_t t_lo = t_q + ACC_COLS + (as * KPS + set) * A_COLS;
          const uint32_t t_hi = t_lo + (16u << 16);
#pragma unroll
          for (int a = 0; a < 4; ++a) {
            const uint4 w = v[a];
            uint32_t l0 = w.x & 0x0F0F0F0Fu, l1 = w.y & 0x0F0F0F0Fu, l2 = w.z & 0x0F0F0F0Fu, l3 = w.w & 0x0F0F0F0Fu;
            uint32_t h0 = (w.x >> 4) & 0x0F0F0F0Fu, h1 = (w.y >> 4) & 0x0F0F0F0Fu, h2 = (w.z >> 4) & 0x0F0F0F0Fu,
                     h3 = (w.w >> 4) & 0x0F0F0F0Fu;
            if (PER_GROUP) {
              // rows: l0,l2 -> c (scale 0); l1,l3 -> c+8 (scale 1); h0,h2 -> c+16 (scale 2); h1,h3 -> c+24 (scale 3)
              l0 = vadd4(l0 * sc[0], zr[0]); l2 = vadd4(l2 * sc[0], zr[0]);
              l1 = vadd4(l1 * sc[1], zr[1]); l3 = vadd4(l3 * sc[1], zr[1]);
              h0 = vadd4(h0 * sc[2], zr[2]); h2 = vadd4(h2 * sc[2], zr[2]);
              h1 = vadd4(h1 * sc[3], zr[3]); h3 = vadd4(h3 * sc[3], zr[3]);
            }
            tmem_st_16x128b_x2(t_lo + a * 8, l0, l1, l2, l3);
            tmem_st_16x128b_x2(t_hi + a * 8, h0, h1, h2, h3);
          }
          tmem_st_wait();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_full[as]);
        if (++as == AB_STAGES) { as = 0; aph ^= 1; }
      }

      // ---------------------------------------------------------------- epilogue of the segment (all eight warps)
      if (!waited) {   // ascales / a_ssums, `out` and the workspace belong to the chain
        if (warp == 4) OB_GT(26);   // first segment unpacked
        pdl_wait();
        waited = true;
        if (warp == 4) OB_GT(27);   // grid dependency resolved
      }
      int nt = sg.tile, m_rows = p.M, row0 = 0, s_off = 0;   // grouped mode: this tile's token rows and expert
      if constexpr (MOE) {
        const int g = sg.tile / p.n_tiles_e;
        nt = sg.tile - g * p.n_tiles_e;
        moe_slot(moe, g, row0, m_rows);
        s_off = moe_expert(moe, g) * p.N;
      }
      const int n_row = nt * BM + q * 32 + lane;
      const bool n_ok = n_row < p.N;
      const bool full_tile = (sg.kb0 == 0 && sg.kb1 == p.kb_per_tile);
      float wsc = 0.f, wsz = 0.f;
      if (n_ok) {
        wsc = __half2float(p.wscales[s_off + n_row]);
        if (!PER_GROUP) wsz = __half2float(p.w_szs[s_off + n_row]);
      }
      if (et < BN) {
        sTok[et] = (et < m_rows) ? __half2float(p.ascales[row0 + et]) : 0.f;
        sTok[BN + et] = (!PER_GROUP && et < m_rows) ? __half2float(p.a_ssums[row0 + et]) : 0.f;
      }
      mbar_wait(acc_full, acc_phase);
      if (warp == 4) OB_GT(28);     // accumulator of the (last) segment complete
      acc_phase ^= 1;
      tc_fence_after();
      bar_epi();   // sTok visible
      constexpr int HALF = BN / 2;                       // tokens per set
      constexpr int CH = HALF >= 16 ? 16 : 8;            // columns per tcgen05.ld
      const int c_base = set * HALF;
      const int first_cta = (int)(((long long)sg.tile * p.kb_per_tile) / p.units_per_cta);
      int32_t* slot = p.ws + (size_t)first_cta * (BN * BM);
#pragma unroll 1
      for (int c0 = c_base; c0 < c_base + HALF; c0 += CH) {
        uint32_t r[16];
        if (CH == 16) {
          tmem_ld_32x32b_x16(t_q + c0, r);
        } else {
          uint32_t r8[8];
          tmem_ld_32x32b_x8(t_q + c0, r8);
#pragma unroll
          for (int j = 0; j < 8; ++j) r[j] = r8[j];
        }
        tmem_ld_wait();
        if (full_tile) {
#pragma unroll
          for (int j = 0; j < CH; ++j) {
            const int m = c0 + j;
            const float ps = __int2float_rn((int)r[j]);
            float o;
            if (PER_GROUP) o = ps * (wsc * sTok[m]);
            else o = __fmaf_rn(-wsz, sTok[BN + m], (ps * wsc) * sTok[m]);
            if (n_ok && m < m_rows) p.out[(size_t)(row0 + m) * p.ldc + n_row] = __float2half_rn(o);
          }
        } else if (!MOE && p.cluster_s > 1) {
          // cluster split-K: park the partial in this CTA's (fully consumed) packed-weight ring, [column][row]
#pragma unroll
          for (int j = 0; j < CH; ++j) reinterpret_cast<int32_t*>(sW)[(c0 + j) * BM + q * 32 + lane] = (int)r[j];
        } else {
#pragma unroll
          for (int j = 0; j < CH; ++j) red_add_s32(slot + (c0 + j) * BM + q * 32 + lane, (int)r[j]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);    // MMAs of the next segment may overwrite the accumulator
      if (!MOE && !full_tile && p.cluster_s > 1) {
        // ---- exact INT32 split-K inside the cluster, over distributed shared memory: no L2 atomics, no arrival counter,
        // no read-back by a "last" CTA -- every CTA finalises its own token columns (profiles/r2_dec_timeline.log: the
        // L2 path costs 4-6 us of dependent round trips per split GEMM).
        cluster_barrier();                       // all partials of the tile are in place (release / acquire, cluster scope)
        const uint32_t rank = cluster_ctarank();
        const int row = et & 127, h = et >> 7;
        int sum[BN / 2];
        int ncol = 0;
        const uint32_t stage_u32 = smem_u32(sW);
        switch (p.cluster_s) {
          case 8: cluster_reduce_cols<BN, 8>(stage_u32, rank, row, h, sum); ncol = BN / 16; break;
          case 4: cluster_reduce_cols<BN, 4>(stage_u32, rank, row, h, sum); ncol = BN / 8; break;
          default: cluster_reduce_cols<BN, 2>(stage_u32, rank, row, h, sum); ncol = BN / 4; break;
        }
        const int col0 = (int)rank * (BN / p.cluster_s) + h;
#pragma unroll
        for (int i = 0; i < BN / 4; ++i) {
          if (i < ncol) {
            const int m = col0 + 2 * i;
            const float ps = __int2float_rn(sum[i]);
            float o;
            if (PER_GROUP) o = ps * (wsc * sTok[m]);
            else o = __fmaf_rn(-wsz, sTok[BN + m], (ps * wsc) * sTok[m]);
            if (n_ok && m < m_rows) p.out[(size_t)(row0 + m) * p.ldc + n_row] = __float2half_rn(o);
          }
        }
        cluster_barrier_relaxed();               // nobody leaves while a peer may still read its shared memory (the remote
                                                 // loads of this thread have returned: their sums were just stored)
      } else if (!full_tile) {
        // exact INT32 split-K: every contributor's reds must be performed before its arrival is counted
        const int last_cta = (int)(((long long)(sg.tile + 1) * p.kb_per_tile - 1) / p.units_per_cta);
        const int contributors = last_cta - first_cta + 1;
        __threadfence();
        bar_epi();
        if (et == 0) {
          const int old = atomicAdd(&p.counters[first_cta], 1);
          *sFlag = (old == contributors - 1) ? 1 : 0;
        }
        bar_epi();
        if (*sFlag) {
          __threadfence();
          // finalize: thread (q, lane, set) owns row n_row and the tokens of its set; L2 reads are batched
          constexpr int BATCH = HALF < 16 ? HALF : 16;
#pragma unroll 1
          for (int c0 = c_base; c0 < c_base + HALF; c0 += BATCH) {
            int a[BATCH];
#pragma unroll
            for (int j = 0; j < BATCH; ++j) a[j] = __ldcg(slot + (c0 + j) * BM + q * 32 + lane);
#pragma unroll
            for (int j = 0; j < BATCH; ++j) {
              const int m = c0 + j;
              __stcg(slot + m * BM + q * 32 + lane, 0);
              const float ps = __int2float_rn(a[j]);
              float o;
              if (PER_GROUP) o = ps * (wsc * sTok[m]);
              else o = __fmaf_rn(-wsz, sTok[BN + m], (ps * wsc) * sTok[m]);
              if (n_ok && m < m_rows) p.out[(size_t)(row0 + m) * p.ldc + n_row] = __float2half_rn(o);
            }
          }
          if (et == 0) p.counters[first_cta] = 0;
        }
      }
      bar_epi();   // sTok / sFlag free for the next segment
      if (warp == 4) OB_GT(29);     // epilogue (incl. finalisation) of the (last) segment done
    }
  }

  if (!MOE && p.cluster_s > 1 && warp < 4) {   // producers / MMA / idle warp: the epilogue's two cluster barriers
    __syncwarp();
    cluster_barrier();
    cluster_barrier_relaxed();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<TMEM_COLS>(tmem_base);
  if (warp == 3) OB_GT(30);   // exit
}

template <int BN, bool DEV = false>
static int launch_moe(const CUtensorMap& amap, const CUtensorMap& wmap, const Params& p, const typename MoeSel<true, DEV>::type& tab,
                      int grid, cudaStream_t st) {
  using C = Cfg<BN>;
  auto kern = w4a8_gemm_decode_kernel<BN, false, true, DEV>;
  static bool attr_done[16] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_done[dev]) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_TOTAL) != cudaSuccess) return OB_ERR_CUDA;
    attr_done[dev] = true;
  }
  return launch_pdl(kern, dim3(grid), dim3(NUM_THREADS), (size_t)C::SMEM_TOTAL, st, amap, wmap, p, tab) == cudaSuccess ? 0 : OB_ERR_CUDA;
}

template <int BN, bool PG>
static int launch(const CUtensorMap& amap, const CUtensorMap& wmap, const Params& p, int grid, cudaStream_t st) {
  using C = Cfg<BN>;
  auto kern = w4a8_gemm_decode_kernel<BN, PG, false, false>;
  static bool attr_done[16] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_done[dev]) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_TOTAL) != cudaSuccess) return OB_ERR_CUDA;
    attr_done[dev] = true;
  }
  const unsigned cluster = p.cluster_s > 1 ? (unsigned)p.cluster_s : 1u;
  return launch_pdl_cluster(kern, dim3(grid), dim3(NUM_THREADS), (size_t)C::SMEM_TOTAL, st, cluster, amap, wmap, p, NoMoe{}) == cudaSuccess
             ? 0 : OB_ERR_CUDA;
}

// Can clusters of `s` CTAs of this kernel be co-scheduled at all on this device (two ~100 KB CTAs per SM, GPC sizes)?
// Queried once per (device, BN, per_group, s); never during stream capture problems: the query launches nothing.
template <int BN, bool PG>
static bool cluster_ok(int dev, int s) {
  static int ok[16][9] = {};   // 0 = unknown, 1 = yes, -1 = no
  if (s < 2 || s > 8) return false;
  if (!ok[dev][s]) {
    using C = Cfg<BN>;
    auto kern = w4a8_gemm_decode_kernel<BN, PG, false, false>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_TOTAL);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(s * 8); cfg.blockDim = dim3(NUM_THREADS); cfg.dynamicSmemBytes = C::SMEM_TOTAL;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = s; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int n = 0;
    const cudaError_t e = cudaOccupancyMaxActiveClusters(&n, kern, &cfg);
    if (e != cudaSuccess) cudaGetLastError();
    ok[dev][s] = (e == cudaSuccess && n >= 1) ? 1 : -1;
  }
  return ok[dev][s] > 0;
}

}  // namespace dec

// Scheduling: every CTA gets `upc` consecutive (tile, K-block) units.  Cost model in us, fitted to the sweep of every
// choice on B200 (profiles/r2_upc_sweep.log; the ~3.5 us launch floor is common to all and left out):
//   * an SM moves one K-block per ~0.2 us however many CTAs share it: streaming = (CTAs per SM) x upc x 0.2;
//   * a tile that is not split ends with a ~0.3 us epilogue (direct fp16 stores);
//   * a split through L2 costs ~5 us (reds, fence, arrival counter, read-back and finalisation by the last contributor:
//     four dependent L2 round trips), plus ~0.01 us per contributing CTA of atomic traffic; an aligned 2 / 4 / 8-way split
//     whose K-slices form one cluster is reduced over distributed shared memory instead and costs ~1.5 us;
//   * ranges that straddle tile boundaries add a second epilogue and an uneven finish (~3 us).
static bool cluster_split(int KB, int upc) {   // an aligned 2 / 4 / 8-way split: the K-slices of a tile form one cluster
  if (upc >= KB || KB % upc) return false;
  const int s = KB / upc;
  return s == 2 || s == 4 || s == 8;
}

static int choose_upc(int n_tiles, int KB, int sms, int ctas_per_sm, int BN, bool use_cluster) {
  (void)BN;
  const long long units = (long long)n_tiles * KB;
  const int max_ctas = sms * ctas_per_sm;
  const int lo = (int)((units + max_ctas - 1) / max_ctas);
  if (lo >= KB) return KB * ((lo + KB - 1) / KB);   // at least a tile per CTA: whole tiles, no split
  const float T_KB = 0.2f, T_FULL = 0.3f, T_SPLIT = 5.0f, T_SPLIT_CL = 1.5f, T_CTA = 0.01f, T_UNALIGNED = 3.0f;
  int best = KB;
  float best_cost = 1e30f;
  for (int upc = lo; upc <= KB; ++upc) {
    const long long n_ctas = (units + upc - 1) / upc;
    const int per_sm = (int)((n_ctas + sms - 1) / sms);
    float cost = per_sm * upc * T_KB;
    if (upc >= KB) cost += T_FULL;
    else if (use_cluster && cluster_split(KB, upc)) cost += T_SPLIT_CL;      // reduced over DSMEM inside the cluster
    else cost += T_SPLIT + n_ctas * T_CTA;
    if (KB % upc) cost += T_UNALIGNED;
    if (cost < best_cost - 1e-6f) { best_cost = cost; best = upc; }
  }
  return best;
}

int w4a8_gemm_decode_run(const W4A8GemmArgs& a, bool per_group, cudaStream_t st) {
  using namespace dec;
  if (a.M <= 0) return 0;
  if (a.M > 64 || a.N % 32 != 0 || a.K % 128 != 0 || a.ldc < a.N || a.tail_hidden_in) return OB_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(a.in_feats) & 15) || (reinterpret_cast<uintptr_t>(a.qweight) & 15)) return OB_ERR_ALIGN;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 16) return OB_ERR_ARG;
  const int sms = dev_sms(dev);
  int32_t* ws = nullptr;
  int32_t* cnt = nullptr;
  if (int e = get_workspace(dev, st, &ws, &cnt)) return e;

  int BN = a.M <= 16 ? 16 : a.M <= 32 ? 32 : 64;
  if (a.force_bn == 16 || a.force_bn == 32 || a.force_bn == 64) BN = std::max(BN, a.force_bn);
  Params p{};
  p.s2_scales = a.s2_scales; p.s2_zeros = a.s2_zeros;
  p.wscales = a.wscales; p.ascales = a.ascales; p.w_szs = a.w_szs; p.a_ssums = a.a_ssums;
  p.out = a.out_feats; p.ws = ws; p.counters = cnt;
  p.M = a.M; p.N = a.N; p.K = a.K; p.ldc = a.ldc;
  p.n_tiles = (a.N + BM - 1) / BM;
  p.kb_per_tile = a.K / BK;
#ifdef OB_DEC_TIMING
  {   // every launch gets its own [1024][32] block of the debug buffer (64 blocks, round robin)
    static int launch_idx = 0;
    const char* e = getenv("OB_DEC_DBGT");
    p.dbg_t = e ? reinterpret_cast<long long*>(strtoull(e, nullptr, 10)) + (size_t)(launch_idx++ % 64) * 1024 * 32 : nullptr;
  }
#endif
  static const int ctas_per_sm = [] { const char* e = getenv("OB_GEMM_DEC_CTAS_PER_SM"); return e ? std::max(1, std::min(2, atoi(e))) : 2; }();
  int max_ctas = a.force_ctas > 0 ? std::min(a.force_ctas, 2 * sms) : ctas_per_sm * sms;
  const long long units = (long long)p.n_tiles * p.kb_per_tile;
  // split-K over distributed shared memory (cluster = the K-slices of one tile): OB_GEMM_DEC_CLUSTER=0 falls back to the L2 path
  static const bool use_cluster = [] { const char* e = getenv("OB_GEMM_DEC_CLUSTER"); return e ? atoi(e) != 0 : OB_DEC_CLUSTER_DEFAULT; }();
  p.units_per_cta = a.force_ctas > 0 ? (int)((units + max_ctas - 1) / max_ctas)
                                     : choose_upc(p.n_tiles, p.kb_per_tile, sms, ctas_per_sm, BN, use_cluster);
  const int grid = (int)((units + p.units_per_cta - 1) / p.units_per_cta);
  p.cluster_s = 0;
  if (use_cluster && cluster_split(p.kb_per_tile, p.units_per_cta)) {
    const int s = p.kb_per_tile / p.units_per_cta;
    bool ok = false;
    switch (BN) {
      case 16: ok = per_group ? cluster_ok<16, true>(dev, s) : cluster_ok<16, false>(dev, s); break;
      case 32: ok = per_group ? cluster_ok<32, true>(dev, s) : cluster_ok<32, false>(dev, s); break;
      default: ok = per_group ? cluster_ok<64, true>(dev, s) : cluster_ok<64, false>(dev, s); break;
    }
    if (ok && grid == p.n_tiles * s) p.cluster_s = s;
  }
  CUtensorMap amap, wmap;
  if (int e = make_act_map(&amap, a.in_feats, a.M, a.K, BN)) return e;
  if (int e = make_w_map(&wmap, a.qweight, a.N, a.K, false)) return e;
  switch (BN) {
    case 16: return per_group ? launch<16, true>(amap, wmap, p, grid, st) : launch<16, false>(amap, wmap, p, grid, st);
    case 32: return per_group ? launch<32, true>(amap, wmap, p, grid, st) : launch<32, false>(amap, wmap, p, grid, st);
    default: return per_group ? launch<64, true>(amap, wmap, p, grid, st) : launch<64, false>(amap, wmap, p, grid, st);
  }
}

// Host-only view of the scheduling decision above (no CUDA call; tests/test_host_logic.py): which token tile, how many
// K-blocks per CTA, how many CTAs and -- if the split is an aligned 2 / 4 / 8-way split -- the cluster size the launch
// would ask for (the run additionally checks that such clusters can be co-scheduled on the device).
int w4a8_gemm_decode_plan(int M, int N, int K, int sms, int ctas_per_sm, int use_cluster, int* bn, int* units_per_cta, int* grid,
                          int* cluster_s) {
  using namespace dec;
  if (M <= 0 || M > 64 || N % 32 != 0 || K % 128 != 0 || sms <= 0 || ctas_per_sm < 1 || ctas_per_sm > 2) return OB_ERR_SHAPE;
  const int BN = M <= 16 ? 16 : M <= 32 ? 32 : 64;
  const int n_tiles = (N + BM - 1) / BM, kb = K / BK;
  const long long units = (long long)n_tiles * kb;
  const int upc = choose_upc(n_tiles, kb, sms, ctas_per_sm, BN, use_cluster != 0);
  const int g = (int)((units + upc - 1) / upc);
  int cs = 0;
  if (use_cluster && cluster_split(kb, upc) && g == n_tiles * (kb / upc)) cs = kb / upc;
  if (bn) *bn = BN;
  if (units_per_cta) *units_per_cta = upc;
  if (grid) *grid = g;
  if (cluster_s) *cluster_s = cs;
  return 0;
}

// Grouped W4A8 per-channel GEMM for mixture-of-experts layers (SURVEY.md section 8 row f3; interface of the reference's
// unreleased op, w4a8_moe_linear.py:83-94: x [T, K] int8 with the token rows sorted by expert, qweight [E, N, K/2] in the
// reference tile layout per expert, s1_scales / s1_szeros [E, N], per-token input_scales / input_sum [T], problem_sizes[e] =
// rows routed to expert e; out [T, N] fp16).  One launch: every (expert chunk of <= 64 rows, 128-row weight tile) is a
// whole-K tile of the decode kernel -- no split, weights streamed once per chunk.
int w4a8_moe_gemm_run(const int8_t* x, const int8_t* qweight, const __half* wscales, const __half* ascales, const __half* w_szs,
                      const __half* a_ssums, __half* out, const int* problem_sizes_host, int num_experts, int T, int N, int K,
                      int ldc, cudaStream_t st) {
  using namespace dec;
  if (T <= 0 || num_experts <= 0) return 0;
  if (N % BM != 0 || K % BK != 0 || ldc < N) return OB_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(qweight) & 15)) return OB_ERR_ALIGN;
  long long tot = 0;
  for (int e = 0; e < num_experts; ++e) {
    if (problem_sizes_host[e] < 0) return OB_ERR_ARG;
    tot += problem_sizes_host[e];
  }
  if (tot != T) return OB_ERR_ARG;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 16) return OB_ERR_ARG;
  const int sms = dev_sms(dev);
  int32_t* ws = nullptr;
  int32_t* cnt = nullptr;
  if (int e = get_workspace(dev, st, &ws, &cnt)) return e;
  CUtensorMap amap, wmap;
  if (int e = make_act_map(&amap, x, T, K, 64)) return e;
  if (int e = make_w_map(&wmap, qweight, num_experts * N, K, false)) return e;   // experts stacked along N
  Params p{};
  p.wscales = wscales; p.ascales = ascales; p.w_szs = w_szs; p.a_ssums = a_ssums; p.out = out; p.ws = ws; p.counters = cnt;
  p.M = 64; p.N = N; p.K = K; p.ldc = ldc;
  p.n_tiles_e = N / BM;
  p.kb_per_tile = K / BK;
  // chunks of <= 64 rows per expert, launched MOE_MAX_GROUPS at a time
  MoeTab tab{};
  int g = 0, row = 0;
  auto flush = [&]() -> int {
    if (g == 0) return 0;
    p.n_tiles = g * p.n_tiles_e;
    const int tiles_per_cta = (p.n_tiles + 2 * sms - 1) / (2 * sms);
    p.units_per_cta = tiles_per_cta * p.kb_per_tile;     // whole tiles per CTA: no split-K
    const int grid = (p.n_tiles + tiles_per_cta - 1) / tiles_per_cta;
    const int e = launch_moe<64>(amap, wmap, p, tab, grid, st);
    g = 0;
    return e;
  };
  for (int e = 0; e < num_experts; ++e) {
    for (int done = 0; done < problem_sizes_host[e]; done += 64) {
      tab.expert[g] = e; tab.row0[g] = row + done; tab.rows[g] = std::min(64, problem_sizes_host[e] - done);
      if (++g == MOE_MAX_GROUPS) { if (int err = flush()) return err; }
    }
    row += problem_sizes_host[e];
  }
  return flush();
}

// Grouped GEMM with DEVICE-resident row ranges (the decode step of a mixture-of-experts layer, which a CUDA graph replays
// with a routing it cannot know on the host).  A token routes to k DISTINCT experts, so with <= 64 tokens no expert gets
// more than one 64-row tile: slot g is statically expert g, the grid and the tiles per CTA depend only on (E, N, K) and the
// device, and the weight producer streams expert g's tiles before griddepcontrol.wait exactly like the dense decode GEMM.
// Only row0 / rows of a slot come from `offsets` [E+1] (the routing's expert_offsets), read after the wait by the
// activation producer and the epilogue; an empty slot streams its weights and stores nothing.  The same whole-K tiles and
// epilogue as w4a8_moe_gemm_run, so both give bit-identical rows.
static void moe_dev_schedule(int E, int N, int sms, int* tiles_per_cta, int* grid) {
  const int n_tiles = E * (N / dec::BM);
  const int tpc = (n_tiles + 2 * sms - 1) / (2 * sms);   // two CTAs per SM, whole tiles per CTA: no split-K
  *tiles_per_cta = tpc;
  *grid = (n_tiles + tpc - 1) / tpc;
}

int w4a8_moe_gemm_dev_run(const int8_t* x, const int8_t* qweight, const __half* wscales, const __half* ascales, const __half* w_szs,
                          const __half* a_ssums, __half* out, const int* offsets, int num_experts, int total_rows, int N, int K,
                          int ldc, cudaStream_t st) {
  using namespace dec;
  if (total_rows <= 0) return 0;
  if (num_experts <= 0 || num_experts > MOE_MAX_GROUPS || N % BM != 0 || K % BK != 0 || ldc < N) return OB_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(qweight) & 15)) return OB_ERR_ALIGN;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 16) return OB_ERR_ARG;
  const int sms = dev_sms(dev);
  CUtensorMap amap, wmap;
  if (int e = make_act_map(&amap, x, total_rows, K, 64)) return e;
  if (int e = make_w_map(&wmap, qweight, num_experts * N, K, false)) return e;   // experts stacked along N
  Params p{};
  p.wscales = wscales; p.ascales = ascales; p.w_szs = w_szs; p.a_ssums = a_ssums; p.out = out;
  p.ws = nullptr; p.counters = nullptr;   // whole tiles only: no split-K workspace
  p.M = 64; p.N = N; p.K = K; p.ldc = ldc;
  p.n_tiles_e = N / BM;
  p.kb_per_tile = K / BK;
  p.n_tiles = num_experts * p.n_tiles_e;
  int tpc = 0, grid = 0;
  moe_dev_schedule(num_experts, N, sms, &tpc, &grid);
  p.units_per_cta = tpc * p.kb_per_tile;
  const MoeDev d{offsets, total_rows};
  return launch_moe<64, true>(amap, wmap, p, d, grid, st);
}

// Host-only view of the launch above for a given offsets table (no CUDA call): grid, tiles per CTA and, per tile in tile
// order, (cta, slot, expert, n-tile, row0, rows) -- the rows after the kernel's clamping (moe_slot_rows).
int w4a8_moe_dev_plan(int num_experts, int N, int K, int sms, const int* offsets_host, int total_rows, int* grid, int* tiles_per_cta,
                      int* entries, int max_entries) {
  using namespace dec;
  if (num_experts <= 0 || num_experts > MOE_MAX_GROUPS || N <= 0 || N % BM != 0 || K <= 0 || K % BK != 0 || sms <= 0 || total_rows < 0)
    return OB_ERR_SHAPE;
  int tpc = 0, g = 0;
  moe_dev_schedule(num_experts, N, sms, &tpc, &g);
  if (grid) *grid = g;
  if (tiles_per_cta) *tiles_per_cta = tpc;
  if (!entries) return 0;
  const int n_tiles_e = N / BM, n_tiles = num_experts * n_tiles_e, KB = K / BK;
  if (!offsets_host || max_entries < n_tiles) return OB_ERR_ARG;
  const long long upc = (long long)tpc * KB;
  for (int tile = 0; tile < n_tiles; ++tile) {
    const int slot = tile / n_tiles_e;
    int row0 = 0, rows = 0;
    moe_slot_rows(offsets_host[slot], offsets_host[slot + 1], total_rows, &row0, &rows);
    int* o = entries + 6 * tile;
    o[0] = (int)((long long)tile * KB / upc);   // the CTA whose unit range holds the tile (SegIter)
    o[1] = slot; o[2] = slot; o[3] = tile - slot * n_tiles_e; o[4] = row0; o[5] = rows;
  }
  return 0;
}

}  // namespace ob
