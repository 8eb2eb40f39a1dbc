// Candidate-batched GEMM with fused squared-error epilogue for sm_100a (tcgen05 + TMEM + TMA).
//
// One 128-row M tile = the 128 candidates of one "unit" (a token, a weight row, a Q/K/V row ...), so TMEM
// lane p holds candidate p and every epilogue thread owns exactly one candidate: the per-candidate error is
// accumulated in a register across the CTA's whole static work list with no cross-thread reduction, which
// keeps equal candidates bit-equal (exact-tie parity, SURVEY.md section 7 hard part 1).
//
// Warp roles (320 threads): warps 0-7 = epilogue (TMEM lanes 32*(w%4)..; two column groups), warp 8 = TMA producer,
// warp 9 = TMEM allocator + MMA issuer (the whole warp runs the issue loop converged, one elected lane issues each K
// block's tcgen05 instructions in a single asm block: tc_common.cuh umma_kblock_commit).  Pipelines: smem full/empty
// ring (kStages) between TMA and MMA; TMEM full/empty (2 accumulator stages of 256 columns) between MMA and epilogue.
#include "common.cuh"
#include "tc_common.cuh"
#include "../../include/adalog_b200.h"
#include <cuda.h>
#include <cudaTypedefs.h>
#include <type_traits>

namespace adalog {

constexpr int kMaxBN = 256;
constexpr int kStages = 4;
constexpr int kAccStages = 2;
constexpr uint32_t kABytes = kBM * kBK * 2;        // 16 KiB
constexpr uint32_t kBBytes = kMaxBN * kBK * 2;     // 32 KiB
constexpr uint32_t kTmemCols = 512;
constexpr int kEpiWarp0 = 0;            // epilogue warps 0-7, then warp 8: TMA producer, warp 9: MMA issuer + TMEM allocator: the
                                        // arbiter favours the highest warp id, and the two single-lane control warps must
                                        // never wait for an issue slot behind the epilogue (no idle warps: the registers
                                        // they would pin are what lets a generator CTA co-reside on the SM)
constexpr int kEpiWarps = 8;            // two epilogue warps per scheduler (16 was measured slower: register cap + barrier cost)
constexpr int kEpiGroups = kEpiWarps / 4; // column groups: group g takes the 32-column slabs g, g+G, g+2G, ...
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kTmaWarp = kEpiWarps, kMmaWarp = kEpiWarps + 1;
constexpr int kThreads = (kMmaWarp + 1) * 32;   // 320

// barriers and the epilogue's per-tile y / column-scale staging live in STATIC shared memory so that the compiler
// keeps the shared address space (LDS/STS, not generic LD/ST); the operand ring is dynamic (1024-byte aligned).
constexpr int kCsCols = 1024;           // MODE_CS: most columns (N tiles per split x BN) one CTA may cover
constexpr int kSlabsPerGroup = (kMaxBN / 32 + kEpiGroups - 1) / kEpiGroups;   // 32-column slabs one epilogue warp handles per tile
struct __align__(16) SmemTail {
  // per-WARP staging of y - cb and cs for the warp's own slabs (16-byte aligned: read back as float4 broadcasts).
  // Private to the warp, so a tile needs two __syncwarp()s and no CTA-wide barrier: the eight epilogue warps drift
  // apart and fill each other's TMEM-load and barrier latencies.
  float ysw[kEpiWarps][kSlabsPerGroup * 32];
  // MODE_CS: column scale / bias of ALL the CTA's N tiles, staged once per CTA (they do not depend on the unit);
  // zero beyond the CTA's columns so ragged / padded columns read 0
  float cs_all[kCsCols + kMaxBN];
  float cb_all[kCsCols + kMaxBN];
  uint64_t full[kStages];
  uint64_t empty[kStages];
  uint64_t tfull[kAccStages];
  uint64_t tempty[kAccStages];
  uint32_t tmem_base;
  uint32_t pad;
  double comb[kEpiGroups - 1][kBM];   // sums of column groups 1.., folded into group 0's in fixed order at the end
};
constexpr size_t kSmemBytes = 1024 /*align slack*/ + (size_t)kStages * (kABytes + kBBytes);

struct KArgs {
  int KB, N, BN, NT, U, UG, upc, cpg;
  int gx, S, split_fast;   // logical grid (gx unit lists x S N-tile splits) laid out on a 1-D launch
  long long brpg, g_base, u_base;
  const float* y; long long ldy;
  const float* rs; const float* rb; long long rs_div, rs_mod;
  const float* cs; const float* cb;
  double* partial;
  float* dbg;   // debug mode: dump D[128, N] of the single tile
  float* out; long long ldo; long long m_rows;   // MODE_STORE: output matrix [m_rows, N], row pitch ldo
};

// ---------------------------------------------------------------- the kernel
// MODE_CS: yhat = rs*(cs[n]*D), y' = y - cb[n] (linear A-side sweeps); MODE_RB: yhat = rs*D + rb (W-side sweeps);
// MODE_PLAIN: yhat = rs*D (attention matmuls)
// MODE_STORE: no error at all -- out[u*128+p, n] = rs*cs[n]*D + cb[n] is written (the fake-quant INFERENCE forward of a
// linear layer: rows p of unit u are 128 consecutive tokens, not candidates)
enum { MODE_CS = 0, MODE_RB = 1, MODE_PLAIN = 2, MODE_STORE = 4 };

template <int MODE, bool DEBUG, bool I8>
// 152 registers x 320 threads leave 16.9k registers of the SM free: one 256-thread generator CTA (64 registers) of the
// next chunk runs beside this kernel's single CTA
__global__ void __maxnreg__(152)
cand_gemm_err_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const KArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = smem + (size_t)kStages * kABytes;
  __shared__ SmemTail tail_s;
  SmemTail* tail = &tail_s;

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;

  // static work list of this CTA.  Logical coordinates (bx = unit list, by = N-tile split) come off a 1-D grid in
  // one of two orders: unit-fast (co-resident CTAs walk the same fixed-operand tiles: those stay in L2) or
  // split-fast (the S CTAs that share one unit list are co-resident: the candidate operand is fetched once).
  const int bx = a.split_fast ? (int)(blockIdx.x / a.S) : (int)(blockIdx.x % a.gx);
  const int by = a.split_fast ? (int)(blockIdx.x % a.S) : (int)(blockIdx.x / a.gx);
  const int g_local = bx / a.cpg;
  const int ci = bx - g_local * a.cpg;
  // the UG units of a group are dealt evenly to its cpg CTAs (sizes differ by at most one)
  const int u0 = g_local * a.UG + (int)(((long long)ci * a.UG) / a.cpg);
  const int u1 = min(g_local * a.UG + (int)(((long long)(ci + 1) * a.UG) / a.cpg), a.U);
  const int nt0 = (int)(((long long)by * a.NT) / a.S);
  const int nt1 = (int)(((long long)(by + 1) * a.NT) / a.S);
  const int n_units = max(u1 - u0, 0);
  const int n_nt = nt1 - nt0;
  const int n_tiles = n_units * n_nt;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(&tail->full[i], 1); mbar_init(&tail->empty[i], 1); }
    for (int i = 0; i < kAccStages; ++i) { mbar_init(&tail->tfull[i], 1); mbar_init(&tail->tempty[i], kEpiWarps); }
    fence_barrier_init();
  }
  if (warp == kTmaWarp && lane == 0) { prefetch_tmap(&tmA); prefetch_tmap(&tmB); }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tail->tmem_base)),
                 "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tail->tmem_base;

  if (warp == kTmaWarp) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      const uint32_t tx = kABytes + (uint32_t)a.BN * kBK * 2;
      int pu = u0, pcnt = 0;
      for (int t = 0; t < n_tiles; ++t) {
        const int u = pu;
        const int nt = nt0 + pcnt;
        if (++pcnt == n_nt) { pcnt = 0; ++pu; }
        const long long brow = (a.g_base + g_local) * a.brpg + (long long)nt * a.BN;
        for (int kb = 0; kb < a.KB; ++kb) {
          mbar_wait(&tail->empty[stage], phase ^ 1);
          mbar_expect_tx(&tail->full[stage], tx);
          const int kel = kb * (I8 ? 2 * kBK : kBK);    // K coordinate in elements (64 bf16 or 128 int8 = 128 bytes)
          tma_load_2d(&tmA, &tail->full[stage], sA + (size_t)stage * kABytes, kel, u * kBM);
          tma_load_2d(&tmB, &tail->full[stage], sB + (size_t)stage * kBBytes, kel, (int)brow);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ===================== MMA issuer =====================
    // all 32 lanes run this loop converged; one elected lane issues the K block's tcgen05 instructions in a single asm
    // block (umma_kblock_commit, tc_common.cuh: the one-lane form cost ~17 SASS instructions per MMA)
    {
      uint32_t stage = 0, phase = 0;
      const uint32_t idesc = I8 ? make_idesc_i8(a.BN) : make_idesc(a.BN);
      const uint32_t sA_u = smem_u32(sA), sB_u = smem_u32(sB);
      for (int t = 0; t < n_tiles; ++t) {
        const uint32_t as = t & 1, aphase = (t >> 1) & 1;
        mbar_wait(&tail->tempty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * kMaxBN;
        for (int kb = 0; kb < a.KB; ++kb) {
          mbar_wait(&tail->full[stage], phase);
          tc_fence_after();
          // UMMA_K = 16 bf16 or 32 int8 = 32 bytes -> +2 in the (addr>>4) field per K slice; the commit frees the
          // smem slot when these MMAs retire
          umma_kblock_commit<I8>(tmem_d, make_smem_desc(sA_u + stage * kABytes), make_smem_desc(sB_u + stage * kBBytes),
                                 idesc, kb != 0 ? 1u : 0u, 4, smem_u32(&tail->empty[stage]));
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit_elect(smem_u32(&tail->tfull[as]));         // accumulator ready for the epilogue
      }
    }
  } else if (warp < kTmaWarp) {
    // ===================== epilogue: TMEM -> registers -> per-candidate squared error =====================
    // 8 warps: warp w reads TMEM lanes 32*(w%4)..+31 (candidate p = that lane); group eg = (w-2)/4 takes the 32-column
    // slabs with index == eg (mod 2).  Every candidate therefore has two partial sums, folded in fixed order at the end.
    constexpr bool HAS_CS = MODE == MODE_CS || MODE == MODE_STORE;   // column scale / bias staged per CTA
    constexpr bool STORE = MODE == MODE_STORE;
    const int ew = warp - kEpiWarp0;
    const int eg = ew >> 2;                                 // column group 0..kEpiGroups-1
    const int et = ((warp & 3) << 5) | lane;                // 0..127 = candidate p = TMEM lane (a warp reaches lanes 32*(warp%4)..)
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    constexpr int G = kEpiGroups;
    float* const ysw = tail_s.ysw[ew];
    TwoSumF acc;                        // hi/lo FP32 pair: see tc_common.cuh
    float rs = 0.0f, rb = 0.0f;
    long long cur_ri = -1;
    float yreg[kSlabsPerGroup];
#pragma unroll
    for (int i = 0; i < kSlabsPerGroup; ++i) yreg[i] = 0.0f;
    if (HAS_CS) {
      const int st = threadIdx.x - kEpiWarp0 * 32;
      const int ncs = n_nt * a.BN;                       // <= kCsCols (validated on the host)
      for (int idx = st; idx < kCsCols + kMaxBN; idx += kEpiThreads) {
        float cv = 0.0f, bv = 0.0f;
        if (idx < ncs) {
          const int ti = idx / a.BN;
          const int c = idx - ti * a.BN;
          const int n = (nt0 + ti) * a.BN + c;
          if (n < a.N) { cv = __ldg(a.cs + n); bv = __ldg(a.cb + n); }
        }
        tail_s.cs_all[idx] = cv;
        tail_s.cb_all[idx] = bv;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
    }
    // global loads of y for tile t+1 (lane l: column l of each of the warp's slabs) are issued before tile t's math and
    // only consumed (y - cb, store to the warp's staging row) at the top of the next iteration, so their latency hides
    // under the epilogue arithmetic.  Columns beyond the tile / beyond N stage as 0.
    auto prefetch = [&](int u, int n0) {
#pragma unroll
      for (int i = 0; i < kSlabsPerGroup; ++i) {
        const int c = (eg + i * G) * 32 + lane;
        const int n = n0 + c;
        yreg[i] = (!STORE && c < a.BN && n < a.N) ? __ldg(a.y + (long long)u * a.ldy + n) : 0.0f;
      }
    };
    // four independent accumulators (same instruction sequence for every lane = candidate, so equal candidates still
    // produce bit-equal sums)
    float acc4[4];
    // accumulator word -> FP32: kind::f16 accumulates in FP32, kind::i8 in S32 (exact integer dot products)
    auto accf = [](uint32_t w) -> float { return I8 ? __int2float_rn((int)w) : __uint_as_float(w); };
    float* orow = nullptr;   // MODE_STORE: this thread's output row (nullptr beyond m_rows)
    int ocol = 0;            // MODE_STORE: output column of the current slab's column 0
    const bool ovec = STORE && (a.ldo & 3) == 0 && (reinterpret_cast<uintptr_t>(a.out) & 15) == 0;
    // four columns j..j+3 of a slab staged at local offset l0; MASKED: columns >= lim contribute nothing
    auto quad = [&](auto masked, const uint32_t (&d)[32], int j, int l0, int cc, int lim, float rs, float rb) {
      constexpr bool MASKED = decltype(masked)::value;
      const float4 yv = *reinterpret_cast<const float4*>(&ysw[l0 + j]);
      const float y4[4] = {yv.x, yv.y, yv.z, yv.w};
      float c4[4] = {1.0f, 1.0f, 1.0f, 1.0f};
      if (HAS_CS) {
        const float4 cv = *reinterpret_cast<const float4*>(&tail_s.cs_all[cc + j]);
        c4[0] = cv.x; c4[1] = cv.y; c4[2] = cv.z; c4[3] = cv.w;
      }
      if (STORE) {
        // rb carries the output row pointer's validity through `orow` (set per tile); columns beyond N are not written
        const float4 bv = *reinterpret_cast<const float4*>(&tail_s.cb_all[cc + j]);
        float4 o;
        o.x = fmaf(rs * c4[0], accf(d[j + 0]), bv.x); o.y = fmaf(rs * c4[1], accf(d[j + 1]), bv.y);
        o.z = fmaf(rs * c4[2], accf(d[j + 2]), bv.z); o.w = fmaf(rs * c4[3], accf(d[j + 3]), bv.w);
        if (orow != nullptr) {
          float* dst = orow + ocol + j;
          if (!MASKED || j + 3 < lim) {
            if (ovec) *reinterpret_cast<float4*>(dst) = o;
            else { dst[0] = o.x; dst[1] = o.y; dst[2] = o.z; dst[3] = o.w; }
          } else {
            if (j + 0 < lim) dst[0] = o.x;
            if (j + 1 < lim) dst[1] = o.y;
            if (j + 2 < lim) dst[2] = o.z;
          }
        }
        return;
      }
      if (!MASKED) {
        // two columns per packed FP32 instruction (FFMA2 / FMUL2 / FADD2: the same IEEE result per lane in half the
        // FMA-pipe slots)
        const float f0 = accf(d[j]), f1 = accf(d[j + 1]), f2 = accf(d[j + 2]), f3 = accf(d[j + 3]);
        float e0, e1, e2, e3;
        if (HAS_CS) {
          float t0, t1, t2, t3;
          fmul2(t0, t1, f0, f1, c4[0], c4[1]);
          fmul2(t2, t3, f2, f3, c4[2], c4[3]);
          ffma2(e0, e1, -rs, -rs, t0, t1, y4[0], y4[1]);
          ffma2(e2, e3, -rs, -rs, t2, t3, y4[2], y4[3]);
        } else if (MODE == MODE_RB) {
          float t0, t1, t2, t3;
          ffma2(t0, t1, rs, rs, f0, f1, rb, rb);
          ffma2(t2, t3, rs, rs, f2, f3, rb, rb);
          fadd2(e0, e1, y4[0], y4[1], -t0, -t1);
          fadd2(e2, e3, y4[2], y4[3], -t2, -t3);
        } else {
          ffma2(e0, e1, -rs, -rs, f0, f1, y4[0], y4[1]);
          ffma2(e2, e3, -rs, -rs, f2, f3, y4[2], y4[3]);
        }
        ffma2(acc4[0], acc4[1], e0, e1, e0, e1, acc4[0], acc4[1]);
        ffma2(acc4[2], acc4[3], e2, e3, e2, e3, acc4[2], acc4[3]);
        return;
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float diff;
        if (HAS_CS) diff = fmaf(-rs, accf(d[j + e]) * c4[e], y4[e]);
        else if (MODE == MODE_RB) diff = y4[e] - fmaf(rs, accf(d[j + e]), rb);
        else diff = fmaf(-rs, accf(d[j + e]), y4[e]);
        diff = (j + e < lim) ? diff : 0.0f;
        acc4[e] = fmaf(diff, diff, acc4[e]);
      }
    };
    // one 32-column slab of the accumulator (tile column c0, y staged at local offset l0, column scales at cs_all[cc],
    // lim valid columns)
    auto consume = [&](const uint32_t (&d)[32], int c0, int l0, int cc, int lim, float rs, float rb, int n0, int ncols) {
      if (DEBUG) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (c0 + j < ncols) a.dbg[(long long)et * a.N + n0 + c0 + j] = accf(d[j]);
      }
      ocol = c0;
      if (lim >= 32) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) quad(std::false_type{}, d, j, l0, cc, 32, rs, rb);
      } else {
        // ragged last slab: whole quads up to the one that holds column lim-1, its excess columns masked
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          if (j < lim) quad(std::true_type{}, d, j, l0, cc, lim, rs, rb);
      }
    };
    // incremental work-list position (no per-tile integer division)
    int cu = u0, cnt = 0;                       // current unit, N tile within the unit
    long long ri = 0, rrem = 0;                 // row-scale group of `cu`, (u_base + cu) % rs_div
    if (n_tiles > 0) {
      const long long gu = a.u_base + cu;
      ri = (gu / a.rs_div) % a.rs_mod;
      rrem = gu % a.rs_div;
      prefetch(cu, (nt0 + cnt) * a.BN);
    }
    for (int t = 0; t < n_tiles; ++t) {
      const int n0 = (nt0 + cnt) * a.BN;
      const int toff = cnt * a.BN;               // this tile's columns inside cs_all / cb_all
      const int ncols = min(a.BN, a.N - n0);
      const long long ri_t = ri;
      if (STORE) {
        const long long row = (a.u_base + cu) * kBM + et;
        orow = row < a.m_rows ? a.out + row * a.ldo + n0 : nullptr;
      }
      // advance to tile t+1
      if (++cnt == n_nt) {
        cnt = 0; ++cu;
        if (++rrem == a.rs_div) { rrem = 0; if (++ri == a.rs_mod) ri = 0; }
      }
      const uint32_t as = t & 1, aphase = (t >> 1) & 1;
      __syncwarp();                      // every lane is done reading the previous tile's staging row
#pragma unroll
      for (int i = 0; i < kSlabsPerGroup; ++i)
        ysw[i * 32 + lane] = HAS_CS ? yreg[i] - tail_s.cb_all[toff + (eg + i * G) * 32 + lane] : yreg[i];
      __syncwarp();
      if (t + 1 < n_tiles) prefetch(cu, (nt0 + cnt) * a.BN);
      if (ri_t != cur_ri) {
        cur_ri = ri_t;
        rs = __ldg(a.rs + ri_t * kBM + et);
        rb = (MODE == MODE_RB) ? __ldg(a.rb + ri_t * kBM + et) : 0.0f;
      }
      mbar_wait(&tail->tfull[as], aphase);
      tc_fence_after();
      acc4[0] = acc4[1] = acc4[2] = acc4[3] = 0.0f;
      const uint32_t tbase = tmem_base + lane_base + as * kMaxBN;
      // this group's slabs eg, eg+G, eg+2G, ...; TMEM -> registers double buffered: the load of the next slab is in
      // flight while the current one is reduced
      const int nslab = (ncols + 31) >> 5;
      uint32_t da[32], db[32];
      if (eg < nslab) tmem_ld32(tbase + eg * 32, da);
      int l0 = 0;
      // MODE_RB (W-side / conv sweeps): the columns are this rank's calibration tokens, so the FP32 partial is folded
      // into the (error-free) accumulator per 32-column slab.  Slabs sit at absolute multiples of 32 tokens (BN % 32 == 0 on this path), hence
      // every FP32 rounding is the same however the tokens are sharded over GPUs (shards of a multiple of 32 tokens)
      // or tiled; what remains order-dependent is the ~2^-48 error of adding FP32-valued terms.  The other modes sum over the
      // output features of whole units (tokens / rows), which no sharding splits: one promotion per tile.
      constexpr bool SLAB64 = MODE == MODE_RB;
      auto flush = [&]() {
        acc.add((acc4[0] + acc4[1]) + (acc4[2] + acc4[3]));
        acc4[0] = acc4[1] = acc4[2] = acc4[3] = 0.0f;
      };
      for (int sl = eg; sl < nslab; sl += 2 * G, l0 += 64) {
        tmem_ld_wait();
        if (sl + G < nslab) tmem_ld32(tbase + (sl + G) * 32, db);
        consume(da, sl * 32, l0, toff + sl * 32, ncols - sl * 32, rs, rb, n0, ncols);
        if (SLAB64) flush();
        if (sl + G < nslab) {
          tmem_ld_wait();
          if (sl + 2 * G < nslab) tmem_ld32(tbase + (sl + 2 * G) * 32, da);
          consume(db, (sl + G) * 32, l0 + 32, toff + (sl + G) * 32, ncols - (sl + G) * 32, rs, rb, n0, ncols);
          if (SLAB64) flush();
        }
      }
      if (!SLAB64) acc.add((acc4[0] + acc4[1]) + (acc4[2] + acc4[3]));
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tail->tempty[as]);
    }
    // fold the column groups in fixed order: ((group 0 + group 1) + group 2) + ...
    const double acc64 = acc.value();
    if (eg > 0) tail_s.comb[eg - 1][et] = acc64;
    asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
    if (eg == 0 && a.partial) {
      double tot = acc64;
#pragma unroll
      for (int g = 1; g < kEpiGroups; ++g) tot += tail_s.comb[g - 1][et];
      a.partial[((long long)by * a.gx + bx) * kBM + et] = tot;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// ---------------------------------------------------------------- host side
static int validate(const adalog_gemm_err_args* a, bool need_partial) {
  ADALOG_REQUIRE(a && a->A && a->Bm, -1, "cand_gemm_err: null operand");
  ADALOG_REQUIRE(a->KB > 0 && a->N > 0 && a->U > 0 && a->UG > 0 && a->upc > 0 && a->S > 0, -1,
                 "cand_gemm_err: non-positive size");
  ADALOG_REQUIRE(a->BN >= 16 && a->BN <= kMaxBN && a->BN % 16 == 0, -1, "cand_gemm_err: BN must be a multiple of 16 in [16,256]");
  ADALOG_REQUIRE(a->dtype == ADALOG_BF16 || a->dtype == ADALOG_I8, -1, "cand_gemm_err: dtype must be ADALOG_BF16 or ADALOG_I8");
  ADALOG_REQUIRE(a->order == ADALOG_ORDER_UNIT_FAST || a->order == ADALOG_ORDER_SPLIT_FAST, -1, "cand_gemm_err: bad order");
  ADALOG_REQUIRE(a->U % a->UG == 0, -1, "cand_gemm_err: U must be a multiple of UG");
  ADALOG_REQUIRE(a->a_rows >= (int64_t)a->U * kBM, -1, "cand_gemm_err: A has fewer than U*128 rows");
  ADALOG_REQUIRE(a->rs_div > 0 && a->rs_mod > 0 && a->rs, -1, "cand_gemm_err: row scale required");
  ADALOG_REQUIRE((a->cs == nullptr) == (a->cb == nullptr), -1, "cand_gemm_err: cs and cb come together");
  ADALOG_REQUIRE(!a->rb || a->cs || a->BN % 32 == 0, -1,
                 "cand_gemm_err: with a row bias (W-side sweeps) BN must be a multiple of 32 (per-slab FP64 promotion)");
  ADALOG_REQUIRE(a->y && (a->partial || !need_partial), -1, "cand_gemm_err: y / partial required");
  const int NT = (a->N + a->BN - 1) / a->BN;
  ADALOG_REQUIRE(a->S <= NT, -1, "cand_gemm_err: more N splits than N tiles");
  ADALOG_REQUIRE(!a->cs || ((NT + a->S - 1) / a->S) * a->BN <= kCsCols, -1,
                 "cand_gemm_err: with column scales a CTA covers at most 1024 columns (raise S)");
  return 0;
}

static int launch(const adalog_gemm_err_args* a, float* dbg, cudaStream_t st, float* out = nullptr, long long ldo = 0,
                  long long m_rows = 0) {
  KArgs k;
  k.out = out; k.ldo = ldo; k.m_rows = m_rows;
  k.KB = a->KB; k.N = a->N; k.BN = a->BN; k.NT = (a->N + a->BN - 1) / a->BN; k.U = a->U; k.UG = a->UG; k.upc = a->upc;
  k.cpg = (a->UG + a->upc - 1) / a->upc;
  k.brpg = a->brpg; k.g_base = a->g_base; k.u_base = a->u_base;
  k.y = a->y; k.ldy = a->ldy; k.rs = a->rs; k.rb = a->rb; k.rs_div = a->rs_div; k.rs_mod = a->rs_mod;
  k.cs = a->cs; k.cb = a->cb; k.partial = a->partial; k.dbg = dbg;
  CUtensorMap tmA, tmB;
  const bool i8 = a->dtype == ADALOG_I8;
  const int64_t cols = (int64_t)a->KB * (i8 ? 2 * kBK : kBK);
  int rc = make_map(&tmA, a->A, a->a_rows, cols, kBM, i8);
  if (rc) return rc;
  rc = make_map(&tmB, a->Bm, a->b_rows, cols, a->BN, i8);
  if (rc) return rc;
  k.gx = (a->U / a->UG) * k.cpg; k.S = a->S; k.split_fast = a->order == ADALOG_ORDER_SPLIT_FAST;
  dim3 grid((unsigned)((long long)k.gx * k.S));
#define ADALOG_LAUNCH_GEMM(MD, DBG, I8)                                                                       \
  do {                                                                                                        \
    cudaFuncSetAttribute(cand_gemm_err_kernel<MD, DBG, I8>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                         (int)kSmemBytes);                                                                    \
    cand_gemm_err_kernel<MD, DBG, I8><<<grid, kThreads, kSmemBytes, st>>>(tmA, tmB, k);                       \
  } while (0)
  if (out) {
    if (i8) ADALOG_LAUNCH_GEMM(MODE_STORE, false, true);
    else    ADALOG_LAUNCH_GEMM(MODE_STORE, false, false);
  } else if (i8) {
    if (dbg)         ADALOG_LAUNCH_GEMM(MODE_PLAIN, true, true);
    else if (a->cs)  ADALOG_LAUNCH_GEMM(MODE_CS, false, true);
    else if (a->rb)  ADALOG_LAUNCH_GEMM(MODE_RB, false, true);
    else             ADALOG_LAUNCH_GEMM(MODE_PLAIN, false, true);
  } else {
    if (dbg)         ADALOG_LAUNCH_GEMM(MODE_PLAIN, true, false);
    else if (a->cs)  ADALOG_LAUNCH_GEMM(MODE_CS, false, false);
    else if (a->rb)  ADALOG_LAUNCH_GEMM(MODE_RB, false, false);
    else             ADALOG_LAUNCH_GEMM(MODE_PLAIN, false, false);
  }
#undef ADALOG_LAUNCH_GEMM
  return check_launch("cand_gemm_err");
}

}  // namespace adalog

using namespace adalog;

extern "C" {

int adalog_cand_gemm_err_grid(const adalog_gemm_err_args* a) {
  int rc = validate(a, false);
  if (rc) return rc;
  return (a->U / a->UG) * ((a->UG + a->upc - 1) / a->upc);
}

int adalog_cand_gemm_err(const adalog_gemm_err_args* a, void* stream) {
  int rc = validate(a, true);
  if (rc) return rc;
  return launch(a, nullptr, (cudaStream_t)stream);
}

int adalog_gemm_dequant(const adalog_gemm_err_args* a, float* out, int64_t ldo, int64_t m_rows, void* stream) {
  ADALOG_REQUIRE(a && out && m_rows > 0 && ldo >= a->N, -1, "gemm_dequant: bad output");
  ADALOG_REQUIRE(a->A && a->Bm && a->rs && a->cs && a->cb && a->KB > 0 && a->N > 0 && a->U > 0 && a->UG == a->U &&
                     a->upc > 0 && a->S > 0 && (int64_t)a->U * kBM >= m_rows && a->rs_div > 0 && a->rs_mod > 0, -1,
                 "gemm_dequant: bad arguments (one group, U = ceil(m_rows / 128), rs / cs / cb required)");
  ADALOG_REQUIRE(a->BN >= 16 && a->BN <= kMaxBN && a->BN % 16 == 0, -1, "gemm_dequant: BN must be a multiple of 16 in [16,256]");
  ADALOG_REQUIRE(a->dtype == ADALOG_BF16 || a->dtype == ADALOG_I8, -1, "gemm_dequant: dtype");
  ADALOG_REQUIRE(a->order == ADALOG_ORDER_UNIT_FAST || a->order == ADALOG_ORDER_SPLIT_FAST, -1, "gemm_dequant: order");
  const int NT = (a->N + a->BN - 1) / a->BN;
  ADALOG_REQUIRE(a->S <= NT && ((NT + a->S - 1) / a->S) * a->BN <= kCsCols, -1,
                 "gemm_dequant: a CTA covers at most 1024 columns (raise S)");
  return launch(a, nullptr, (cudaStream_t)stream, out, ldo, m_rows);
}

int adalog_debug_gemm_tile(const void* A, const void* Bm, int KB, int N, float* D, const float* zeros, const float* ones,
                           double* partial, int dtype, void* stream) {
  // y = 0, rs = 1 come from the caller (zeros [N], ones [128], partial [64 * 128] doubles): no library-owned device state
  ADALOG_REQUIRE(A && Bm && D && zeros && ones && partial && KB > 0 && N > 0, -1, "debug_gemm_tile: bad arguments");
  double* part = partial;
  adalog_gemm_err_args a;
  memset(&a, 0, sizeof(a));
  a.A = A; a.Bm = Bm; a.a_rows = kBM; a.b_rows = N; a.KB = KB; a.N = N; a.dtype = dtype;
  a.BN = N >= kMaxBN ? kMaxBN : ((N + 15) / 16) * 16;
  a.U = 1; a.UG = 1; a.upc = 1; a.S = 1; a.brpg = N; a.g_base = 0; a.u_base = 0;
  a.y = zeros; a.ldy = 0; a.rs = ones; a.rb = nullptr; a.rs_div = 1; a.rs_mod = 1; a.cs = nullptr; a.cb = nullptr;
  a.partial = part;
  int rc = validate(&a, true);
  if (rc) return rc;
  return launch(&a, D, (cudaStream_t)stream);
}

}  // extern "C"
