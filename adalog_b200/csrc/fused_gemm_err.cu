// Fused candidate generator + GEMM + squared-error epilogue for the attention matmul sweeps (sm_100a).
//
// replaces: quant_layers/matmul.py:135-163 (_search_best_A_scale), :173-201 (_search_best_B_scale) and :321-351
// (post-softmax AdaLog base search) of the reference -- per candidate: fake-quantise one operand, A @ B, squared error
// against raw_out, mean.
//
// Why a second GEMM kernel.  In these sweeps K is the head dimension (64) or the key count (197) and the product has a
// single N tile, so the tensor work per unit is tiny (<= 512 clocks) and the two-kernel path (generator -> HBM
// workspace -> TMA -> MMA) is bound by writing and re-reading the 128x-expanded candidate operand (PV base search:
// 9.9 GB out + 9.9 GB in per sweep).  Here the expansion never leaves the SM:
//   * the group's fixed operand (<= 256 rows x <= 4 K blocks) is loaded ONCE per CTA by TMA and stays in shared memory;
//   * the producer warps generate the unit's 128 x K candidate tile straight into the 128B-swizzled K-major layout the
//     UMMA descriptor expects (exact fast path + IEEE fallback of quant_device.cuh, same as the generator kernels),
//     fence it to the async proxy and hand it to the MMA warp through an mbarrier;
//   * the epilogue warps reduce the error (TMEM lane p = candidate p, one register accumulator per candidate, static
//     work list => equal candidates give bit-equal sums), so produce(t+1), MMA(t) and epilogue(t-1) overlap.
// Warp roles (512 threads x 128 registers = the whole register file): warp 0 = TMA of the fixed operand, warp 1 = TMEM
// allocator + MMA issuer, then E = 4 or 8 epilogue warps and 14 - E producer warps (E chosen per shape by the host).
// (A first version that let the same eight warps alternate between producing and the epilogue was latency bound at
// two warps per scheduler: 2.4 ms per QK^T sweep against 1.3 + 1.1 ms for the two-kernel path.  ptxas 12.9 does not
// re-budget registers after setmaxnreg here, so the split is 8 + 4 warps at one uniform register count.)
#include "common.cuh"
#include "tc_common.cuh"
#include "quant_device.cuh"
#include "../../include/adalog_b200.h"
#include <type_traits>


namespace adalog {
namespace fused {

constexpr int kMaxBN = 256;
constexpr int kMaxKB = 4;               // K blocks of 128 bytes: K <= 256 (bf16) / 512 (int8)
constexpr int kAccStages = 8;            // TMEM accumulator stages: 512 columns / (BN rounded up to 64, 128 or 256)
constexpr uint32_t kTmemCols = 512;
constexpr int kEpiWarp0 = 2;
constexpr int kMaxEpiWarps = 8;         // 4 or 8 epilogue warps (one or two column groups), the other workers produce:
constexpr int kWorkWarps = 14;          // the split follows the shape (PV: N = 64, K = 197 wants 4 + 10; QK^T 8 + 6)
constexpr int kThreads = (kEpiWarp0 + kWorkWarps) * 32;    // 512 threads x 128 registers = the whole register file
constexpr int kMaxStages = 4;                              // candidate-tile stages (as many as fit in shared memory)
constexpr int kSlabsPerGroup = kMaxBN / 32;                // slabs one epilogue warp may handle (one column group)
constexpr uint32_t kABlock = kBM * 128;                    // bytes of one K block of the candidate tile (16 KiB)

struct __align__(16) Tail {
  float ysw[kMaxEpiWarps][kSlabsPerGroup * 32];
  float4 cand[ADALOG_P];        // uniform: {r/2n, zp/2n, L/2n, 1.5*2^23 - zp};  log: {1/(q 2n), 0, 0, q}
  float2 cand_sz[ADALOG_P];     // uniform: {s, zp} for the IEEE path
  float cthr[ADALOG_P];         // rounding-boundary threshold (negative: always IEEE path)
  float mt[64];
  double comb[kBM];             // sums of column group 1, folded into group 0's at the end
  uint64_t bfull, afull[kMaxStages], afree[kMaxStages];
  uint64_t tfull[kAccStages], tempty[kAccStages];
  uint32_t tmem_base;
};

struct FArgs {
  const float* x; long long ldx; int K;
  const float* cs; const float* cz; long long pstride, gstride, g_div, g_mod;
  const long long* cq; const float* mtab;
  int P, nl;
  int KB, N, BN, U, UG, cpg, nst, nacc, acc_cols, epi_warps;
  long long brpg, g_base, u_base;
  const float* y; long long ldy;
  const float* rs; long long rs_div, rs_mod;
  double* partial;
};

enum { GEN_UNIFORM = 0, GEN_LOG = 1 };

template <int GEN, bool I8>
__global__ void __launch_bounds__(kThreads, 1)
fused_cand_gemm_err_kernel(const __grid_constant__ CUtensorMap tmB, const FArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;                                            // [nst][KB][128 rows][128 B], SWIZZLE_128B
  uint8_t* sB = smem + (size_t)a.nst * a.KB * kABlock;           // [KB][BN rows][128 B]
  float* lut = reinterpret_cast<float*>(sB + (size_t)a.KB * a.BN * 128);   // GEN_LOG: [128][2n + 1]
  __shared__ Tail tl;

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int kProdWarp0 = kEpiWarp0 + a.epi_warps;
  const int kProdThreads = (kWorkWarps - a.epi_warps) * 32;
  const int kEpiThreads = a.epi_warps * 32;
  constexpr int EL = I8 ? 128 : 64;        // elements per 128-byte K block
  constexpr int EPT = I8 ? 16 : 8;         // elements per 16-byte chunk

  // static work list: the UG units of group g_local are dealt evenly to its cpg CTAs
  const int g_local = blockIdx.x / a.cpg;
  const int ci = blockIdx.x - g_local * a.cpg;
  const int u0 = g_local * a.UG + (int)(((long long)ci * a.UG) / a.cpg);
  const int u1 = min(g_local * a.UG + (int)(((long long)(ci + 1) * a.UG) / a.cpg), a.U);
  const int n_units = max(u1 - u0, 0);

  if (threadIdx.x == 0) {
    mbar_init(&tl.bfull, 1);
    for (int i = 0; i < kMaxStages; ++i) { mbar_init(&tl.afull[i], kWorkWarps - a.epi_warps); mbar_init(&tl.afree[i], 1); }
    for (int i = 0; i < kAccStages; ++i) { mbar_init(&tl.tfull[i], 1); mbar_init(&tl.tempty[i], a.epi_warps); }
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) prefetch_tmap(&tmB);
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tl.tmem_base)),
                 "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // per-candidate constants of this CTA's group (the candidates of a matmul sweep depend on the head only)
  const float ncode_f = (float)(2 * a.nl);
  if (warp >= kProdWarp0) {
    const int w = threadIdx.x - kProdWarp0 * 32;
    if (GEN == GEN_UNIFORM) {
      const long long g = ((a.u_base + u0) / a.g_div) % a.g_mod;
      const float L = (float)(2 * a.nl - 1);
      for (int p = w; p < ADALOG_P; p += kProdThreads) {
        const int pp = min(p, a.P - 1);          // pad rows repeat the last candidate
        const float s = __ldg(a.cs + pp * a.pstride + g * a.gstride);
        const float z = __ldg(a.cz + pp * a.pstride + g * a.gstride);
        const float r = __fdiv_rn(1.0f, s);
        const bool fast = z == rintf(z) && z >= 0.0f && z <= L && r == r && fabsf(r) <= 3.0e38f;
        tl.cand[p] = make_float4(r / ncode_f, z / ncode_f, L / ncode_f, kMagic - z);
        tl.cand_sz[p] = make_float2(s, z);
        tl.cthr[p] = fast ? kFracSafe : -1.0f;
      }
    } else {
      for (int j = w; j < 37; j += kProdThreads) tl.mt[j] = a.mtab[j];
      for (int p = w; p < ADALOG_P; p += kProdThreads) {
        const float qf = (float)a.cq[min(p, a.P - 1)];
        tl.cand[p] = make_float4(__fdiv_rn(1.0f, qf) / ncode_f, 0.0f, 0.0f, qf);
        tl.cthr[p] = kFracSafe;
      }
    }
  }
  // the candidate-tile stages start as zeros: chunks beyond K are never written again
  for (int i = threadIdx.x; i < a.nst * a.KB * (int)(kABlock / 16); i += kThreads)
    reinterpret_cast<uint4*>(sA)[i] = make_uint4(0u, 0u, 0u, 0u);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tl.tmem_base;
  if (GEN == GEN_LOG && warp >= kProdWarp0) {
    // lut[p][c] = mtab[(c q_p) % 37] * 2^-floor(c q_p / 37), 0 for the masked code c = 2n
    const int lw = 2 * a.nl + 1;
    for (int i = threadIdx.x - kProdWarp0 * 32; i < ADALOG_P * lw; i += kProdThreads) {
      const int p = i / lw, c = i - p * lw;
      float val = 0.0f;
      if (c < 2 * a.nl) {
        const int cqi = c * (int)tl.cand[p].w;
        const int e = cqi / 37;
        if (e <= 120) val = ldexpf(tl.mt[cqi - e * 37], -e);
      }
      lut[i] = val;
    }
    asm volatile("bar.sync 2, %0;" ::"r"(kProdThreads) : "memory");
  }

  if (warp == 0) {
    // ===================== fixed operand: once per CTA =====================
    if (lane == 0 && n_units > 0) {
      const uint32_t blk = (uint32_t)a.BN * 128u;
      mbar_expect_tx(&tl.bfull, blk * (uint32_t)a.KB);
      const long long brow = (a.g_base + g_local) * a.brpg;
      for (int kb = 0; kb < a.KB; ++kb) tma_load_2d(&tmB, &tl.bfull, sB + (size_t)kb * blk, kb * EL, (int)brow);
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // all 32 lanes run this loop converged; one elected lane issues each K block's tcgen05 instructions in a single
    // asm block (umma_kblock_commit, tc_common.cuh: the one-lane form cost ~17 SASS instructions per MMA, more than
    // the 104 clocks an N = 208, K = 16 MMA takes -- the issuing warp, not TMEM, bounded this kernel)
    if (n_units > 0) {
      const uint32_t idesc = I8 ? make_idesc_i8(a.BN) : make_idesc(a.BN);
      const uint32_t blk = (uint32_t)a.BN * 128u;
      const uint32_t sA_u = smem_u32(sA), sB_u = smem_u32(sB);
      mbar_wait(&tl.bfull, 0);
      // ring positions advance incrementally: a division by a run-time stage count is a dependent chain of ~25
      // instructions, and four of them per unit sat on the issuing warp's critical path
      uint32_t as = 0, aphase = 0, st = 0, sphase = 0;
      for (int t = 0; t < n_units; ++t) {
        mbar_wait(&tl.tempty[as], aphase ^ 1);
        mbar_wait(&tl.afull[st], sphase);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * a.acc_cols;
        for (int kb = 0; kb < a.KB; ++kb) {
          // UMMA_K = 16 bf16 / 32 int8 = 32 bytes; K slices that are all padding are skipped.  The last block's
          // commit frees the candidate tile once these MMAs retire.
          const int ks = min(4, (a.K - kb * EL + EL / 4 - 1) / (EL / 4));
          umma_kblock_commit<I8>(tmem_d, make_smem_desc(sA_u + (uint32_t)(st * a.KB + kb) * kABlock),
                                 make_smem_desc(sB_u + (uint32_t)kb * blk), idesc, kb != 0 ? 1u : 0u, ks,
                                 kb == a.KB - 1 ? smem_u32(&tl.afree[st]) : 0u);
        }
        umma_commit_elect(smem_u32(&tl.tfull[as]));      // accumulator ready for the epilogue
        if (++as == (uint32_t)a.nacc) { as = 0; aphase ^= 1; }
        if (++st == (uint32_t)a.nst) { st = 0; sphase ^= 1; }
      }
    }
  } else if (warp >= kEpiWarp0 && warp < kProdWarp0) {
    // ===================== epilogue: TMEM -> registers -> per-candidate squared error =====================
    const int ew = warp - kEpiWarp0;
    const int eg = ew >> 2;                                   // column group
    const int et = ((warp & 3) << 5) | lane;                  // candidate p = TMEM lane this thread reads
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    const int G = a.epi_warps >> 2;                           // column groups: 1 or 2
    float* const ysw = tl.ysw[ew];
    float rs = 0.0f;
    if (n_units > 0) rs = __ldg(a.rs + (((a.u_base + u0) / a.rs_div) % a.rs_mod) * kBM + et);
    TwoSumF acc;                                               // hi/lo FP32 pair: see tc_common.cuh
    float acc4[4];
    float yreg[kSlabsPerGroup];
    const int my_slabs = max(0, (((a.N + 31) >> 5) - eg + G - 1) / G);     // slabs eg, eg+G, ... below N
    auto load_y = [&](int u) {
#pragma unroll
      for (int i = 0; i < kSlabsPerGroup; ++i) {
        if (i >= my_slabs) break;
        const int c = (eg + i * G) * 32 + lane;
        yreg[i] = (c < a.N) ? __ldg(a.y + (long long)u * a.ldy + c) : 0.0f;
      }
    };
    auto accf = [](uint32_t v) -> float { return I8 ? __int2float_rn((int)v) : __uint_as_float(v); };
    const float nrs = -rs;
    auto quad = [&](auto masked, const uint32_t (&d)[32], int j, int l0, int lim) {
      constexpr bool MASKED = decltype(masked)::value;
      const float4 yv = *reinterpret_cast<const float4*>(&ysw[l0 + j]);
      if (!MASKED) {
        // two columns per packed FP32 instruction (FFMA2: same IEEE result per lane, half the FMA-pipe slots)
        float e0, e1, e2, e3;
        ffma2(e0, e1, nrs, nrs, accf(d[j]), accf(d[j + 1]), yv.x, yv.y);
        ffma2(e2, e3, nrs, nrs, accf(d[j + 2]), accf(d[j + 3]), yv.z, yv.w);
        ffma2(acc4[0], acc4[1], e0, e1, e0, e1, acc4[0], acc4[1]);
        ffma2(acc4[2], acc4[3], e2, e3, e2, e3, acc4[2], acc4[3]);
        return;
      }
      const float y4[4] = {yv.x, yv.y, yv.z, yv.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float diff = fmaf(-rs, accf(d[j + e]), y4[e]);
        diff = (j + e < lim) ? diff : 0.0f;
        acc4[e] = fmaf(diff, diff, acc4[e]);
      }
    };
    auto consume = [&](const uint32_t (&d)[32], int l0, int lim) {
      if (lim >= 32) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) quad(std::false_type{}, d, j, l0, 32);
      } else {
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          if (j < lim) quad(std::true_type{}, d, j, l0, lim);
      }
    };
    const int nslab = (a.N + 31) >> 5;
    if (n_units > 0) load_y(u0);
    uint32_t as = 0, aphase = 0;
    for (int t = 0; t < n_units; ++t) {
      __syncwarp();                      // every lane is done reading the previous unit's staging row
#pragma unroll
      for (int i = 0; i < kSlabsPerGroup; ++i) {
        if (i >= my_slabs) break;
        ysw[i * 32 + lane] = yreg[i];
      }
      __syncwarp();
      if (t + 1 < n_units) load_y(u0 + t + 1);   // consumed at the top of the next iteration
      mbar_wait(&tl.tfull[as], aphase);
      tc_fence_after();
      acc4[0] = acc4[1] = acc4[2] = acc4[3] = 0.0f;
      const uint32_t tbase = tmem_base + lane_base + as * a.acc_cols;
      uint32_t da[32], db[32];
      if (eg < nslab) tmem_ld32(tbase + eg * 32, da);
      int l0 = 0;
      for (int sl = eg; sl < nslab; sl += 2 * G, l0 += 64) {
        tmem_ld_wait();
        if (sl + G < nslab) tmem_ld32(tbase + (sl + G) * 32, db);
        consume(da, l0, a.N - sl * 32);
        if (sl + G < nslab) {
          tmem_ld_wait();
          if (sl + 2 * G < nslab) tmem_ld32(tbase + (sl + 2 * G) * 32, da);
          consume(db, l0 + 32, a.N - (sl + G) * 32);
        }
      }
      acc.add((acc4[0] + acc4[1]) + (acc4[2] + acc4[3]));
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tl.tempty[as]);
      if (++as == (uint32_t)a.nacc) { as = 0; aphase ^= 1; }
    }
    // fold the column groups in fixed order
    const double acc64 = acc.value();
    if (eg > 0) tl.comb[et] = acc64;
    asm volatile("bar.sync 1, %0;" ::"r"(kEpiThreads) : "memory");
    if (eg == 0) a.partial[(long long)blockIdx.x * kBM + et] = G > 1 ? acc64 + tl.comb[et] : acc64;
  } else if (warp >= kProdWarp0) {
    // ===================== producers: the unit's 128 x K candidate tile, straight into swizzled smem =====================
    // thread -> one 16-byte chunk of the row (ch) for candidates cg, cg + ncg, ...
    const int w = threadIdx.x - kProdWarp0 * 32;
    const int cpr = (a.K + EPT - 1) / EPT;                    // chunks that hold real K elements (the padding chunks of
    const int ncg = kProdThreads / cpr;                       // every stage were zeroed once, before the loop)
    const int ch = w % cpr, cg = w / cpr;
    const bool prod = cg < ncg;
    const int kc = ch * EPT;
    const bool tail = kc + EPT > a.K;
    const uint32_t c_in = (uint32_t)(ch & 7);
    const int lw = 2 * a.nl + 1;
    const uint32_t lut_bias = smem_u32(lut) - 0x2D000000u;    // addr = bits(t + 1.5*2^23) * 4 + lut_bias (mod 2^32)
    float xn[EPT];
    auto load_x = [&](int u) {
#pragma unroll
      for (int j = 0; j < EPT; ++j)
        xn[j] = (prod && kc + j < a.K) ? __ldg(a.x + (long long)u * a.ldx + kc + j) : (GEN == GEN_LOG ? 1.0f : 0.0f);
    };
    if (n_units > 0) load_x(u0);
    uint32_t st = 0, sphase = 0;
    for (int t = 0; t < n_units; ++t) {
      const uint32_t a_chunk = smem_u32(sA) + (uint32_t)(st * a.KB + (ch >> 3)) * kABlock;
      float xv[EPT];
#pragma unroll
      for (int j = 0; j < EPT; ++j) xv[j] = xn[j];
      if (t + 1 < n_units) load_x(u0 + t + 1);
      mbar_wait(&tl.afree[st], sphase ^ 1);     // the MMAs that read this stage have retired
      if (prod) {
        if (GEN == GEN_UNIFORM) {
          int nan_flag = 0;
#pragma unroll
          for (int j = 0; j < EPT; ++j) nan_flag |= (xv[j] != xv[j]) ? 1 : 0;
          asm volatile("" : "+r"(nan_flag));
          const float L = (float)(2 * a.nl - 1);
          // two candidates per iteration: 2 x EPT independent dependency chains per thread (a producer warp on its own
          // reaches ~0.15 IPC on one chain set; the register file leaves no room for more producer warps)
          auto u_gen = [&](int p, float (&tm)[EPT]) -> bool {
            const float4 c = tl.cand[p];
            const float thr = tl.cthr[p];
            // uq_code_fast (quant_device.cuh) on two elements per packed FP32 instruction; the distances to the rounded
            // values are reduced by a max tree and tested once per (candidate, chunk)
            float dm[EPT];
#pragma unroll
            for (int j = 0; j < EPT; j += 2) {
              const float ts0 = fminf(__saturatef(fmaf(xv[j], c.x, c.y)), c.z);
              const float ts1 = fminf(__saturatef(fmaf(xv[j + 1], c.x, c.y)), c.z);
              float n0, n1;
              ffma2(tm[j], tm[j + 1], ts0, ts1, ncode_f, ncode_f, c.w, c.w);        // (code - zp) + 1.5*2^23
              fadd2(n0, n1, c.w, c.w, -tm[j], -tm[j + 1]);                          // -(rounded clamped value)
              ffma2(dm[j], dm[j + 1], ts0, ts1, ncode_f, ncode_f, n0, n1);          // clamped - rint(clamped)
            }
#pragma unroll
            for (int w2 = EPT / 2; w2 > 0; w2 >>= 1) {
#pragma unroll
              for (int j = 0; j < w2; ++j) dm[j] = fmaxf(fabsf(dm[j]), fabsf(dm[j + w2]));
            }
            return nan_flag != 0 || !(dm[0] <= thr);
          };
          auto u_fix = [&](int p, float (&tm)[EPT], bool unsafe) {
            if (unsafe) {
              const float2 sz = tl.cand_sz[p];
#pragma unroll
              for (int j = 0; j < EPT; ++j) tm[j] = __fadd_rn(uq_int(xv[j], sz.x, sz.y, L), kMagic);
            }
            if (tail) {
#pragma unroll
              for (int j = 0; j < EPT; ++j) if (kc + j >= a.K) tm[j] = kMagic;
            }
          };
          auto u_store = [&](int p, const float (&tm)[EPT]) {
            uint32_t o0, o1, o2, o3;
            if (I8) {
              o0 = pack_i8x4_bits(tm[0], tm[1], tm[2], tm[3]);   o1 = pack_i8x4_bits(tm[4], tm[5], tm[6], tm[7]);
              o2 = pack_i8x4_bits(tm[8 % EPT], tm[9 % EPT], tm[10 % EPT], tm[11 % EPT]);
              o3 = pack_i8x4_bits(tm[12 % EPT], tm[13 % EPT], tm[14 % EPT], tm[15 % EPT]);
            } else {
              o0 = pack_bf16x2(__fsub_rn(tm[0], kMagic), __fsub_rn(tm[1], kMagic));
              o1 = pack_bf16x2(__fsub_rn(tm[2], kMagic), __fsub_rn(tm[3], kMagic));
              o2 = pack_bf16x2(__fsub_rn(tm[4 % EPT], kMagic), __fsub_rn(tm[5 % EPT], kMagic));
              o3 = pack_bf16x2(__fsub_rn(tm[6 % EPT], kMagic), __fsub_rn(tm[7 % EPT], kMagic));
            }
            const uint32_t addr = a_chunk + (uint32_t)p * 128u + ((c_in ^ ((uint32_t)p & 7u)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(o0), "r"(o1), "r"(o2), "r"(o3)
                         : "memory");
          };
          for (int p = cg; p < ADALOG_P; p += 2 * ncg) {
            const int p2 = p + ncg;
            const bool two = p2 < ADALOG_P;
            const int q2 = two ? p2 : p;
            float ta[EPT], tb[EPT];
            const bool ua = u_gen(p, ta);
            const bool ub = u_gen(q2, tb);
            u_fix(p, ta, ua);
            u_fix(q2, tb, ub);
            u_store(p, ta);
            if (two) u_store(p2, tb);
          }
        } else {
          // post-softmax AdaLog base search (matmul.py:337-342): c = rint(-log2(x) * 37 / q), no scale, no clamp.
          // (Every thread logs its own 8-element chunk; sharing one log2f per element through shared memory was
          // measured slower -- 11.1 -> 13.2 ms on the Swin window shape -- because of the per-unit producer barrier.)
          float lx[EPT], e1[EPT];
          int bad = 0;
#pragma unroll
          for (int j = 0; j < EPT; ++j) {
            lx[j] = -log2f(xv[j]);
            e1[j] = __fmul_rn(lx[j], 37.0f);
            bad |= !(lx[j] <= __int_as_float(0x7f800000)) ? 1 : 0;      // NaN
          }
          asm volatile("" : "+r"(bad));
          auto l_gen = [&](int p, float (&v)[EPT]) -> bool {
            const float4 c = tl.cand[p];
            uint32_t row = lut_bias + (uint32_t)(p * lw) * 4u;
            asm volatile("" : "+r"(row));
            float dm[EPT];
#pragma unroll
            for (int j = 0; j < EPT; j += 2) {
              const float ts0 = __saturatef(__fmul_rn(e1[j], c.x));
              const float ts1 = __saturatef(__fmul_rn(e1[j + 1], c.x));
              float tm0, tm1, n0, n1;
              ffma2(tm0, tm1, ts0, ts1, ncode_f, ncode_f, kMagic, kMagic);
              fadd2(n0, n1, kMagic, kMagic, -tm0, -tm1);
              ffma2(dm[j], dm[j + 1], ts0, ts1, ncode_f, ncode_f, n0, n1);
              float val0, val1;
              asm("ld.shared.f32 %0, [%1];" : "=f"(val0) : "r"(__float_as_uint(tm0) * 4u + row));
              asm("ld.shared.f32 %0, [%1];" : "=f"(val1) : "r"(__float_as_uint(tm1) * 4u + row));
              v[j] = val0; v[j + 1] = val1;
            }
#pragma unroll
            for (int w2 = EPT / 2; w2 > 0; w2 >>= 1) {
#pragma unroll
              for (int j = 0; j < w2; ++j) dm[j] = fmaxf(fabsf(dm[j]), fabsf(dm[j + w2]));
            }
            return bad != 0 || !(dm[0] <= kFracSafe);
          };
          auto l_fix = [&](int p, float (&v)[EPT], bool unsafe) {
            if (unsafe) {
              const float qf = tl.cand[p].w;
#pragma unroll
              for (int j = 0; j < EPT; ++j) v[j] = log_value_slow(xv[j], lx[j], false, 1.0f, qf, tl.mt, ncode_f);
            }
            if (tail) {
#pragma unroll
              for (int j = 0; j < EPT; ++j) if (kc + j >= a.K) v[j] = 0.0f;
            }
          };
          auto l_store = [&](int p, const float (&v)[EPT]) {
            const uint32_t o0 = pack_bf16x2(v[0], v[1]), o1 = pack_bf16x2(v[2], v[3]);
            const uint32_t o2 = pack_bf16x2(v[4 % EPT], v[5 % EPT]), o3 = pack_bf16x2(v[6 % EPT], v[7 % EPT]);
            const uint32_t addr = a_chunk + (uint32_t)p * 128u + ((c_in ^ ((uint32_t)p & 7u)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(o0), "r"(o1), "r"(o2), "r"(o3)
                         : "memory");
          };
          for (int p = cg; p < ADALOG_P; p += 2 * ncg) {
            const int p2 = p + ncg;
            const bool two = p2 < ADALOG_P;
            const int q2 = two ? p2 : p;
            float va[EPT], vb[EPT];
            const bool ua = l_gen(p, va);
            const bool ub = l_gen(q2, vb);
            l_fix(p, va, ua);
            l_fix(q2, vb, ub);
            l_store(p, va);
            if (two) l_store(p2, vb);
          }
        }
      }
      fence_proxy_async();               // generic-proxy stores -> visible to the tensor core's async proxy
      __syncwarp();
      if (lane == 0) mbar_arrive(&tl.afull[st]);
      if (++st == (uint32_t)a.nst) { st = 0; sphase ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

static size_t smem_bytes(const adalog_fused_args* a, int nst) {
  size_t b = 1024 + (size_t)nst * a->KB * kABlock + (size_t)a->KB * a->BN * 128;
  if (a->gen == ADALOG_GEN_LOG) b += (size_t)ADALOG_P * (2 * a->n_levels + 1) * sizeof(float);
  return b;
}
constexpr size_t kSmemLimit = 227 * 1024 - sizeof(Tail);
// as many candidate-tile stages as fit (<= 4): the producers then run units ahead of the MMA, which with up to 8
// accumulator stages in TMEM turns the per-unit produce -> MMA -> epilogue hand-offs from a latency chain into queues
static int stages(const adalog_fused_args* a) {
  int n = 1;
  while (n < kMaxStages && smem_bytes(a, n + 1) <= kSmemLimit) ++n;
  return n;
}

static int validate(const adalog_fused_args* a, bool need_partial) {
  ADALOG_REQUIRE(a && a->x && a->Bm && a->y && a->rs, -1, "fused_cand_gemm_err: null pointer");
  ADALOG_REQUIRE(a->gen == ADALOG_GEN_UNIFORM || a->gen == ADALOG_GEN_LOG, -1, "fused_cand_gemm_err: bad gen");
  ADALOG_REQUIRE(a->dtype == ADALOG_BF16 || a->dtype == ADALOG_I8, -1, "fused_cand_gemm_err: bad dtype");
  ADALOG_REQUIRE(a->gen == ADALOG_GEN_UNIFORM ? (a->cs && a->cz) : (a->cq && a->mtab), -1,
                 "fused_cand_gemm_err: candidate arrays missing");
  ADALOG_REQUIRE(a->gen != ADALOG_GEN_LOG || (a->dtype == ADALOG_BF16 && 2 * a->n_levels <= 64), -2,
                 "fused_cand_gemm_err: AdaLog candidates are bf16 operands with n_bits <= 6");
  ADALOG_REQUIRE(a->dtype != ADALOG_I8 || a->n_levels <= 64, -2, "fused_cand_gemm_err: int8 operands need n_bits <= 7");
  ADALOG_REQUIRE(a->K > 0 && a->KB >= 1 && a->KB <= kMaxKB && a->K <= a->KB * (a->dtype == ADALOG_I8 ? 128 : 64) &&
                     a->K > (a->KB - 1) * (a->dtype == ADALOG_I8 ? 128 : 64), -1,
                 "fused_cand_gemm_err: K / KB mismatch (KB = ceil(K / 64|128) <= 4)");
  ADALOG_REQUIRE(a->N > 0 && a->BN >= a->N && a->BN <= kMaxBN && a->BN % 16 == 0, -1,
                 "fused_cand_gemm_err: one N tile: N <= BN <= 256, BN a multiple of 16");
  ADALOG_REQUIRE(a->U > 0 && a->UG > 0 && a->U % a->UG == 0 && a->upc > 0 && a->P > 0 && a->P <= ADALOG_P, -1,
                 "fused_cand_gemm_err: bad unit partition");
  ADALOG_REQUIRE(a->epi_warps == 4 || a->epi_warps == 8, -1, "fused_cand_gemm_err: epi_warps must be 4 or 8");
  ADALOG_REQUIRE(a->g_div > 0 && a->g_mod > 0 && a->rs_div > 0 && a->rs_mod > 0, -1, "fused_cand_gemm_err: bad group map");
  // one CTA works inside one group, and the candidates / row scales must be constant over it
  ADALOG_REQUIRE(a->g_div % a->UG == 0 && a->rs_div % a->UG == 0 && a->u_base % a->UG == 0, -1,
                 "fused_cand_gemm_err: candidate and row-scale groups must be whole unit groups");
  ADALOG_REQUIRE(smem_bytes(a, 1) <= kSmemLimit, -3, "fused_cand_gemm_err: operands do not fit in shared memory");
  ADALOG_REQUIRE(a->partial || !need_partial, -1, "fused_cand_gemm_err: partial required");
  return 0;
}

static int launch(const adalog_fused_args* a, cudaStream_t st) {
  FArgs k;
  k.x = a->x; k.ldx = a->ldx; k.K = a->K;
  k.cs = a->cs; k.cz = a->cz; k.pstride = a->pstride; k.gstride = a->gstride; k.g_div = a->g_div; k.g_mod = a->g_mod;
  k.cq = a->cq; k.mtab = a->mtab; k.P = a->P; k.nl = a->n_levels;
  k.KB = a->KB; k.N = a->N; k.BN = a->BN; k.U = a->U; k.UG = a->UG; k.cpg = (a->UG + a->upc - 1) / a->upc;
  k.nst = stages(a);
  k.acc_cols = a->BN <= 64 ? 64 : (a->BN <= 128 ? 128 : 256);
  k.nacc = (int)kTmemCols / k.acc_cols;
  k.epi_warps = a->epi_warps;
  k.brpg = a->brpg; k.g_base = a->g_base; k.u_base = a->u_base;
  k.y = a->y; k.ldy = a->ldy; k.rs = a->rs; k.rs_div = a->rs_div; k.rs_mod = a->rs_mod; k.partial = a->partial;
  const bool i8 = a->dtype == ADALOG_I8;
  CUtensorMap tmB;
  int rc = make_map(&tmB, a->Bm, a->b_rows, (int64_t)a->KB * (i8 ? 128 : 64), a->BN, i8);
  if (rc) return rc;
  const unsigned grid = (unsigned)((a->U / a->UG) * k.cpg);
  const size_t smem = smem_bytes(a, k.nst);
#define ADALOG_LAUNCH_FUSED(GN, I8)                                                                            \
  do {                                                                                                         \
    cudaFuncSetAttribute(fused_cand_gemm_err_kernel<GN, I8>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                         (int)smem);                                                                           \
    fused_cand_gemm_err_kernel<GN, I8><<<grid, kThreads, smem, st>>>(tmB, k);                                  \
  } while (0)
  if (a->gen == ADALOG_GEN_LOG) ADALOG_LAUNCH_FUSED(GEN_LOG, false);
  else if (i8)                  ADALOG_LAUNCH_FUSED(GEN_UNIFORM, true);
  else                          ADALOG_LAUNCH_FUSED(GEN_UNIFORM, false);
#undef ADALOG_LAUNCH_FUSED
  return check_launch("fused_cand_gemm_err");
}

}  // namespace fused
}  // namespace adalog

extern "C" {

int adalog_fused_cand_gemm_err_grid(const adalog_fused_args* a) {
  int rc = adalog::fused::validate(a, false);
  if (rc) return rc;
  return (a->U / a->UG) * ((a->UG + a->upc - 1) / a->upc);
}

int adalog_fused_cand_gemm_err(const adalog_fused_args* a, void* stream) {
  int rc = adalog::fused::validate(a, true);
  if (rc) return rc;
  return adalog::fused::launch(a, (cudaStream_t)stream);
}

}  // extern "C"
