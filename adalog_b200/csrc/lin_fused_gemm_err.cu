// Linear-layer activation sweeps with the candidate operand generated INSIDE the GEMM kernel (sm_100a).
//
// replaces: quant_layers/linear.py:394-423 (_search_best_a_scale: 128 uniform (scale, zero-point) candidates on the
// layer input), :816-854 / :856-890 / :898-931 (post-GELU AdaLog scale, base and joint scale x base searches) of the
// reference -- per candidate: fake-quantise the input, F.linear against the quantised weight, squared error against
// raw_out, mean.
//
// Why.  The two-kernel path (generator -> 2 GiB HBM workspace -> TMA -> MMA) wrote and re-read the 128x-expanded
// candidate operand: 9.9 GB each way per DeiT-B fc2 evaluation against 0.39 GB of algorithmic bytes (x and raw_out
// read once), and the generator kernels were 20-28% of a calibration step although they were meant to hide under the
// GEMM of the previous chunk (one 8-warp generator CTA per SM next to the GEMM CTA ran at a fraction of its rate).
// Here one persistent CTA per SM owns a static list of units (tokens):
//   * 8 producer warps turn the unit's x row into the 128-candidate x 128-byte K-block tiles of the UMMA A operand,
//     straight into the 128B-swizzled shared-memory layout (exact fast path + IEEE fallback of quant_device.cuh, as in
//     the generator kernels: bit-identical operands), fence them to the async proxy and hand them over by mbarrier;
//   * warp 0 streams the fixed operand (the quantised weight, K-block x N-tile boxes) through a TMA ring -- it is the
//     same for every unit and stays in L2;
//   * warp 1 issues tcgen05.mma into TMEM; 4 epilogue warps (TMEM lane p = candidate p, one register accumulator per
//     candidate, static work list => equal candidates give bit-equal sums) reduce the error against y.
// Two schedules, chosen on the host by the shape:
//   RESIDENT (K small: all K blocks of a unit fit in shared memory).  The A tiles of a unit are generated ONCE and
//     used by every N tile; loop order unit > N tile > K block with two 256-column TMEM accumulators, so the epilogue
//     of tile t overlaps the MMAs of tile t+1 (these shapes are bound by the 64 B/clk TMEM read-out).  The A ring has
//     more stages than a unit has K blocks, so producers already write unit u+1 while unit u's last tiles multiply.
//   STREAMED (K large: fc2).  The unit's N columns (<= 512 per pass) sit in TMEM at once; loop order unit > pass >
//     K block > N tile, each generated K-block tile is consumed by all N tiles of the pass and freed.  N > 512 takes
//     ceil(N/512) passes that regenerate the operand (DeiT-B fc2: 2 passes; the generation then still costs less
//     issue time than the pass's MMAs take).
// Both are one loop nest: tile jobs t = 0,1,2,.. use TMEM slot t % NSLOT; a group of G consecutive tile jobs shares
// each A tile (G = 1 resident, G = N tiles per pass streamed).
#include "common.cuh"
#include "tc_common.cuh"
#include "quant_device.cuh"
#include "../../include/adalog_b200.h"
#include <algorithm>
#include <type_traits>

namespace adalog {
namespace linf {

// Warp roles.  20 worker warps split between producers (candidate generation) and epilogue (TMEM read-out + error):
//   uniform sweeps: 12 producers + 8 epilogue warps (two per TMEM lane quadrant, alternate 32-column slabs): the
//     epilogue costs ~3 issue slots per accumulator element and N is 1-4 x K;
//   AdaLog sweeps (fc2: N = K/4): 16 producers + 4 epilogue warps -- 64 candidate groups = exactly two candidates per
//     producer thread, and the epilogue has 1/16 of the generation's work.
// Warp order = issue priority (the arbiter favours the highest warp id of a scheduler): producers lowest, then the
// epilogue, and the single-lane control warps on top.
// 23 warps x 80 registers (the register file is allocated in 512-register units per warp: 23 x 2560): the generation is
// latency bound per warp (dependent FMA chains, LUT loads), so the producers get as many warps as the register file allows;
// the epilogue reads TMEM in 16-column pieces to fit the same budget.
constexpr int kWorkWarps = 20;
constexpr int kTmaWarp = kWorkWarps;                  // 20: TMA of the fixed operand
constexpr int kMmaWarp = kTmaWarp + 1;                // 21: MMA issuer + TMEM allocator
constexpr int kRelayWarp = kMmaWarp + 1;              // 22: turns "accumulator full" mbarrier phases into named-barrier arrivals
constexpr int kThreads = (kRelayWarp + 1) * 32;       // 736
constexpr int kBarTile0 = 3;                          // named barriers 3, 4: accumulator slot 0 / 1 is full
__host__ __device__ constexpr int prod_warps(int gen) { return gen == 1 ? 16 : 12; }
constexpr int kMaxSA = 12, kMaxSB = 8, kMaxSlots = 4;
constexpr uint32_t kATile = kBM * 128;                // one K block of the candidate tile: 128 rows x 128 bytes
constexpr uint32_t kTmemCols = 512;

struct __align__(16) Tail {
  float ysw[8 * 128];          // per epilogue warp: y - cb of its slabs of the current tile (0 beyond the tile)
  float csw[8 * 128];          // per epilogue warp: column scales of its slabs (0 beyond the tile: those columns add nothing)
  float4 cand[ADALOG_P];       // uniform: {r/2n, zp/2n, L/2n, 1.5*2^23 - zp};  log: {mul/2n, off/2n, lim, mul}
  float2 cand_sz[ADALOG_P];    // uniform: {s, zp};  log: {q, s}   (IEEE path)
  float cthr[ADALOG_P];        // uniform: rounding-boundary threshold (negative: always IEEE);  log: 0.5 - candidate margin
  float mt[64];
  double comb[kBM];            // sums of column group 1, folded into group 0's at the end
  float lim_min;
  uint32_t lut_bias[3];        // AdaLog: LUT base of this thread's i-th candidate minus 4 * bits(1.5*2^23), see the producers
  uint32_t tmem_base;
  uint64_t afull[kMaxSA], afree[kMaxSA], bfull[kMaxSB], bfree[kMaxSB], tfull[kMaxSlots], tempty[kMaxSlots];
};

struct LArgs {
  const float* x; long long ldx; int K, U;
  const float* cs; const float* cz; const long long* cq; const float* shift; const float* mtab;
  int P, nl;
  int KB, N, BN, NT, G, NG, nslot, slotw, SA, SB, streamed, vec;
  const float* y; long long ldy;
  const float* rs; const float* ccs; const float* ccb;
  double* partial;
};

enum { GEN_UNIFORM = 0, GEN_LOG = 1 };

// IEEE fallback of the AdaLog form, kept out of line (log2f, ldexpf, divisions: it would triple the producer code; the
// first version was 126 KB of SASS and lost 12% of the producers' issue slots to instruction-cache misses).  It runs
// for ~1e-4 of the chunks and returns its 8 values already packed (four bf16x2 words, in registers): an array parameter
// in local memory would drag the fast path's registers through the stack as well (measured: STL/LDL per candidate in
// the hot loop).
__device__ __noinline__ uint4 log_chunk_slow(const float* __restrict__ x, long long ldx, int u, int kc, int K, float sh,
                                             bool shifted, float s, float qf, const float* mt, float ncode) {
  const float* xsrc = x + (long long)u * ldx + kc;           // (computed here: the hot loop would otherwise carry it)
  const int n_valid = min(8, K - kc);
  uint32_t o[4];
  for (int j2 = 0; j2 < 4; ++j2) {
    float v2[2];
    for (int h = 0; h < 2; ++h) {
      const int j = 2 * j2 + h;
      float val = 0.0f;
      if (j < n_valid) {
        const float xs = shifted ? __fadd_rn(__ldg(xsrc + j), sh) : __ldg(xsrc + j);
        val = log_value_slow(xs, 0.0f, true, s, qf, mt, ncode);
      }
      v2[h] = val;
    }
    o[j2] = pack_bf16x2(v2[0], v2[1]);
  }
  return make_uint4(o[0], o[1], o[2], o[3]);
}

// IEEE path of a uniform chunk (uq_int: the reference's own operation order), out of line for the same reason; the
// chunk's source values are re-read from their shared-memory staging row (float4 q of the chunk at src_s + 128 q).
template <bool I8>
__device__ __noinline__ uint4 uq_chunk_slow(uint32_t src_s, float s, float z, float L) {
  uint32_t o[4];
  for (int w = 0; w < 4; ++w) {
    if (I8) {
      float4 x4;
      asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x4.x), "=f"(x4.y), "=f"(x4.z), "=f"(x4.w)
                   : "r"(src_s + (uint32_t)w * 128u));
      o[w] = pack_i8x4(uq_int(x4.x, s, z, L), uq_int(x4.y, s, z, L), uq_int(x4.z, s, z, L), uq_int(x4.w, s, z, L));
    } else {
      float x0, x1;
      asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(x0), "=f"(x1) : "r"(src_s + (uint32_t)(w >> 1) * 128u + (uint32_t)(w & 1) * 8u));
      o[w] = pack_bf16x2(uq_int(x0, s, z, L), uq_int(x1, s, z, L));
    }
  }
  return make_uint4(o[0], o[1], o[2], o[3]);
}

template <int GEN, bool I8>
__global__ void __maxnreg__(80)
lin_fused_kernel(const __grid_constant__ CUtensorMap tmB, const LArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;                                          // [SA][128 rows][128 B], SWIZZLE_128B
  uint8_t* sB = smem + (size_t)a.SA * kATile;                  // [SB][BN rows][128 B]
  const uint32_t bstage = (uint32_t)a.BN * 128u;
  float* lut = reinterpret_cast<float*>(sB + (size_t)a.SB * bstage);   // GEN_LOG: [128][2n + 1]
  // the unit's K source values, staged once per generation: x (uniform) or -log2(x + shift) (AdaLog)
  float* srcs = lut + (GEN == GEN_LOG ? ADALOG_P * (2 * a.nl + 1) : 0);
  // per 16-byte chunk of the staged row: the element part of the rounding margin (+inf: the chunk takes the IEEE path)
  float* chunk_g = srcs + a.KB * (GEN == GEN_LOG ? 64 : (I8 ? 128 : 64));
  __shared__ Tail tl;

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  constexpr int kProdWarps = prod_warps(GEN);
  constexpr int kEpiWarps = kWorkWarps - kProdWarps;       // 8 or 4
  constexpr int kEpiGroups = kEpiWarps / 4;                // column groups: warps of a TMEM lane quadrant take alternate slabs
  constexpr int kProdWarp0 = 0, kEpiWarp0 = kProdWarps;    // TMEM lane quadrant of an epilogue warp = warp % 4
  constexpr int kProdThreads = kProdWarps * 32;            // 8 chunks x 48 / 64 candidate groups
  constexpr int kCandGroups = kProdThreads / 8;
  constexpr int kCPT = (ADALOG_P + kCandGroups - 1) / kCandGroups;   // candidates per producer thread: cg + kCandGroups i
  constexpr int kEpiThreads = kEpiWarps * 32;
  constexpr int EL = I8 ? 128 : 64;        // elements per 128-byte K block
  constexpr int EPT = I8 ? 16 : 8;         // elements per 16-byte chunk

  // static unit list: the U units are dealt evenly to the CTAs (sizes differ by at most one)
  const int u0 = (int)(((long long)blockIdx.x * a.U) / gridDim.x);
  const int u1 = (int)(((long long)(blockIdx.x + 1) * a.U) / gridDim.x);
  const int n_units = u1 - u0;
  const int gen_per_unit = a.streamed ? a.NG : 1;       // how often a unit's A tiles are generated

  if (threadIdx.x == 0) {
    for (int i = 0; i < kMaxSA; ++i) { mbar_init(&tl.afull[i], kProdWarps); mbar_init(&tl.afree[i], 1); }
    for (int i = 0; i < kMaxSB; ++i) { mbar_init(&tl.bfull[i], 1); mbar_init(&tl.bfree[i], 1); }
    for (int i = 0; i < kMaxSlots; ++i) { mbar_init(&tl.tfull[i], 1); mbar_init(&tl.tempty[i], kEpiWarps); }
    fence_barrier_init();
  }
  if (warp == kTmaWarp && lane == 0) prefetch_tmap(&tmB);
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tl.tmem_base)),
                 "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // per-candidate constants (the candidates of a linear activation sweep are per-tensor: the same for every unit)
  const float ncode_f = (float)(2 * a.nl);
  const float sh = (GEN == GEN_LOG && a.shift) ? __ldg(a.shift) : 0.0f;
  if (warp >= kProdWarp0 && warp < kEpiWarp0) {
    const int w = threadIdx.x - kProdWarp0 * 32;
    if (GEN == GEN_UNIFORM) {
      const float L = (float)(2 * a.nl - 1);
      for (int p = w; p < ADALOG_P; p += kProdThreads) {
        const int pp = min(p, a.P - 1);          // pad rows repeat the last candidate
        const float s = __ldg(a.cs + pp), z = __ldg(a.cz + pp);
        const float r = __fdiv_rn(1.0f, s);
        const bool fast = z == rintf(z) && z >= 0.0f && z <= L && r == r && fabsf(r) <= 3.0e38f;
        tl.cand[p] = make_float4(r / ncode_f, z / ncode_f, L / ncode_f, kMagic - z);
        tl.cand_sz[p] = make_float2(s, z);
        tl.cthr[p] = fast ? kFracSafe : -1.0f;
      }
    } else {
      for (int j = w; j < 37; j += kProdThreads) tl.mt[j] = a.mtab[j];
      for (int p = w; p < ADALOG_P; p += kProdThreads) {
        const int pp = min(p, a.P - 1);
        const float qf = (float)a.cq[pp];
        const float s = __ldg(a.cs + pp);
        const float ls = -log2f(s);
        const float mul = __fdiv_rn(37.0f, qf);
        tl.cand[p] = make_float4(mul / ncode_f, -__fmul_rn(ls, mul) / ncode_f, __fadd_rn(ls, 49.0f), mul);
        tl.cand_sz[p] = make_float2(qf, s);
        tl.cthr[p] = 0.5f - (mul * 7.6e-7f * fabsf(ls) + 4e-7f * ncode_f);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tl.tmem_base;
  if (warp >= kEpiWarp0 && warp < kEpiWarp0 + 4) {
    // TMEM is not cleared by the allocator: zero it once, so that the columns of a slot the MMAs never write (between
    // BN and the next multiple of 32) read as 0 and not as whatever bit pattern (possibly NaN) was left there
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    for (int c = 0; c < (int)kTmemCols; c += 32) tmem_st32_zero(tmem_base + lane_base + c);
    tmem_st_wait();
  }
  if (GEN == GEN_LOG && warp >= kProdWarp0 && warp < kEpiWarp0) {
    const int w = threadIdx.x - kProdWarp0 * 32;
    // lut[p][c] = mtab[(c q_p) % 37] * 2^-floor(c q_p / 37), 0 for the masked code c = 2n
    const int lw = 2 * a.nl + 1;
    for (int i = w; i < ADALOG_P * lw; i += kProdThreads) {
      const int p = i / lw, c = i - p * lw;
      float val = 0.0f;
      if (c < 2 * a.nl) {
        const int cqi = c * (int)tl.cand_sz[p].x;
        const int e = cqi / 37;
        if (e <= 120) val = ldexpf(tl.mt[cqi - e * 37], -e);
      }
      // four candidates interleaved per code: lut[p >> 2][c][p & 3].  The 32 lanes of a producer warp look up four
      // consecutive candidates x eight elements at once; with one row of 2n + 1 words per candidate they spread over
      // 4 (2n + 1) words of 32 banks (ncu: 1.5 wavefronts per load); interleaved, two lanes collide only when their codes
      // differ by a multiple of 8 for the SAME candidate
      lut[((p >> 2) * lw + c) * 4 + (p & 3)] = val;
    }
    if (w == 0) {
      // byte address of lut[(p >> 2)][c][p & 3] = bits(c + (cg >> 2) lw + 1.5*2^23) * 16 + lut_bias[i] + (cg & 3) * 4  (mod 2^32)
      // for candidate p = cg + kCandGroups i: 16 * bits(1.5*2^23) = 0xB4000000 (mod 2^32)
      for (int i = 0; i < 3; ++i) tl.lut_bias[i] = smem_u32(lut) - 0xB4000000u + (uint32_t)(i * (kCandGroups / 4) * lw) * 16u;
      float m = __int_as_float(0x7f800000);
      for (int p = 0; p < ADALOG_P; ++p) m = fminf(m, tl.cand[p].z);
      tl.lim_min = m;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp == kTmaWarp) {
    // ===================== TMA: fixed operand, K-block x N-tile boxes in consumption order =====================
    if (lane == 0) {
      // (ring positions are advanced incrementally everywhere: a division by a run-time stage count costs a dependent
      // chain of ~25 instructions, and six of them per K step made the single issuing thread the bottleneck)
      uint32_t bs = 0, bph = 0;
      for (int u = 0; u < n_units; ++u)
        for (int g = 0; g < a.NG; ++g)
          for (int kb = 0; kb < a.KB; ++kb)
            for (int j = 0; j < a.G; ++j) {
              mbar_wait(&tl.bfree[bs], bph ^ 1);
              mbar_expect_tx(&tl.bfull[bs], bstage);
              tma_load_2d(&tmB, &tl.bfull[bs], sB + (size_t)bs * bstage, kb * EL, (g * a.G + j) * a.BN);
              if (++bs == (uint32_t)a.SB) { bs = 0; bph ^= 1; }
            }
    }
  } else if (warp == kMmaWarp) {
    // ===================== MMA issuer =====================
    // All 32 lanes run this loop converged; the tcgen05 instructions of a K block are issued by one elected lane in a
    // single asm block (umma_kblock_commit, tc_common.cuh).
    {
      const uint32_t idesc = I8 ? make_idesc_i8(a.BN) : make_idesc(a.BN);
      const int last_ks = min(4, (a.K - (a.KB - 1) * EL + EL / 4 - 1) / (EL / 4));   // live K slices of the last block
      uint32_t as0 = 0, aph0 = 0;          // ring position of the current generation's K block 0
      uint32_t bs = 0, bph = 0, tj = 0;
      const uint32_t sA_u = smem_u32(sA), sB_u = smem_u32(sB);
      for (int u = 0; u < n_units; ++u) {
        for (int g = 0; g < a.NG; ++g) {
          const bool a_first = a.streamed || g == 0;
          const bool a_last = a.streamed || g == a.NG - 1;
          uint32_t as = as0, aph = aph0;
          for (int kb = 0; kb < a.KB; ++kb) {
            if (a_first) mbar_wait(&tl.afull[as], aph);
            const uint64_t adesc = make_smem_desc(sA_u + as * kATile);
            for (int j = 0; j < a.G; ++j) {
              const uint32_t t = tj + j, ts = t & 1;
              if (kb == 0) mbar_wait(&tl.tempty[ts], ((t >> 1) & 1) ^ 1);
              mbar_wait(&tl.bfull[bs], bph);
              tc_fence_after();
              umma_kblock_commit<I8>(tmem_base + ts * 256u, adesc, make_smem_desc(sB_u + bs * bstage), idesc,
                                     kb != 0 ? 1u : 0u, kb == a.KB - 1 ? last_ks : 4, smem_u32(&tl.bfree[bs]));
              if (++bs == (uint32_t)a.SB) { bs = 0; bph ^= 1; }
            }
            if (a_last) umma_commit_elect(smem_u32(&tl.afree[as]));
            if (++as == (uint32_t)a.SA) { as = 0; aph ^= 1; }
          }
          for (int j = 0; j < a.G; ++j) umma_commit_elect(smem_u32(&tl.tfull[(tj + j) & 1]));
          tj += a.G;
          if (a_last) { as0 = as; aph0 = aph; }
        }
      }
    }
  } else if (warp == kRelayWarp) {
    // ===================== relay: tfull mbarrier phase -> named-barrier arrival (one polling warp instead of eight) ====
    const int n_jobs = n_units * a.NT;
    for (int t = 0; t < n_jobs; ++t) {
      mbar_wait(&tl.tfull[t & 1], ((uint32_t)t >> 1) & 1);
      asm volatile("bar.arrive %0, %1;" ::"r"(kBarTile0 + (t & 1)), "n"(kEpiThreads + 32) : "memory");
    }
  } else if (warp >= kEpiWarp0 && warp < kTmaWarp) {
    // ===================== epilogue: TMEM -> registers -> per-candidate squared error =====================
    // warp w reads TMEM lanes 32*(w%4).. (candidate p = that lane); column group eg = (w - kEpiWarp0)/4 takes the
    // 32-column slabs eg, eg+2, ...  Every candidate therefore has two partial sums, folded in fixed order at the end.
    const int ew = warp - kEpiWarp0;
    const int eg = ew >> 2;                                  // < kEpiGroups
    const int et = ((warp & 3) << 5) | lane;                 // candidate p = TMEM lane this thread reads
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    constexpr int kSlabs = 8 / kEpiGroups;                   // slabs of one column group in a 256-column slot
    float* const ysw = tl.ysw + ew * (kSlabs * 32);
    float* const csw = tl.csw + ew * (kSlabs * 32);
    const float nrs = -__ldg(a.rs + et);
    TwoSumF acc;                                              // hi/lo FP32 pair: see tc_common.cuh
    float acc4[4];
    float yreg[kSlabs], creg[kSlabs];
    auto accf = [](uint32_t v) -> float { return I8 ? __int2float_rn((int)v) : __uint_as_float(v); };
    // (y - cb, cs) for column lane of this group's slabs of tile nt of unit u; (0, 0) beyond the tile / beyond N
    auto load_y = [&](int u, int nt) {
      const int n0 = nt * a.BN;
#pragma unroll
      for (int i = 0; i < kSlabs; ++i) {
        const int c = (eg + kEpiGroups * i) * 32 + lane;
        const int n = n0 + c;
        const bool ok = c < a.BN && n < a.N;
        yreg[i] = ok ? __ldg(a.y + (long long)u * a.ldy + n) - __ldg(a.ccb + n) : 0.0f;
        creg[i] = ok ? __ldg(a.ccs + n) : 0.0f;
      }
    };
    // 16 columns: yhat = rs * (cs * D), e += (y' - yhat)^2, two columns per packed FP32 instruction
    auto consume = [&](const uint32_t (&d)[16], int l0) {
#pragma unroll
      for (int j = 0; j < 16; j += 4) {
        const float4 yv = *reinterpret_cast<const float4*>(&ysw[l0 + j]);
        const float4 cv = *reinterpret_cast<const float4*>(&csw[l0 + j]);
        float t0, t1, t2, t3, e0, e1, e2, e3;
        fmul2(t0, t1, accf(d[j]), accf(d[j + 1]), cv.x, cv.y);
        fmul2(t2, t3, accf(d[j + 2]), accf(d[j + 3]), cv.z, cv.w);
        ffma2(e0, e1, nrs, nrs, t0, t1, yv.x, yv.y);
        ffma2(e2, e3, nrs, nrs, t2, t3, yv.z, yv.w);
        ffma2(acc4[0], acc4[1], e0, e1, e0, e1, acc4[0], acc4[1]);
        ffma2(acc4[2], acc4[3], e2, e3, e2, e3, acc4[2], acc4[3]);
      }
    };
    const int n_jobs = n_units * a.NT;
    int cu = u0, cnt = 0;
    if (n_jobs > 0) load_y(cu, cnt);
    for (int t = 0; t < n_jobs; ++t) {
      const int n0 = cnt * a.BN;
      const int ncols = min(a.BN, a.N - n0);
      if (++cnt == a.NT) { cnt = 0; ++cu; }
      const uint32_t ts = (uint32_t)t & 1u;
      __syncwarp();                          // every lane is done reading the previous tile's staging rows
#pragma unroll
      for (int i = 0; i < kSlabs; ++i) { ysw[i * 32 + lane] = yreg[i]; csw[i * 32 + lane] = creg[i]; }
      __syncwarp();
      if (t + 1 < n_jobs) load_y(cu, cnt);   // consumed at the top of the next iteration
      // "slot ts is full": the relay warp watches the mbarrier and arrives on a named barrier, so that the eight
      // epilogue warps block in hardware instead of polling (ncu, AdaLog fc2 sweep: the nanosleep poll loop of these
      // warps came back every ~45 clocks and was 47% of all executed warp instructions)
      asm volatile("bar.sync %0, %1;" ::"r"(kBarTile0 + (int)ts), "n"(kEpiThreads + 32) : "memory");
      tc_fence_after();
      acc4[0] = acc4[1] = acc4[2] = acc4[3] = 0.0f;
      const uint32_t tbase = tmem_base + lane_base + ts * 256u;
      const int nslab = (ncols + 31) >> 5;
      // this group's 32-column slabs eg, eg+2, ... in 16-column pieces, TMEM -> registers double buffered
      uint32_t da[16], db[16];
      if (eg < nslab) tmem_ld16(tbase + eg * 32, da);
      int l0 = 0;
      for (int sl = eg; sl < nslab; sl += kEpiGroups, l0 += 32) {
        tmem_ld_wait();
        tmem_ld16(tbase + sl * 32 + 16, db);
        consume(da, l0);
        tmem_ld_wait();
        if (sl + kEpiGroups < nslab) tmem_ld16(tbase + (sl + kEpiGroups) * 32, da);
        consume(db, l0 + 16);
      }
      acc.add((acc4[0] + acc4[1]) + (acc4[2] + acc4[3]));
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tl.tempty[ts]);
    }
    const double acc64 = acc.value();
    if (kEpiGroups == 2) {
      if (eg == 1) tl.comb[et] = acc64;
      asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
      if (eg == 0) a.partial[(long long)blockIdx.x * kBM + et] = acc64 + tl.comb[et];
    } else {
      a.partial[(long long)blockIdx.x * kBM + et] = acc64;
    }
  } else {
    // ===================== producers: K-block tiles of the candidate operand, straight into swizzled smem =====================
    // thread -> 16-byte chunk ch of the row, candidates p_i = cg + kCandGroups i (i < kCPT, p_i < 128).  The candidates of a
    // thread never change, so their constants, LUT rows and store offsets live in registers for the whole kernel.
    const int w = threadIdx.x - kProdWarp0 * 32;
    const int ch = w & 7, cg = w >> 3;
    const int lw = 2 * a.nl + 1;
    // AdaLog LUT address = bits(code + row + 1.5*2^23) * 16 + bias (mod 2^32), see the LUT construction above: the
    // (cg >> 2) lw part of the row rides in the rounding constant kw, the candidate step and (cg & 3) in the bias -- read
    // back from shared memory so that ptxas cannot split the constant off again (it rematerialised shift + two adds per
    // element instead of ONE LEA when the value was computed in registers)
    const uint32_t lb0 = tl.lut_bias[0] + (uint32_t)(cg & 3) * 4u, lb1 = tl.lut_bias[1] + (uint32_t)(cg & 3) * 4u,
                   lb2 = tl.lut_bias[kCPT - 1] + (uint32_t)(cg & 3) * 4u;
    uint32_t srcs_s = smem_u32(srcs), sA_s = smem_u32(sA);
    asm volatile("" : "+r"(srcs_s), "+r"(sA_s));              // (ptxas otherwise rematerialises the aligned smem base per store)
    float kx[kCPT], ky[kCPT], kw[kCPT], kt[kCPT];
#pragma unroll
    for (int i = 0; i < kCPT; ++i) {
      const int p = min(cg + i * kCandGroups, ADALOG_P - 1);
      const float4 c = tl.cand[p];
      kx[i] = c.x; ky[i] = c.y; kt[i] = tl.cthr[p];
      // uniform: 1.5*2^23 - zp;  AdaLog: 1.5*2^23 + (cg >> 2) lw for all of them, so that the bits of the rounded value index
      // the LUT directly (exact ties, where the parity of this constant would matter, always take the IEEE path)
      kw[i] = GEN == GEN_LOG ? kMagic + (float)((cg >> 2) * lw) : c.w;
    }
    // row p = cg + 48 i of the tile: 128 bytes per row, chunk position swizzled by p & 7 == cg & 7 (48 % 8 == 0)
    const uint32_t so0 = (uint32_t)cg * 128u + (((uint32_t)ch ^ ((uint32_t)cg & 7u)) << 4);
    constexpr uint32_t kSoStep = (uint32_t)kCandGroups * 128u;
    const bool has3 = kCPT == 3 && cg + 2 * kCandGroups < ADALOG_P;   // warp-uniform: cg = 4 consecutive values per warp
    const float Lq = (float)(2 * a.nl - 1) / ncode_f;          // uniform: upper clamp L / 2n
    const float lim_min = GEN == GEN_LOG ? tl.lim_min : 0.0f;
    const int n_gen = n_units * gen_per_unit;                 // (unit, pass) pairs
    uint32_t as = 0, aph = 0;
    // The source row of the NEXT generation is fetched into registers while the current one is generated: the staging
    // below then starts from registers instead of waiting ~1.5k clocks for global memory between two barriers, with
    // the operand ring running empty meanwhile.  (kPre x kProdThreads elements; longer rows load the rest directly.)
    constexpr int kPre = 6;
    float pre[kPre];
    auto fetch_row = [&](int u) {
      const float* xrow = a.x + (long long)u * a.ldx;
#pragma unroll
      for (int i = 0; i < kPre; ++i) {
        const int k = w + i * kProdThreads;
        pre[i] = k < a.K ? __ldg(xrow + k) : (GEN == GEN_LOG ? 1.0f : 0.0f);
      }
    };
    if (n_gen > 0) fetch_row(u0);
    for (int gi = 0; gi < n_gen; ++gi) {
      const int u = u0 + (a.streamed ? gi / a.NG : gi);
      {
        // The unit's K source values, once per generation, shared by all producer threads through shared memory:
        // uniform: x itself;  AdaLog: -log2(x + shift) with the reference's full-precision log2f (~30 instructions)
        // ONCE per element instead of once per (element, candidate group).  Elements beyond K are staged as a benign
        // finite value: whatever they generate meets the zero K padding of the fixed operand.
        // Per 16-byte chunk, also once per generation: the element part of the rounding margin --
        //   AdaLog: (6e-7 max|lx| + 2e-7) 2n, or +inf when an element sits near the reference's 1e-15 clamp, x <= 0 or NaN;
        //   uniform: +inf when the chunk holds a NaN (FFMA.SAT turns it into 0), else 0
        // -- so the inner loops test ONE threshold per (candidate, chunk) and +inf routes the chunk to the IEEE path.
        asm volatile("bar.sync 2, %0;" ::"n"(kProdThreads) : "memory");      // everybody is done with the previous unit's values
        const float* xrow = a.x + (long long)u * a.ldx;
        auto stage = [&](int k, float v) {
          if (GEN == GEN_LOG && a.shift && k < a.K) v = __fadd_rn(v, sh);
          const float sv = GEN == GEN_LOG ? -log2f(v) : v;
          // staged per K block as [float4 index q][chunk][4]: the eight 16-byte pieces a quarter warp reads at once are
          // contiguous (one wavefront; the natural layout put them 32 bytes apart: two-way bank conflicts, ncu: 8
          // wavefronts per LDS.128 against 4)
          srcs[(k & ~(EL - 1)) + (((k & (EPT - 1)) >> 2) << 5) + (((k & (EL - 1)) / EPT) << 2) + (k & 3)] = sv;
          const float inf = __int_as_float(0x7f800000);
          float g = GEN == GEN_LOG ? (!(sv <= lim_min) ? inf : fabsf(sv)) : (sv != sv ? inf : 0.0f);
#pragma unroll
          for (int m = 1; m < EPT; m <<= 1) g = fmaxf(g, __shfl_xor_sync(0xffffffffu, g, m));
          if ((lane & (EPT - 1)) == 0) chunk_g[k / EPT] = GEN == GEN_LOG ? fmaf(6e-7f, g, 2e-7f) * ncode_f : g;
        };
        const int kend = a.KB * EL;                             // a multiple of 32: every loop below is warp-uniform
#pragma unroll
        for (int i = 0; i < kPre; ++i) {
          const int k = w + i * kProdThreads;
          if (k < kend) stage(k, pre[i]);
        }
        for (int k = w + kPre * kProdThreads; k < kend; k += kProdThreads)
          stage(k, k < a.K ? __ldg(xrow + k) : (GEN == GEN_LOG ? 1.0f : 0.0f));
        asm volatile("bar.sync 2, %0;" ::"n"(kProdThreads) : "memory");
        if (gi + 1 < n_gen) fetch_row(u0 + (a.streamed ? (gi + 1) / a.NG : gi + 1));
      }
      for (int kb = 0; kb < a.KB; ++kb) {
        const uint32_t a_tile = sA_s + as * kATile + so0;
        const int kc = kb * EL + ch * EPT;
        const bool live = kc < a.K;                           // chunks beyond K are written as zeros
        float xv[EPT];
#pragma unroll
        const uint32_t xsrc = srcs_s + (uint32_t)(kb * EL + ch * 4) * 4u;      // + 128 bytes per float4 of the chunk
        for (int j = 0; j < EPT; j += 4)
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                       : "=f"(xv[j]), "=f"(xv[j + 1]), "=f"(xv[j + 2]), "=f"(xv[j + 3]) : "r"(xsrc + (uint32_t)j * 32u));
        const float gch = chunk_g[kc / EPT];
        mbar_wait(&tl.afree[as], aph ^ 1);                   // the MMAs that read this stage have retired
        auto store = [&](int i, uint32_t o0, uint32_t o1, uint32_t o2, uint32_t o3) {      // i: compile-time after unrolling
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a_tile + (uint32_t)i * kSoStep), "r"(o0), "r"(o1), "r"(o2), "r"(o3) : "memory");
        };
        if (!live) {
          // a chunk beyond K (partial last block): the ring stage may hold another block's data from its last use
#pragma unroll
          for (int i = 0; i < kCPT; ++i) if (i < 2 || has3) store(i, 0u, 0u, 0u, 0u);
        } else if (GEN == GEN_UNIFORM) {
          // uq_code_fast (quant_device.cuh) on two elements per packed FP32 instruction; tm = (code - zp) + 1.5*2^23
          auto u_gen = [&](int i) -> uint4 {
            // distance to the rounded value of every element, reduced by a max TREE (a chain of `unsafe |= ...`
            // compiles to EPT serially dependent FSETPs); d is finite: ts is saturated to [0, 1]
            float tm[EPT], dm[EPT];
#pragma unroll
            for (int j = 0; j < EPT; j += 2) {
              const float ts0 = fminf(__saturatef(fmaf(xv[j], kx[i], ky[i])), Lq);
              const float ts1 = fminf(__saturatef(fmaf(xv[j + 1], kx[i], ky[i])), Lq);
              float n0, n1;
              ffma2(tm[j], tm[j + 1], ts0, ts1, ncode_f, ncode_f, kw[i], kw[i]);      // (code - zp) + 1.5*2^23
              fadd2(n0, n1, kw[i], kw[i], -tm[j], -tm[j + 1]);                        // -(rounded clamped value)
              ffma2(dm[j], dm[j + 1], ts0, ts1, ncode_f, ncode_f, n0, n1);            // clamped - rint(clamped)
            }
#pragma unroll
            for (int w2 = EPT / 2; w2 > 0; w2 >>= 1) {
#pragma unroll
              for (int j = 0; j < w2; ++j) dm[j] = fmaxf(fabsf(dm[j]), fabsf(dm[j + w2]));
            }
            if (!(fmaxf(dm[0], gch) <= kt[i])) {              // rare: redo the chunk on the IEEE path (out of line)
              const float2 sz = tl.cand_sz[min(cg + i * kCandGroups, ADALOG_P - 1)];
              return uq_chunk_slow<I8>(xsrc, sz.x, sz.y, (float)(2 * a.nl - 1));
            }
            if (I8)
              return make_uint4(pack_i8x4_bits(tm[0], tm[1], tm[2], tm[3]), pack_i8x4_bits(tm[4], tm[5], tm[6], tm[7]),
                                pack_i8x4_bits(tm[8 % EPT], tm[9 % EPT], tm[10 % EPT], tm[11 % EPT]),
                                pack_i8x4_bits(tm[12 % EPT], tm[13 % EPT], tm[14 % EPT], tm[15 % EPT]));
            return make_uint4(pack_bf16x2(__fsub_rn(tm[0], kMagic), __fsub_rn(tm[1], kMagic)),
                              pack_bf16x2(__fsub_rn(tm[2], kMagic), __fsub_rn(tm[3], kMagic)),
                              pack_bf16x2(__fsub_rn(tm[4 % EPT], kMagic), __fsub_rn(tm[5 % EPT], kMagic)),
                              pack_bf16x2(__fsub_rn(tm[6 % EPT], kMagic), __fsub_rn(tm[7 % EPT], kMagic)));
          };
#pragma unroll
          for (int i = 0; i < kCPT; ++i) {
            if (i < 2 || has3) {
              const uint4 o = u_gen(i);
              store(i, o.x, o.y, o.z, o.w);
            }
          }
        } else {
          // post-GELU AdaLog search form (linear.py:872-878, :913-919): see gen_log_cand_lut_kernel (quant_kernels.cu)
          // for the derivation of the exact fast path; same arithmetic, same margins, same IEEE fallback.  xv = lx here.
          // The chunk's LARGEST element margin (gch, staged above) is used for all of its elements -- conservative (a
          // few more chunks take the IEEE path, still ~1e-4 of them) -- so the per-element check shrinks to
          // |d| <= 0.5 - candidate margin - gch * mul / 2n.
          auto l_gen = [&](int i) -> uint4 {
            float dm[EPT], v[EPT];
            const float lim_d = fmaf(-gch, kx[i], kt[i]);
            const uint32_t lb = i == 0 ? lb0 : (i == 1 ? lb1 : lb2);
#pragma unroll
            for (int j = 0; j < EPT; j += 2) {
              const float ts0 = __saturatef(fmaf(xv[j], kx[i], ky[i]));
              const float ts1 = __saturatef(fmaf(xv[j + 1], kx[i], ky[i]));
              float tm0, tm1, n0, n1;
              ffma2(tm0, tm1, ts0, ts1, ncode_f, ncode_f, kw[i], kw[i]);              // code + LUT row + 1.5*2^23
              fadd2(n0, n1, kw[i], kw[i], -tm0, -tm1);
              ffma2(dm[j], dm[j + 1], ts0, ts1, ncode_f, ncode_f, n0, n1);
              float val0, val1;
              asm("ld.shared.f32 %0, [%1];" : "=f"(val0) : "r"(__float_as_uint(tm0) * 16u + lb));
              asm("ld.shared.f32 %0, [%1];" : "=f"(val1) : "r"(__float_as_uint(tm1) * 16u + lb));
              v[j] = val0; v[j + 1] = val1;
            }
#pragma unroll
            for (int w2 = EPT / 2; w2 > 0; w2 >>= 1) {
#pragma unroll
              for (int j = 0; j < w2; ++j) dm[j] = fmaxf(fabsf(dm[j]), fabsf(dm[j + w2]));
            }
            if (!(dm[0] <= lim_d)) {
              const float2 qs = tl.cand_sz[min(cg + i * kCandGroups, ADALOG_P - 1)];
              return log_chunk_slow(a.x, a.ldx, u, kc, a.K, sh, a.shift != nullptr, qs.y, qs.x, tl.mt, ncode_f);
            }
            return make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4 % EPT], v[5 % EPT]),
                              pack_bf16x2(v[6 % EPT], v[7 % EPT]));
          };
          // two candidates per iteration: 2 x EPT independent dependency chains per thread
          {
            const uint4 oa = l_gen(0);
            const uint4 ob = l_gen(1);
            store(0, oa.x, oa.y, oa.z, oa.w);
            store(1, ob.x, ob.y, ob.z, ob.w);
          }
          if (kCPT == 3 && has3) {
            const uint4 oa = l_gen(kCPT - 1);
            store(kCPT - 1, oa.x, oa.y, oa.z, oa.w);
          }
        }
        fence_proxy_async();               // generic-proxy stores -> visible to the tensor core's async proxy
        __syncwarp();
        if (lane == 0) mbar_arrive(&tl.afull[as]);
        if (++as == (uint32_t)a.SA) { as = 0; aph ^= 1; }
      }
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

// ---------------------------------------------------------------- host side: the schedule for a shape
struct Plan { int KB, BN, NT, G, NG, nslot, slotw, SA, SB, streamed; size_t smem; };
constexpr size_t kSmemLimit = 227 * 1024 - sizeof(Tail) - 1024;

static int make_plan(const adalog_lin_fused_args* a, Plan* pl) {
  const bool i8 = a->dtype == ADALOG_I8;
  const int EL = i8 ? 128 : 64;
  const bool log = a->gen == ADALOG_GEN_LOG;
  pl->KB = (a->K + EL - 1) / EL;
  // the unit's K staged source values, and for GEN_LOG the per-candidate value LUT
  const size_t lut = ((log ? (size_t)ADALOG_P * (2 * a->n_levels + 1) : 0) + (size_t)pl->KB * EL + (size_t)pl->KB * 8) * sizeof(float);
  auto r16 = [](int v) { return ((v + 15) / 16) * 16; };
  // RESIDENT: every K block of a unit in shared memory at once, at least one spare stage, at least 2 B stages
  {
    const int nt = (a->N + 255) / 256;
    const int BN = std::min(256, std::max(16, r16((a->N + nt - 1) / nt)));
    const size_t bst = (size_t)BN * 128;
    for (int SB = 3; SB >= 2; --SB) {
      const long long room = (long long)kSmemLimit - (long long)lut - (long long)SB * (long long)bst;
      const int SA = (int)std::min<long long>(kMaxSA, room / (long long)kATile);
      if (SA >= pl->KB + 1) {
        pl->BN = BN; pl->NT = (a->N + BN - 1) / BN; pl->G = 1; pl->NG = pl->NT; pl->nslot = 2; pl->slotw = 256;
        pl->SA = std::min(SA, 2 * pl->KB); pl->SB = SB; pl->streamed = 0;
        pl->smem = 1024 + (size_t)pl->SA * kATile + (size_t)SB * bst + lut;
        return 0;
      }
    }
  }
  // STREAMED: <= 512 columns per pass, the operand regenerated per pass
  {
    const int passes = (a->N + 511) / 512;
    const int per_pass = (a->N + passes - 1) / passes;
    const int G = (per_pass + 255) / 256;
    const int BN = std::min(256, std::max(16, r16((per_pass + G - 1) / G)));
    const size_t bst = (size_t)BN * 128;
    pl->BN = BN; pl->G = G; pl->NG = passes; pl->NT = passes * G; pl->nslot = 2; pl->slotw = 256; pl->streamed = 1;
    for (int SB = 4; SB >= 2; --SB) {
      const long long room = (long long)kSmemLimit - (long long)lut - (long long)SB * (long long)bst;
      const int SA = (int)std::min<long long>(6, room / (long long)kATile);
      if (SA >= 3) {
        pl->SA = SA; pl->SB = SB;
        pl->smem = 1024 + (size_t)SA * kATile + (size_t)SB * bst + lut;
        return 0;
      }
    }
  }
  return fail(-3, "lin_fused_cand_gemm_err: the shape does not fit in shared memory");
}

static int validate(const adalog_lin_fused_args* a, bool need_partial) {
  ADALOG_REQUIRE(a && a->x && a->Bm && a->y && a->rs && a->ccs && a->ccb && a->cs, -1, "lin_fused_cand_gemm_err: null pointer");
  ADALOG_REQUIRE(a->gen == ADALOG_GEN_UNIFORM || a->gen == ADALOG_GEN_LOG, -1, "lin_fused_cand_gemm_err: bad gen");
  ADALOG_REQUIRE(a->dtype == ADALOG_BF16 || a->dtype == ADALOG_I8, -1, "lin_fused_cand_gemm_err: bad dtype");
  ADALOG_REQUIRE(a->gen == ADALOG_GEN_UNIFORM ? (a->cz != nullptr) : (a->cq && a->mtab), -1,
                 "lin_fused_cand_gemm_err: candidate arrays missing");
  ADALOG_REQUIRE(a->gen != ADALOG_GEN_LOG || (a->dtype == ADALOG_BF16 && 2 * a->n_levels <= 64), -2,
                 "lin_fused_cand_gemm_err: AdaLog candidates are bf16 operands with n_bits <= 6");
  ADALOG_REQUIRE(a->dtype != ADALOG_I8 || a->n_levels <= 64, -2, "lin_fused_cand_gemm_err: int8 operands need n_bits <= 7");
  ADALOG_REQUIRE(a->n_levels >= 1 && a->n_levels <= 128 && (a->n_levels & (a->n_levels - 1)) == 0, -2,
                 "lin_fused_cand_gemm_err: n_levels must be a power of two <= 128");
  ADALOG_REQUIRE(a->K > 0 && a->N > 0 && a->U > 0 && a->P > 0 && a->P <= ADALOG_P && a->ldx >= a->K && a->ldy >= a->N, -1,
                 "lin_fused_cand_gemm_err: bad sizes");
  ADALOG_REQUIRE((a->N & 3) == 0 && (reinterpret_cast<uintptr_t>(a->ccs) & 15) == 0, -2,
                 "lin_fused_cand_gemm_err: N must be a multiple of 4 and the column scales 16-byte aligned");
  ADALOG_REQUIRE(a->b_rows >= a->N, -1, "lin_fused_cand_gemm_err: fixed operand has fewer than N rows");
  ADALOG_REQUIRE(a->partial || !need_partial, -1, "lin_fused_cand_gemm_err: partial required");
  return 0;
}

static int grid_for(const adalog_lin_fused_args* a) { return std::min(a->U, kNumSMs); }

static int launch(const adalog_lin_fused_args* a, cudaStream_t st) {
  Plan pl;
  int rc = make_plan(a, &pl);
  if (rc) return rc;
  LArgs k;
  k.x = a->x; k.ldx = a->ldx; k.K = a->K; k.U = a->U;
  k.cs = a->cs; k.cz = a->cz; k.cq = a->cq; k.shift = a->shift; k.mtab = a->mtab; k.P = a->P; k.nl = a->n_levels;
  k.KB = pl.KB; k.N = a->N; k.BN = pl.BN; k.NT = pl.NT; k.G = pl.G; k.NG = pl.NG; k.nslot = pl.nslot; k.slotw = pl.slotw;
  k.SA = pl.SA; k.SB = pl.SB; k.streamed = pl.streamed;
  k.vec = ((a->ldx & 3) == 0 && (a->K & 3) == 0 && (reinterpret_cast<uintptr_t>(a->x) & 15) == 0) ? 1 : 0;
  k.y = a->y; k.ldy = a->ldy; k.rs = a->rs; k.ccs = a->ccs; k.ccb = a->ccb; k.partial = a->partial;
  const bool i8 = a->dtype == ADALOG_I8;
  CUtensorMap tmB;
  rc = make_map(&tmB, a->Bm, a->b_rows, (int64_t)pl.KB * (i8 ? 128 : 64), pl.BN, i8);
  if (rc) return rc;
  const unsigned grid = (unsigned)grid_for(a);
#define ADALOG_LAUNCH_LINF(GN, I8)                                                                       \
  do {                                                                                                   \
    cudaFuncSetAttribute(lin_fused_kernel<GN, I8>, cudaFuncAttributeMaxDynamicSharedMemorySize,          \
                         (int)pl.smem);                                                                  \
    lin_fused_kernel<GN, I8><<<grid, kThreads, pl.smem, st>>>(tmB, k);                                   \
  } while (0)
  if (a->gen == ADALOG_GEN_LOG) ADALOG_LAUNCH_LINF(GEN_LOG, false);
  else if (i8)                  ADALOG_LAUNCH_LINF(GEN_UNIFORM, true);
  else                          ADALOG_LAUNCH_LINF(GEN_UNIFORM, false);
#undef ADALOG_LAUNCH_LINF
  return check_launch("lin_fused_cand_gemm_err");
}

}  // namespace linf
}  // namespace adalog

extern "C" {

int adalog_lin_fused_cand_gemm_err_grid(const adalog_lin_fused_args* a) {
  int rc = adalog::linf::validate(a, false);
  if (rc) return rc;
  adalog::linf::Plan pl;
  rc = adalog::linf::make_plan(a, &pl);
  if (rc) return rc;
  return adalog::linf::grid_for(a);
}

int adalog_lin_fused_cand_gemm_err_passes(const adalog_lin_fused_args* a) {
  int rc = adalog::linf::validate(a, false);
  if (rc) return rc;
  adalog::linf::Plan pl;
  rc = adalog::linf::make_plan(a, &pl);
  if (rc) return rc;
  return pl.streamed ? pl.NG : 1;
}

int adalog_lin_fused_cand_gemm_err(const adalog_lin_fused_args* a, void* stream) {
  int rc = adalog::linf::validate(a, true);
  if (rc) return rc;
  return adalog::linf::launch(a, (cudaStream_t)stream);
}

}  // extern "C"
