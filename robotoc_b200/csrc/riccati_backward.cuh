// riccati_backward.cuh -- batched backward Riccati recursion, one CTA per OCP instance, sm_100a.
//
// Restates (as a different program) what the reference does in
//   RiccatiRecursion::backwardRiccatiRecursion                 src/riccati/riccati_recursion.cpp:32-80
//   RiccatiFactorizer::backwardRiccatiRecursion (all overloads) src/riccati/riccati_factorizer.cpp:44-197
//   BackwardRiccatiRecursionFactorizer::*                      src/riccati/backward_riccati_recursion_factorizer.cpp:31-174
//
// Design (not a translation):
//  * CTA = one OCP; the serial sweep i = N-1..0 runs inside the kernel with P_next resident in shared memory.
//  * [Fxx|Fvu|Fx|lx|lu] of a stage arrives by ONE cp.async.bulk (TMA 1-D) + mbarrier, issued as soon as the previous
//    stage stops reading the staging buffer, so the copy overlaps the tail of the stage.
//    Qxx/Qxu/Quu never touch shared memory: they are loaded straight into DMMA accumulator fragments.
//  * All dense contractions run on the fp64 tensor pipe (mma.sync m8n8k4): GEMM warp w owns the 8-row band w of every
//    product; extents that are not multiples of 8 use one pulled-back (overlapping) tile instead of padding.
//  * Warp specialisation: TX "GEMM warps" do A^T P, (A^T P) A, H; one extra "factor warp" builds
//    G = Quu + Bv^T P_vv Bv, its Cholesky L and L^-1 concurrently (r1 profile: 53 % of all stall samples were warps
//    parked at barriers behind a single-warp Cholesky + per-thread triangular solves).
//  * algebra: z = s+ - P+ Fx gives  lu' = lu - Bv^T z_v,  t1 = A^T z - lx;  with  Y = L^-1 H^T,  y = L^-1 lu':
//        P = sym(F - Y^T Y),   s = t1 + Y^T y,   K = -L^-T Y,   k = -L^-T y
//    so the critical path needs no triangular solve and no K; K, k are produced by the factor warp off the critical
//    path.  (The reference forms K = -G^-1 H^T, G K and K^T (G K).)  Rounding differs from the reference at the
//    1e-15 level; the parity tolerance is 1e-6 relative (BASELINE.json).
//  * switching-constraint (Schur) stages and STO terms follow the reference formulas with plain shared-memory loops:
//    they are 2 of 47 stages (trot) / vector-only work.
#pragma once
#include "rbt_device.cuh"
#include "../../include/rbt_layout.h"

namespace rbt {

struct BwdParams {
  rbt_layout L;
  const rbt_stage_ctrl* ctrl;  // device, [n_grid]
  int n_grid;
  int batch;
  double max_dts0;
  const double* kkt;  // [batch][n_grid][k_stride]
  double* ric;        // [batch][n_grid][r_stride]
  double* fact;       // [batch][n_grid][f_stride] or nullptr
  int* info;          // [batch]
  const int* struct_flag;  // device: 0 = every Fxx of the batch has the mechanical structure (nullptr: run unconditionally)
};

// NP = dim_passive (6: floating base, 0: fixed base).  STRUCT: the state-equation blocks have the structure every robotoc
// linearisation has (state_equation.cpp:52-55, 68-87): Fqq = I and Fqv = dt I outside their top-left NP x NP blocks.
template <int NV, int NU, int NS, int NP = 6>
struct BwdCfg {
  static constexpr int NX = 2 * NV;
  static constexpr int KR = NP + NV;  // rows of Fxx that are not structural: {0..NP-1} and {NV..2NV-1}
  static constexpr int LDF = NX + 1;  // padded row stride of the F scratch (conflict-free transpose reads)
  static constexpr int TX = num_tiles(NX);
  static constexpr int TU = num_tiles(NU);
  static constexpr int TV = num_tiles(NV);
  static constexpr int NGEMM = 32 * TX;        // threads in the GEMM warps
  static constexpr int NTHREADS = NGEMM + 32;  // + the factor warp
  // shared-memory carve-up (doubles)
  static constexpr int STAGE = NX * NX + ((NV * NU + 1) & ~1) + 2 * ((NX + 1) & ~1) + ((NU + 1) & ~1);
  static constexpr int EXTRA = ((NS * NX + 1) & ~1) + ((NS * NU + 1) & ~1) + ((NS + 1) & ~1) + 2 * ((NX + 1) & ~1) +
                               ((NU + 1) & ~1) + ((NS + 1) & ~1) + 4;
  static constexpr int o_P = 0;
  static constexpr int o_AtP = o_P + NX * NX;  // AtP (ld NX) -> [Schur: K^T] -> F scratch (ld LDF)
  static constexpr int o_In = o_AtP + ((NX * LDF + 1) & ~1);
  static constexpr int o_Ex = o_In + STAGE;
  static constexpr int o_Y = o_Ex + EXTRA;  // Y = L^-1 H^T (col-major, ld NU); Schur: G K
  static constexpr int o_H = o_Y + NU * NX;
  static constexpr int o_G = o_H + NX * NU;
  static constexpr int o_Li = o_G + NU * NU;   // L^-1 (col-major)
  static constexpr int o_Bp = o_Li + NU * NU;  // Bv^T P+_vv (row-major, ld NV)
  static constexpr int o_vec = o_Bp + ((NU * NV + 1) & ~1);
  // vectors
  static constexpr int v_sn = 0, v_z = v_sn + NX, v_t1 = v_z + NX, v_Psin = v_t1 + NX, v_Phin = v_Psin + NX,
                       v_psix = v_Phin + NX, v_phix = v_psix + NX, v_Psi = v_phix + NX, v_Phi = v_Psi + NX,
                       v_Pf = v_Phi + NX, v_Fxs = v_Pf + NX, v_lu2 = v_Fxs + NX, v_k = v_lu2 + NU, v_ylu = v_k + NU,
                       v_psiu = v_ylu + NU, v_phiu = v_psiu + NU, v_tps = v_phiu + NU, v_tph = v_tps + NU,
                       v_T = v_tph + NU, v_W = v_T + NU, v_dinv = v_W + NU, v_m = v_dinv + NU, v_mt = v_m + NS,
                       v_mtn = v_mt + NS, v_dinvS = v_mtn + NS, v_scn = v_dinvS + NS, v_sc = v_scn + 8,
                       v_end = v_sc + 8;
  static constexpr int o_bar = (o_vec + v_end + 1) & ~1;
  static constexpr int SMEM_DOUBLES = o_bar + 2;
  static constexpr size_t SMEM_BYTES = size_t(SMEM_DOUBLES) * 8;
  // Schur scratch inside the (dead) staging buffer
  static constexpr int x_Ginv = 0, x_DG = x_Ginv + NU * NU, x_S = x_DG + NS * NU, x_SDG = x_S + NS * NS,
                       x_M = x_SDG + NS * NU, x_DtM = x_M + NS * NX, x_Gc = x_DtM + NU * NX, x_end = x_Gc + NU * NU;
  static_assert(x_end <= STAGE, "Schur scratch must fit in the staging buffer");
  static_assert(NX >= 8 && NU >= 8 && NV >= 8, "DMMA tiling needs extents >= 8");
  static_assert(NX % 2 == 0 && NV % 2 == 0 && NP % 2 == 0, "nx, nv, np even (paired fragment loads)");
  static_assert(NU <= 32 && NS <= 32, "one-warp Cholesky");
};

__device__ __forceinline__ void named_bar_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int count) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory");
}

// In-place lower Cholesky of an n x n (n <= NMAX <= 32) column-major matrix in shared memory by ONE warp
// (lane = row; the row being updated lives in registers, finished columns are broadcast through shared memory).
// dinv[j] = 1 / L_jj.  Returns false on a non-positive pivot (factor then holds garbage).
template <int NMAX>
__device__ __forceinline__ bool warp_cholesky(double* A, int n, double* dinv) {
  const int lane = threadIdx.x & 31;
  double a[NMAX];
#pragma unroll
  for (int k = 0; k < NMAX; ++k) a[k] = (lane < n && k <= lane && k < n) ? A[lane + k * n] : 0.0;
  bool ok = true;
#pragma unroll
  for (int j = 0; j < NMAX; ++j) {
    if (j < n) {
      const double d = __shfl_sync(0xffffffffu, a[j], j);
      if (!(d > 0.0)) ok = false;
      const double inv = rsqrt(d);
      const double lij = (lane == j) ? d * inv : a[j] * inv;
      a[j] = lij;
      if (lane == j) dinv[j] = inv;
      if (lane >= j && lane < n) A[lane + j * n] = lij;
      __syncwarp();
#pragma unroll
      for (int k = j + 1; k < NMAX; ++k) {
        if (k < n) {
          const double lkj = A[k + j * n];  // broadcast read
          if (lane >= k) a[k] = fma(-lij, lkj, a[k]);
        }
      }
    }
  }
  return ok;
}

// b <- (L L^T)^-1 b for a strided vector in shared memory; L column-major n x n, dinv = 1/diag(L).  One thread.
__device__ __forceinline__ void chol_solve_smem(const double* Lm, const double* dinv, int n, double* b, int stride) {
  for (int i = 0; i < n; ++i) {
    double v = b[i * stride];
    for (int k = 0; k < i; ++k) v = fma(-Lm[i + k * n], b[k * stride], v);
    b[i * stride] = v * dinv[i];
  }
  for (int i = n - 1; i >= 0; --i) {
    double v = b[i * stride];
    for (int k = i + 1; k < n; ++k) v = fma(-Lm[k + i * n], b[k * stride], v);
    b[i * stride] = v * dinv[i];
  }
}

#ifndef RBT_BWD_MIN_CTAS
#define RBT_BWD_MIN_CTAS 4
#endif
template <int NV, int NU, int NS, int NP, bool STRUCT>
__global__ void __launch_bounds__(BwdCfg<NV, NU, NS, NP>::NTHREADS, RBT_BWD_MIN_CTAS) riccati_backward_kernel(const BwdParams p) {
  using C = BwdCfg<NV, NU, NS, NP>;
  constexpr int NX = C::NX, LDF = C::LDF, TX = C::TX, TU = C::TU, TV = C::TV, NTHR = C::NTHREADS, NG = C::NGEMM, KR = C::KR;
  // STRUCT launches are gated by the structure flag written by check_fxx_structure_kernel (or set by the condensing kernel,
  // which produces the structure by construction); the general instance runs when the flag says otherwise.
  if (p.struct_flag != nullptr && (*p.struct_flag == 0) != STRUCT) return;  // flag = number of violations seen (0: conforming)
  extern __shared__ __align__(16) double smem[];
  double* sP = smem + C::o_P;
  double* sAtP = smem + C::o_AtP;  // AtP row-major (ld NX); later F scratch row-major (ld LDF)
  double* sKt = sAtP;              // Schur stages only: K^T col-major (ld NX), between AtP's death and the F spill
  double* sIn = smem + C::o_In;
  double* sA = sIn;            // Fxx col-major
  double* sB = sIn + NX * NX;  // Fvu col-major (ld NV)
  double* sEx = smem + C::o_Ex;
  double* sY = smem + C::o_Y;    // Y col-major (ld NU)
  double* sH = smem + C::o_H;    // H col-major (ld NX)
  double* sG = smem + C::o_G;    // G, then its Cholesky factor
  double* sLi = smem + C::o_Li;  // L^-1 col-major (ld NU), lower triangular (upper part zero)
  double* sBp = smem + C::o_Bp;  // Bv^T P+_vv row-major (ld NV)
  double* vec = smem + C::o_vec;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::o_bar);

  const rbt_layout& L = p.L;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const bool gemm_warp = warp < TX;
  const int b = blockIdx.x;
  if (b >= p.batch) return;
  const int N = p.n_grid - 1;
  const double* kkt_b = p.kkt + size_t(b) * p.n_grid * L.k_stride;
  double* ric_b = p.ric + size_t(b) * p.n_grid * L.r_stride;
  double* fact_b = p.fact ? p.fact + size_t(b) * p.n_grid * L.f_stride : nullptr;

  const double* sFx = sIn + (L.k_Fx - L.k_Fxx);
  const double* slx = sIn + (L.k_lx - L.k_Fxx);
  const double* slu = sIn + (L.k_lu - L.k_Fxx);
  // extras (valid only on ns>0 / sto stages)
  const double* sPhix = sEx;
  const double* sPhiu = sEx + (L.k_Phiu - L.k_Phix);
  const double* sp = sEx + (L.k_p - L.k_Phix);
  const double* sfx = sEx + (L.k_fx - L.k_Phix);
  const double* shx = sEx + (L.k_hx - L.k_Phix);
  const double* shu = sEx + (L.k_hu - L.k_Phix);
  const double* sPhit = sEx + (L.k_Phit - L.k_Phix);
  const double* sksc = sEx + (L.k_sc - L.k_Phix);

  double* s_n = vec + C::v_sn;
  double* z = vec + C::v_z;
  double* t1 = vec + C::v_t1;
  double* Psin = vec + C::v_Psin;
  double* Phin = vec + C::v_Phin;
  double* psix = vec + C::v_psix;
  double* phix = vec + C::v_phix;
  double* Psi = vec + C::v_Psi;
  double* Phi = vec + C::v_Phi;
  double* Pf = vec + C::v_Pf;
  double* Fxs = vec + C::v_Fxs;  // copy of Fx (the staging buffer is reused / refilled early)
  double* lu2 = vec + C::v_lu2;
  double* kv = vec + C::v_k;
  double* ylu = vec + C::v_ylu;
  double* psiu = vec + C::v_psiu;
  double* phiu = vec + C::v_phiu;
  double* tps = vec + C::v_tps;  // L^-1 psi_u
  double* tph = vec + C::v_tph;  // L^-1 phi_u
  double* Tv = vec + C::v_T;
  double* Wv = vec + C::v_W;
  double* dinv = vec + C::v_dinv;
  double* mvec = vec + C::v_m;
  double* mt = vec + C::v_mt;
  double* mtn = vec + C::v_mtn;
  double* dinvS = vec + C::v_dinvS;
  double* scn = vec + C::v_scn;  // next-stage {xi, chi, rho, eta, iota}
  double* sc = vec + C::v_sc;

  int bad = 0;  // Cholesky failure flags (thread-local, OR-reduced at the end)

  auto issue_stage_load = [&](int st) {
    // one elected thread: stage st's [Fxx|Fvu|Fx|lx|lu] (+ extras when flagged)
    const rbt_stage_ctrl cs = p.ctrl[st];
    const double* rec = kkt_b + size_t(st) * L.k_stride;
    fence_proxy_async();
    mbar_expect_tx(&bars[0], uint32_t(L.k_stage_size) * 8u);
    tma_load_1d(sIn, rec + L.k_Fxx, uint32_t(L.k_stage_size) * 8u, &bars[0]);
    // Qxx | Qxu | Quu are read as accumulator fragments straight from global memory in phase B: pull them into L2 now
    l2_prefetch_bulk(rec + L.k_Qxx, uint32_t(L.k_core_size - L.k_stage_size) * 8u);
    if (cs.ns > 0 || cs.sto) {
      mbar_expect_tx(&bars[1], uint32_t(L.k_extra_size) * 8u);
      tma_load_1d(sEx, rec + L.k_Phix, uint32_t(L.k_extra_size) * 8u, &bars[1]);
    }
  };

  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (tid == 0 && N > 0) issue_stage_load(N - 1);

  // ---- terminal stage: P_N = Qxx_N, s_N = -lx_N          riccati_recursion.cpp:37-38
  {
    const double* recN = kkt_b + size_t(N) * L.k_stride;
    double* ricN = ric_b + size_t(N) * L.r_stride;
    for (int e = tid; e < NX * NX; e += NTHR) {
      const double v = recN[L.k_Qxx + e];
      sP[e] = v;
      ricN[L.r_P + e] = v;
    }
    for (int e = tid; e < NX; e += NTHR) {
      const double v = -recN[L.k_lx + e];
      s_n[e] = v;
      ricN[L.r_s + e] = v;
      Psin[e] = 0.0;
      Phin[e] = 0.0;
    }
    if (tid < 8) scn[tid] = 0.0;
  }
  __syncthreads();

  uint32_t par0 = 0, par1 = 0;

  for (int i = N - 1; i >= 0; --i) {
    const rbt_stage_ctrl cs = p.ctrl[i];
    const bool impact = (cs.type == RBT_IMPACT);
    const int ns = impact ? 0 : cs.ns;
    const bool sto = cs.sto != 0, sto_next = cs.sto_next != 0;
    const bool extras = (cs.ns > 0 || cs.sto);
    const bool plain = !impact && ns == 0;  // factor-warp fast path
    const double* rec = kkt_b + size_t(i) * L.k_stride;
    double* ric = ric_b + size_t(i) * L.r_stride;
    double* fct = fact_b ? fact_b + size_t(i) * L.f_stride : nullptr;

    // ---- phase transition on the in-shared "next" factorization     riccati_recursion.cpp:42-62, riccati_factorizer.cpp:145-175
    {
      bool do_pt = false;
      double* pol = nullptr;
      if (impact) {
        do_pt = (i > 0 && p.ctrl[i - 1].sto) || sto;
        pol = ric;
      } else if (p.ctrl[i + 1].type == RBT_LIFT) {
        do_pt = sto || sto_next;
        pol = ric_b + size_t(i + 1) * L.r_stride;
      }
      if (do_pt) {
        const double xi = scn[0], chi = scn[1], rho = scn[2], eta = scn[3], iota = scn[4];
        __syncthreads();
        if (sto_next) {
          double sgm = xi - 2.0 * chi + rho;
          if ((sgm * p.max_dts0) < fabs(eta - iota) || sgm < 1.4901161193847656e-08 /* sqrt(DBL_EPSILON) */)
            sgm = fabs(sgm) + fabs(eta - iota) / p.max_dts0;
          const double is = 1.0 / sgm;
          if (tid < NX) {
            const double dpp = Psin[tid] - Phin[tid];
            pol[L.r_dtsdx + tid] = -is * dpp;
            s_n[tid] += is * dpp * (eta - iota);
            Phin[tid] = Psin[tid] - is * dpp * (xi - chi);  // m.Phi = Psi - (1/sgm)(Psi-Phi)(xi-chi)
            Psin[tid] = 0.0;
          }
          if (tid == 0) {
            pol[L.r_stosc + 0] = is * (xi - chi);
            pol[L.r_stosc + 1] = -is * (eta - iota);
            scn[0] = 0.0;
            scn[1] = 0.0;
            scn[2] = xi - is * (xi - chi) * (xi - chi);
            scn[3] = 0.0;
            scn[4] = eta - is * (xi - chi) * (eta - iota);
          }
        } else {
          if (tid < NX) {
            Phin[tid] = Psin[tid];
            Psin[tid] = 0.0;
          }
          if (tid == 0) {
            scn[0] = 0.0;
            scn[1] = 0.0;
            scn[2] = xi;
            scn[3] = 0.0;
            scn[4] = eta;
          }
        }
        __syncthreads();
      }
    }

    const int i0 = tile_off(gemm_warp ? warp : 0, NX);  // this GEMM warp's row band
    double cF[TX][2];                                   // F fragments (GEMM warps only)
    double cH[TU][2];                                   // H fragments (GEMM warps only; feed Y = L^-1 H^T from registers)
    const double dtS = cs.dt;                           // structural Fqv = dt I (0 on an impact stage)
    // F = Qxx + A^T P+ A and F - Y^T Y are symmetric: band w only computes the tiles on / right of its diagonal tile and P
    // takes F[min(r,c)][max(r,c)] (every element with r <= c lies in such a tile, also under the pulled-back last band).
    // Not on switching-constraint stages: their correction K^T D^T M is symmetrised by averaging (riccati_factorizer.cpp:85-87).
    const bool symF = (ns == 0);
    const int nb0 = (symF && gemm_warp) ? warp : 0;
    // non-structural rows of Fxx: {0..NP-1} (floating-base block rows) and {NV..2NV-1} (velocity rows)
    auto rho_of = [](int k) { return k < NP ? k : k - NP + NV; };
    // STRUCT: rows NP..NV-1 of Fxx are [e_rho^T, dt e_rho^T] (structural); rows {0..NP-1} and {NV..2NV-1} are contracted
    // in full (K = KR = NP + NV), the structural rows contribute a shifted copy of the other operand.

    // factor warp: Quu -> accumulator fragments of G, issued before it parks at the Bp barrier (L2 latency off its chain)
    double cG[TU][TU][2];
    if (!gemm_warp && !impact) {
#pragma unroll
      for (int ub = 0; ub < TU; ++ub)
#pragma unroll
        for (int n = 0; n < TU; ++n) {
          const int u0 = tile_off(ub, NU), v0 = tile_off(n, NU);
          cG[ub][n][0] = __ldg(rec + L.k_Quu + (u0 + g) + (v0 + 2 * t) * NU);
          cG[ub][n][1] = __ldg(rec + L.k_Quu + (u0 + g) + (v0 + 2 * t + 1) * NU);
        }
    }

    // ---- wait for this stage's blocks
    mbar_wait(&bars[0], par0);
    par0 ^= 1;
    if (extras) {
      mbar_wait(&bars[1], par1);
      par1 ^= 1;
    }

    if (gemm_warp) {
      // ================= phase A (GEMM warps): Bp = Bv^T P+_vv (for the factor warp) ; AtP = A^T P+ ; z = s+ - P+ Fx
      if (!impact) {
        // TU*TV tiles of the NU x NV product, dealt round-robin to the GEMM warps (K = NV)
        for (int tile = warp; tile < TU * TV; tile += TX) {
          const int u0 = tile_off(tile / TV, NU), j0 = tile_off(tile % TV, NV);
          double acc[1][2] = {{0.0, 0.0}};
          warp_mma_band<NV, 1, 8, false>(
              acc, u0, [&](int u, int k) { return sB[k + u * NV]; },
              [&](int k, int jj) { return sP[(NV + k) + (NV + j0 + jj) * NX]; });
          *reinterpret_cast<double2*>(&sBp[(u0 + g) * NV + j0 + 2 * t]) = make_double2(acc[0][0], acc[0][1]);
        }
        named_bar_arrive(3, NTHR);  // Bp ready (non-blocking for the GEMM warps)
      }
      {
        double acc[TX][2];
        if constexpr (STRUCT) {
          // (A^T P+)[r][c] = sum_{rho in R} A[rho][r] P+[rho][c]  +  (structural rows NP <= rho < NV:)  P+[r][c] if NP <= r < NV,
          //                                                                                       dt P+[r-NV][c] if NV+NP <= r
          const int r = i0 + g, rr = r < NV ? r : r - NV;
          const double sc = (rr < NP) ? 0.0 : (r < NV ? 1.0 : dtS);
#pragma unroll
          for (int n = 0; n < TX; ++n) {
            const int j0 = tile_off(n, NX);
            const double2 pv = *reinterpret_cast<const double2*>(&sP[(j0 + 2 * t) + rr * NX]);  // P+ symmetric: row rr
            acc[n][0] = sc * pv.x;
            acc[n][1] = sc * pv.y;
          }
          warp_mma_band<KR, TX, NX, false>(
              acc, i0, [&](int ii, int k) { return sA[rho_of(k) + ii * NX]; }, [&](int k, int j) { return sP[rho_of(k) + j * NX]; });
        } else {
#pragma unroll
          for (int n = 0; n < TX; ++n) acc[n][0] = acc[n][1] = 0.0;
          warp_mma_band<NX, TX, NX, false>(
              acc, i0, [&](int ii, int k) { return sA[k + ii * NX]; }, [&](int k, int j) { return sP[k + j * NX]; });
        }
        // The last band is pulled back (NX = 36: rows 28..35) and recomputes rows the band before it owns: only the owner stores
        // them (the values are bit-identical, but two warps storing and loading the same words without a barrier is a data race).
        constexpr int OWN0 = 8 * (TX - 1);  // first row only the last band computes
        const bool mine = !(NX % 8 != 0 && warp == TX - 1 && i0 + g < OWN0);
#pragma unroll
        for (int n = 0; n < TX; ++n) {
          const int j0 = tile_off(n, NX);
          if (mine) *reinterpret_cast<double2*>(&sAtP[(i0 + g) * NX + j0 + 2 * t]) = make_double2(acc[n][0], acc[n][1]);
        }
      }
      // Qxx -> accumulator fragments of F: issued here so the loads fly during z, but are not live across GEMM1
#pragma unroll
      for (int n = 0; n < TX; ++n) {
        const int j0 = tile_off(n, NX);
        if (n >= nb0) {
          cF[n][0] = __ldg(rec + L.k_Qxx + (i0 + g) + (j0 + 2 * t) * NX);
          cF[n][1] = __ldg(rec + L.k_Qxx + (i0 + g) + (j0 + 2 * t + 1) * NX);
        } else {
          cF[n][0] = cF[n][1] = 0.0;
        }
      }
      if (!impact) {
#pragma unroll
        for (int n = 0; n < TU; ++n) {
          const int u0 = tile_off(n, NU);
          cH[n][0] = __ldg(rec + L.k_Qxu + (i0 + g) + (u0 + 2 * t) * NX);
          cH[n][1] = __ldg(rec + L.k_Qxu + (i0 + g) + (u0 + 2 * t + 1) * NX);
        }
      }
      matvec_N4(sP, NX, NX, NX, sFx, tid, NG, [&](int r, double a) { z[r] = s_n[r] - a; });
      if (sto) {
        if (!impact) matvec_N4(sP, NX, NX, NX, sfx, tid, NG, [&](int r, double a) { Pf[r] = a; });
        if (tid < NX) Fxs[tid] = sFx[tid];
      }
      __syncwarp();  // this warp's rows of AtP are all the next two products read of it ...
      if (NX % 8 != 0 && warp >= TX - 2) named_bar_sync(5, 64);  // ... plus, for the last band, the rows the band before it stored

      // ================= phase B (GEMM warps): F = Qxx + AtP A ; H = Qxu + AtP[:,nv:] Bv
      if constexpr (STRUCT) {
        // (AtP A)[r][c] = sum_{rho in R} AtP[r][rho] A[rho][c]  +  AtP[r][c] if NP <= c < NV,  dt AtP[r][c-NV] if NV+NP <= c
        const int r = i0 + g;
#pragma unroll
        for (int n = 0; n < TX; ++n) {
          const int c = tile_off(n, NX) + 2 * t;  // NP, NV even: the pair (c, c+1) never straddles a boundary
          const int cc = c < NV ? c : c - NV;
          if (n >= nb0) {
            const double2 av = *reinterpret_cast<const double2*>(&sAtP[r * NX + cc]);
            const double sc = (cc < NP) ? 0.0 : (c < NV ? 1.0 : dtS);
            cF[n][0] = fma(sc, av.x, cF[n][0]);
            cF[n][1] = fma(sc, av.y, cF[n][1]);
          }
        }
        warp_mma_band<KR, TX, NX, false>(
            cF, i0, [&](int ii, int k) { return sAtP[ii * NX + rho_of(k)]; }, [&](int k, int j) { return sA[rho_of(k) + j * NX]; }, nb0);
      } else {
        warp_mma_band<NX, TX, NX, false>(
            cF, i0, [&](int ii, int k) { return sAtP[ii * NX + k]; }, [&](int k, int j) { return sA[k + j * NX]; }, nb0);
      }
      if (!impact) {
        warp_mma_band<NV, TU, NU, false>(
            cH, i0, [&](int ii, int k) { return sAtP[ii * NX + NV + k]; }, [&](int k, int u) { return sB[k + u * NV]; });
        if (!plain || fct) {  // H in shared memory is only read by the switching-constraint (Schur) path
#pragma unroll
          for (int n = 0; n < TU; ++n) {
            const int u0 = tile_off(n, NU);
            if (!plain) {
              sH[(i0 + g) + (u0 + 2 * t) * NX] = cH[n][0];
              sH[(i0 + g) + (u0 + 2 * t + 1) * NX] = cH[n][1];
            }
            if (fct) {
              fct[L.f_H + (i0 + g) + (u0 + 2 * t) * NX] = cH[n][0];
              fct[L.f_H + (i0 + g) + (u0 + 2 * t + 1) * NX] = cH[n][1];
            }
          }
        }
      }
      named_bar_sync(1, NG);  // z (and, for the STO terms, every row of AtP) complete among the GEMM warps
      if (!impact) {
        // lu' = lu - Bv^T z_v      (== lu + BtP Fx - Bv^T s+_v, backward_..factorizer.cpp:43-44)
        matvec_T(sB, NV, NV, NU, z + NV, tid, NG, [&](int u, double a) {
          const double v = slu[u] - a;
          lu2[u] = v;
          if (fct) fct[L.f_lu + u] = v;
        });
      }
      matvec_T(sA, NX, NX, NX, z, tid, NG, [&](int c, double a) { t1[c] = a - slx[c]; });
      if (sto) {
        if (!impact) {
          // factorizeHamiltonian (x part): backward_riccati_recursion_factorizer.cpp:48-66; the same lane owns psix[c]
          matvec_T(sAtP, NX, NX, NX, sfx, tid, NG, [&](int c, double a) { psix[c] = a + shx[c]; });  // AtP fx + hx
          matvec_T(sA, NX, NX, NX, Psin, tid, NG, [&](int c, double a) { psix[c] += a; });
          if (sto_next) {
            matvec_T(sA, NX, NX, NX, Phin, tid, NG, [&](int c, double a) { phix[c] = a; });
          } else if (tid < NX) {
            phix[tid] = 0.0;
          }
        } else {
          // impact + sto: Phi = A^T Phi+      backward_riccati_recursion_factorizer.cpp:160-174
          matvec_T(sA, NX, NX, NX, Phin, tid, NG, [&](int c, double a) { Phi[c] = a; });
        }
      }
    } else {
      // ================= factor warp: G = Quu + (Bv^T P+_vv) Bv, then L (G = L L^T) and L^-1 in registers
      if (!impact) {
        named_bar_sync(3, NTHR);  // Bp = Bv^T P+[nv:, nv:] from the GEMM warps
#pragma unroll
        for (int ub = 0; ub < TU; ++ub) {  // G = Quu + Bp Bv
          const int u0 = tile_off(ub, NU);
          warp_mma_band<NV, TU, NU, false>(
              cG[ub], u0, [&](int u, int k) { return sBp[u * NV + k]; }, [&](int k, int v) { return sB[k + v * NV]; });
#pragma unroll
          for (int n = 0; n < TU; ++n) {
            const int v0 = tile_off(n, NU);
            sG[(u0 + g) + (v0 + 2 * t) * NU] = cG[ub][n][0];
            sG[(u0 + g) + (v0 + 2 * t + 1) * NU] = cG[ub][n][1];
            if (fct) {
              fct[L.f_G + (u0 + g) + (v0 + 2 * t) * NU] = cG[ub][n][0];
              fct[L.f_G + (u0 + g) + (v0 + 2 * t + 1) * NU] = cG[ub][n][1];
            }
          }
        }
        __syncwarp();
        if (plain) {
          // Cholesky factor (rows on lanes 0..NU-1) and its inverse (columns on lanes 16..16+NU-1), broadcasts by shuffle
          double gc[NU], rs;
          const int idx = (lane & 15) < NU ? (lane & 15) : NU - 1;
#pragma unroll
          for (int k = 0; k < NU; ++k) gc[k] = sG[idx + k * NU];  // row of G (its lower part is read)
          __syncwarp();  // every lane has read its row before any lane overwrites G with L below
          if (!warp_chol_inv_reg<NU>(gc, rs)) bad |= 1;
          if ((lane & 15) < NU) {
            if (lane < 16) {
#pragma unroll
              for (int k = 0; k < NU; ++k) sG[idx + k * NU] = (k <= idx) ? gc[k] : 0.0;  // L, col-major, lower triangular
              dinv[idx] = rs;
            } else {
#pragma unroll
              for (int k = 0; k < NU; k += 2)  // column idx of L^-1, col-major: contiguous
                *reinterpret_cast<double2*>(&sLi[k + idx * NU]) = make_double2(gc[k], gc[k + 1]);
            }
          }
          __syncwarp();
        }
      }
    }
    if (tid == 0) tma_store_wait_read();  // the previous stage's bulk store of P has long read shared memory (issued ~3 us ago)
    __syncthreads();  // ---- barrier 2: AtP/H/t1 (GEMM warps) and G = L L^T, lu' (factor warp) are complete

    // staging buffer is dead on plain stages: prefetch the next stage now (overlaps the rest of the stage)
    const bool early_prefetch = !extras;
    if (early_prefetch && tid == 0 && i > 0) issue_stage_load(i - 1);

    if (!impact) {
      if (sto) {
        // psi_u = BtP fx + hu + Bv^T Psi+_v = Bv^T (P+ fx)_v + hu + Bv^T Psi+_v ; phi_u = Bv^T Phi+_v   (:53-60)
        // and their images under L^-1 (all small; the factor warp owns them)
        if (!gemm_warp) {
          matvec_T(sB, NV, NV, NU, Pf + NV, lane, 32, [&](int u, double a) { psiu[u] = a + shu[u]; });
          matvec_T(sB, NV, NV, NU, Psin + NV, lane, 32, [&](int u, double a) { psiu[u] += a; });
          if (sto_next) {
            matvec_T(sB, NV, NV, NU, Phin + NV, lane, 32, [&](int u, double a) { phiu[u] = a; });
          } else if (lane < NU) {
            phiu[lane] = 0.0;
          }
        }
        __syncthreads();
      }
      if (plain) {
        // ================= phase C: Y = L^-1 H^T on the tensor pipe, straight from the H accumulator fragments: with the
        // contraction index u dealt to the lanes as u = u0 + 2t (+1), the C fragment of H (rows i0+g, columns u0+2t, u0+2t+1) IS
        // the B operand H^T[u][i0+g] of  Y[:, band] = L^-1 (H[band, :])^T  -- H never goes through shared memory.  The second,
        // pulled-back H tile overlaps the first in columns u0 .. 7: its A operand is zeroed there.
        if (gemm_warp) {
#pragma unroll
          for (int mt = 0; mt < TU; ++mt) {
            const int m0 = tile_off(mt, NU);
            double y0 = 0.0, y1 = 0.0;
#pragma unroll
            for (int n = 0; n < TU; ++n) {
              const int u0 = tile_off(n, NU);
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const int u = u0 + 2 * t + e;
                const bool dup = (n > 0) && (u < 8 * n);  // already contracted by the previous tile
                const double a = dup ? 0.0 : sLi[(m0 + g) + u * NU];
                dmma884(y0, y1, a, cH[n][e]);
              }
            }
            sY[(m0 + g) + (i0 + 2 * t) * NU] = y0;
            sY[(m0 + g) + (i0 + 2 * t + 1) * NU] = y1;
          }
        } else if (lane < NU) {
          // y = L^-1 lu'   (row `lane` of L^-1 is contiguous in k with stride NU)
          double a = 0.0;
#pragma unroll
          for (int k = 0; k < NU; ++k) a = fma(sLi[lane + k * NU], lu2[k], a);
          ylu[lane] = a;
        }
        __syncthreads();  // ---- barrier 3: Y complete
        // ================= phase D
        if (gemm_warp) {
          // F -= Y^T Y
          warp_mma_band<NU, TX, NX, false>(
              cF, i0, [&](int ii, int k) { return -sY[k + ii * NU]; }, [&](int k, int j) { return sY[k + j * NU]; }, nb0);
          // s = t1 + Y^T y            (== A^T z - lx - H k)
          matvec_T(sY, NU, NU, NX, ylu, tid, NG, [&](int c, double a) {
            const double v = t1[c] + a;
            s_n[c] = v;
            ric[L.r_s + c] = v;
          });
        } else {
          // K = -L^-T Y  (off the critical path) ; k = -L^-T y
#pragma unroll
          for (int ub = 0; ub < TU; ++ub) {
            const int u0 = tile_off(ub, NU);
            double acc[TX][2];
#pragma unroll
            for (int n = 0; n < TX; ++n) acc[n][0] = acc[n][1] = 0.0;
            warp_mma_band<NU, TX, NX, false>(
                acc, u0, [&](int u, int k) { return -sLi[k + u * NU]; }, [&](int k, int j) { return sY[k + j * NU]; });
#pragma unroll
            for (int n = 0; n < TX; ++n) {
              const int j0 = tile_off(n, NX);
              *reinterpret_cast<double2*>(&ric[L.r_K + (j0 + 2 * t) + (u0 + g) * NX]) = make_double2(acc[n][0], acc[n][1]);
            }
          }
          if (lane < NU) {
            double a = 0.0;
#pragma unroll
            for (int v = 0; v < NU; ++v) a = fma(sLi[v + lane * NU], ylu[v], a);
            kv[lane] = -a;
            ric[L.r_k + lane] = -a;
          }
          if (sto) {  // images of psi_u / phi_u under L^-1, then T = -L^-T (L^-1 psi_u), W likewise   riccati_factorizer.cpp:126-128
            __syncwarp();
            if (lane < NU) {
              double a = 0.0, bq = 0.0;
#pragma unroll
              for (int v = 0; v < NU; ++v) {
                a = fma(sLi[lane + v * NU], psiu[v], a);
                bq = fma(sLi[lane + v * NU], phiu[v], bq);
              }
              tps[lane] = a;
              tph[lane] = bq;
            }
            __syncwarp();
            if (lane < NU) {
              double a = 0.0, bq = 0.0;
#pragma unroll
              for (int v = 0; v < NU; ++v) {
                a = fma(sLi[v + lane * NU], tps[v], a);
                bq = fma(sLi[v + lane * NU], tph[v], bq);
              }
              Tv[lane] = -a;
              Wv[lane] = sto_next ? -bq : 0.0;
              ric[L.r_T + lane] = -a;
              ric[L.r_W + lane] = sto_next ? -bq : 0.0;
            }
          }
        }
      } else {
        // ================= Schur-complement path (switching constraint)      riccati_factorizer.cpp:58-89
        double* xs = sIn;  // scratch in the dead staging buffer
        double* Ginv = xs + C::x_Ginv;
        double* DG = xs + C::x_DG;    // ns x nu (ld ns)
        double* Sm = xs + C::x_S;     // ns x ns
        double* SDG = xs + C::x_SDG;  // ns x nu (ld ns)
        double* Mm = xs + C::x_M;     // ns x nx (ld ns)
        double* DtM = xs + C::x_DtM;  // nu x nx (ld nu)
        double* Gc = xs + C::x_Gc;    // copy of G
        for (int e = tid; e < NU * NU; e += NTHR) {
          Gc[e] = sG[e];
          Ginv[e] = ((e % NU) == (e / NU)) ? 1.0 : 0.0;
        }
        for (int e = tid; e < ns * NU; e += NTHR) DG[e] = sPhiu[e];  // DG^T <- D^T
        __syncthreads();
        if (!gemm_warp) {
          if (!warp_cholesky<NU>(sG, NU, dinv)) bad |= 1;
        }
        __syncthreads();
        if (tid < NU) chol_solve_smem(sG, dinv, NU, Ginv + tid * NU, 1);            // Ginv = G^-1             :60
        else if (tid < NU + ns) chol_solve_smem(sG, dinv, NU, DG + (tid - NU), ns);  // DGinv^T = G^-1 D^T      :61
        __syncthreads();
        for (int e = tid; e < ns * ns; e += NTHR) {  // S = DGinv D^T                                          :62
          const int r = e % ns, q = e / ns;
          double a = 0.0;
          for (int u = 0; u < NU; ++u) a = fma(DG[r + u * ns], sPhiu[q + u * ns], a);
          Sm[e] = a;
        }
        for (int e = tid; e < ns * NU; e += NTHR) SDG[e] = DG[e];
        for (int e = tid; e < ns * NX; e += NTHR) Mm[e] = sPhix[e];
        if (tid < ns) mvec[tid] = sp[tid];
        if (tid < ns) mt[tid] = sto ? sPhit[tid] : 0.0;
        __syncthreads();
        if (!gemm_warp) {
          if (!warp_cholesky<NS>(Sm, ns, dinvS)) bad |= 2;
        }
        __syncthreads();
        // SDG = S^-1 DGinv (:65);  M = S^-1 C (:71);  m = S^-1 p (:73);  mt = S^-1 Phit (:116)
        for (int c = tid; c < NU + NX + 2; c += NTHR) {
          if (c < NU) chol_solve_smem(Sm, dinvS, ns, SDG + c * ns, 1);
          else if (c < NU + NX) chol_solve_smem(Sm, dinvS, ns, Mm + (c - NU) * ns, 1);
          else if (c == NU + NX) chol_solve_smem(Sm, dinvS, ns, mvec, 1);
          else if (sto) chol_solve_smem(Sm, dinvS, ns, mt, 1);
        }
        __syncthreads();
        for (int e = tid; e < NU * NU; e += NTHR) {  // Ginv -= SDG^T DGinv                                    :66
          const int a = e % NU, c = e / NU;
          double acc = 0.0;
          for (int r = 0; r < ns; ++r) acc = fma(SDG[r + a * ns], DG[r + c * ns], acc);
          Ginv[e] -= acc;
        }
        __syncthreads();
        // K = -Ginv H^T - SDG^T C (:67-68);  M -= SDG H^T (:72)       (AtP is dead: K^T lives in its buffer)
        for (int e = tid; e < NU * NX; e += NTHR) {
          const int j = e % NX, u = e / NX;
          double a = 0.0;
          for (int v = 0; v < NU; ++v) a = fma(Ginv[u + v * NU], sH[j + v * NX], a);
          for (int r = 0; r < ns; ++r) a = fma(SDG[r + u * ns], sPhix[r + j * ns], a);
          sKt[j + u * NX] = -a;
          ric[L.r_K + j + u * NX] = -a;
        }
        for (int e = tid; e < ns * NX; e += NTHR) {
          const int r = e % ns, j = e / ns;
          double a = 0.0;
          for (int u = 0; u < NU; ++u) a = fma(SDG[r + u * ns], sH[j + u * NX], a);
          Mm[e] -= a;
        }
        if (tid < NU) {  // k = -Ginv lu' - SDG^T p (:69-70); T, W (:111-114)
          const int u = tid;
          double a = 0.0, tt = 0.0, ww = 0.0;
          for (int v = 0; v < NU; ++v) {
            a = fma(Ginv[u + v * NU], lu2[v], a);
            if (sto) tt = fma(Ginv[u + v * NU], psiu[v], tt);
            if (sto && sto_next) ww = fma(Ginv[u + v * NU], phiu[v], ww);
          }
          for (int r = 0; r < ns; ++r) {
            a = fma(SDG[r + u * ns], sp[r], a);
            if (sto) tt = fma(SDG[r + u * ns], sPhit[r], tt);
          }
          kv[u] = -a;
          ric[L.r_k + u] = -a;
          if (sto) {
            Tv[u] = -tt;
            Wv[u] = -ww;
            ric[L.r_T + u] = -tt;
            ric[L.r_W + u] = -ww;
          }
        } else if (tid >= 32 && tid < 32 + ns) {  // m -= SDG lu' (:74); mt -= SDG psi_u (:117); mt_next = -SDG phi_u (:119)
          const int r = tid - 32;
          double a = 0.0, bq = 0.0, cq = 0.0;
          for (int u = 0; u < NU; ++u) {
            a = fma(SDG[r + u * ns], lu2[u], a);
            if (sto) bq = fma(SDG[r + u * ns], psiu[u], bq);
            if (sto && sto_next) cq = fma(SDG[r + u * ns], phiu[u], cq);
          }
          mvec[r] -= a;
          if (sto) {
            mt[r] -= bq;
            mtn[r] = -cq;
          }
        }
        __syncthreads();
        // outputs M, m (+ mt, mt_next);  GK = G K (:82) -> sY;  DtM = D^T M (:84)
        for (int e = tid; e < ns * NX; e += NTHR) ric[L.r_M + e] = Mm[e];
        if (tid < ns) {
          ric[L.r_m + tid] = mvec[tid];
          if (sto) {
            ric[L.r_mt + tid] = mt[tid];
            ric[L.r_mtn + tid] = mtn[tid];
          }
        }
        for (int e = tid; e < NU * NX; e += NTHR) {
          const int u = e % NU, j = e / NU;
          double a = 0.0, d2 = 0.0;
          for (int v = 0; v < NU; ++v) a = fma(Gc[u + v * NU], sKt[j + v * NX], a);
          for (int r = 0; r < ns; ++r) d2 = fma(sPhiu[r + u * ns], Mm[r + j * ns], d2);
          sY[e] = a;
          DtM[e] = d2;
        }
        // s = t1 - H k - C^T m           backward_..factorizer.cpp:87-90, riccati_factorizer.cpp:88
        if (tid >= NG - NX && tid < NG) {
          const int r = tid - (NG - NX);
          double v = t1[r];
          for (int u = 0; u < NU; ++u) v = fma(-sH[r + u * NX], kv[u], v);
          for (int q = 0; q < ns; ++q) v = fma(-sPhix[q + r * ns], mvec[q], v);
          s_n[r] = v;
          ric[L.r_s + r] = v;
        }
        __syncthreads();
        if (gemm_warp) {
          // F -= K^T (G K)                                                                   backward_..factorizer.cpp:83
          warp_mma_band<NU, TX, NX, false>(
              cF, i0, [&](int ii, int k) { return -sKt[ii + k * NX]; }, [&](int k, int j) { return sY[k + j * NU]; });
          if (fct) {  // the reference leaves Qxx = F - K^T G K here; spill it before the constraint correction
#pragma unroll
            for (int n = 0; n < TX; ++n) {
              const int j0 = tile_off(n, NX);
              fct[L.f_F + (i0 + g) + (j0 + 2 * t) * NX] = cF[n][0];
              fct[L.f_F + (i0 + g) + (j0 + 2 * t + 1) * NX] = cF[n][1];
            }
          }
          // P = sym(F) - KtDtM - KtDtM^T = sym(F - 2 K^T DtM)                                 riccati_factorizer.cpp:85-87
          warp_mma_band<NU, TX, NX, false>(
              cF, i0, [&](int ii, int k) { return -2.0 * sKt[ii + k * NX]; }, [&](int k, int j) { return DtM[k + j * NU]; });
        }
        if (sto) {
          // Psi = psi_x + K^T psi_u + M^T Phit ; Phi = phi_x + K^T phi_u   (K^T still valid in the AtP buffer)
          if (!gemm_warp) {
            for (int c = lane; c < NX; c += 32) {
              double a = psix[c], bq = sto_next ? phix[c] : 0.0;
              for (int u = 0; u < NU; ++u) {
                a = fma(sKt[c + u * NX], psiu[u], a);
                if (sto_next) bq = fma(sKt[c + u * NX], phiu[u], bq);
              }
              for (int q = 0; q < ns; ++q) a = fma(Mm[q + c * ns], sPhit[q], a);
              Psi[c] = a;
              Phi[c] = bq;
            }
          }
        }
        __syncthreads();  // all reads of K^T (AtP buffer) are done before F is spilled into it
      }
    }
    if (impact && tid < NX) {
      s_n[tid] = t1[tid];  // s = A^T z - lx
      ric[L.r_s + tid] = t1[tid];
    }

    // ================= P = F - Y^T Y.  Symmetric stages (no switching constraint, no factorized-KKT output): the accumulator
    // fragments with r <= c go straight to BOTH mirror positions of the next stage's P in shared memory (P+ is dead: its last
    // readers were the phase A / B products, two barriers ago), and P leaves for HBM as ONE bulk shared -> global copy after
    // the barrier.  (The element-wise symmetrise-and-store loop this replaces was 16 % of the sweep's instructions.)
    const bool fastP = symF && fct == nullptr;
    if (gemm_warp) {
      // rows the pulled-back last band shares with the band before it are stored by their owner only (identical values)
      const bool mine = !(NX % 8 != 0 && warp == TX - 1 && i0 + g < 8 * (TX - 1));
#pragma unroll
      for (int n = 0; n < TX; ++n) {
        const int j0 = tile_off(n, NX);
        if (n >= nb0 && mine) {
          if (fastP) {
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const int r = i0 + g, c = j0 + 2 * t + q;
              if (r <= c) {
                sP[r + c * NX] = cF[n][q];
                sP[c + r * NX] = cF[n][q];
              }
            }
          } else {  // spill F (row-major, ld LDF)
            sAtP[(i0 + g) * LDF + j0 + 2 * t] = cF[n][0];
            sAtP[(i0 + g) * LDF + j0 + 2 * t + 1] = cF[n][1];
          }
        }
      }
    }
    __syncthreads();  // ---- barrier 4: P (or the F scratch), s, k complete

    if (fastP) {
      if (tid == 0) {
        tma_store_fence();
        tma_store_1d(ric + L.r_P, sP, uint32_t(NX * NX) * 8u);
        tma_store_commit();
      }
    } else {  // ================= phase E: P = (F + F^T)/2 -> shared (next stage) and HBM
      int r = tid % NX, c = tid / NX;  // (r, c) of e = tid + k * NTHR, advanced without a division per element
      for (int e = tid; e < NX * NX; e += NTHR) {
        double v, f_rc;
        if (symF) {  // only the tiles on / above the diagonal were computed: mirror
          v = f_rc = (r <= c) ? sAtP[r * LDF + c] : sAtP[c * LDF + r];
        } else {
          f_rc = sAtP[r * LDF + c];
          v = 0.5 * (f_rc + sAtP[c * LDF + r]);
        }
        sP[e] = v;
        ric[L.r_P + e] = v;
        if (fct && ns == 0) fct[L.f_F + e] = f_rc;
        r += NTHR % NX;
        c += NTHR / NX;
        if (r >= NX) {
          r -= NX;
          ++c;
        }
      }
    }
    if (sto) {
      if (!impact) {
        // factorizeSTOFactorization: backward_riccati_recursion_factorizer.cpp:94-143 (+ riccati_factorizer.cpp:136-141)
        if (plain) {
          // Psi = psi_x + K^T psi_u = psi_x - Y^T (L^-1 psi_u) ; Phi likewise
          matvec_T(sY, NU, NU, NX, tps, tid, NTHR, [&](int c, double a) { Psi[c] = psix[c] - a; });
          if (sto_next) {
            matvec_T(sY, NU, NU, NX, tph, tid, NTHR, [&](int c, double a) { Phi[c] = phix[c] - a; });
          } else if (tid < NX) {
            Phi[tid] = 0.0;
          }
        }
        if (tid == NTHR - 1) {
          double xi = dot_serial(sfx, Pf, NX) + sksc[0] + 2.0 * dot_serial(Psin, sfx, NX) + dot_serial(Tv, psiu, NU) + scn[0];
          double chi = 0.0, rho = 0.0, iota = 0.0;
          if (sto_next) {
            chi = sksc[1] + dot_serial(Phin, sfx, NX) + dot_serial(Tv, phiu, NU) + scn[1];
            rho = dot_serial(Wv, phiu, NU) + scn[2];
          }
          // Pf2 = P+ Fx - s+ = -z
          double eta = -dot_serial(sfx, z, NX) + sksc[2] + dot_serial(Psin, Fxs, NX) + dot_serial(psiu, kv, NU) + scn[3];
          if (sto_next) iota = dot_serial(Phin, Fxs, NX) + dot_serial(phiu, kv, NU) + scn[4];
          if (ns > 0) {
            xi += dot_serial(mt, sPhit, ns);
            if (sto_next) chi += dot_serial(mtn, sPhit, ns);
            eta += dot_serial(mvec, sPhit, ns);
          }
          sc[0] = xi; sc[1] = chi; sc[2] = rho; sc[3] = eta; sc[4] = iota;
        }
      } else {
        if (tid == NTHR - 1) {
          sc[0] = 0.0; sc[1] = 0.0; sc[2] = scn[2]; sc[3] = 0.0;
          sc[4] = scn[4] + dot_serial(Phin, Fxs, NX);
        }
        if (tid < NX) Psi[tid] = 0.0;
      }
      __syncthreads();
      if (tid < NX) {
        Psin[tid] = Psi[tid];
        Phin[tid] = Phi[tid];
        ric[L.r_Psi + tid] = Psi[tid];
        ric[L.r_Phi + tid] = Phi[tid];
        if (!impact) {
          ric[L.r_psix + tid] = psix[tid];
          ric[L.r_phix + tid] = phix[tid];
        }
      }
      if (!impact && tid < NU) {
        ric[L.r_psiu + tid] = psiu[tid];
        ric[L.r_phiu + tid] = phiu[tid];
      }
      if (tid < 5) {
        scn[tid] = sc[tid];
        ric[L.r_sc + tid] = sc[tid];
      }
    } else {
      // !sto: Psi = 0, xi = chi = eta = 0 (riccati_factorizer.cpp:99-105); Phi, rho, iota keep their constructor zeros
      if (tid < NX) {
        Psin[tid] = 0.0;
        Phin[tid] = 0.0;
      }
      if (tid < 8) scn[tid] = 0.0;
    }
    __syncthreads();  // ---- barrier 5: P+ / s+ / STO state rolled
    if (!early_prefetch && tid == 0 && i > 0) issue_stage_load(i - 1);
  }

  if (tid == 0) tma_store_wait_read();  // the last bulk store of P must have read shared memory before the CTA retires
  // ---- final phase transition at stage 0                       riccati_recursion.cpp:75-79
  {
    const rbt_stage_ctrl c0 = p.ctrl[0];
    if (c0.sto && c0.sto_next && N > 0) {
      const double xi = scn[0], chi = scn[1], rho = scn[2], eta = scn[3], iota = scn[4];
      double sgm = xi - 2.0 * chi + rho;
      if ((sgm * p.max_dts0) < fabs(eta - iota) || sgm < 1.4901161193847656e-08) sgm = fabs(sgm) + fabs(eta - iota) / p.max_dts0;
      const double is = 1.0 / sgm;
      if (tid < NX) ric_b[L.r_dtsdx + tid] = -is * (Psin[tid] - Phin[tid]);
      if (tid == 0) {
        ric_b[L.r_stosc + 0] = is * (xi - chi);
        ric_b[L.r_stosc + 1] = -is * (eta - iota);
      }
    }
  }
  bad = __reduce_or_sync(0xffffffffu, bad);
  if (lane == 0 && bad) atomicOr(&p.info[b], bad);
}

// One warp per (OCP, stage < N): *viol = 1 if Fxx deviates from [[I, dt I], [*, *]] outside the top-left NP x NP blocks of
// Fqq and Fqv (rows NP..NV-1 entirely, rows < NP outside the two blocks).  Reads 18 of the 36 rows of every Fxx once.
template <int NV, int NP>
__global__ void check_fxx_structure_kernel(const BwdParams p, int* viol) {
  constexpr int NX = 2 * NV;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int N = p.n_grid - 1;
  if (w >= p.batch * N) return;
  const int b = w / N, i = w % N;
  const double dt = p.ctrl[i].dt;
  const double* A = p.kkt + (size_t(b) * p.n_grid + i) * p.L.k_stride + p.L.k_Fxx;
  bool bad = false;
  for (int e = lane; e < NV * NX; e += 32) {
    const int rho = e % NV, c = e / NV;
    if (rho < NP && (c < NP || (c >= NV && c < NV + NP))) continue;  // the floating-base blocks are free
    const double want = (c == rho) ? 1.0 : ((c == rho + NV) ? dt : 0.0);
    bad |= !(A[rho + c * NX] == want);
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicExch(viol, 1);
}

}  // namespace rbt
