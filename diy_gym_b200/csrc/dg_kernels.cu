// dg_kernels.cu - sm_100a kernels and the C ABI (include/diygym_b200.h) of the batched DIYGym backend.
//
// dg_step_kernel<T>: persistent grid; a block holds blockDim/T teams of T lanes, each team advances one
// environment at a time with its whole working set (dg_scene.h workspace plan) in dynamic shared memory, and
// walks the environment list with a grid stride.  Scene constants are read-only global arrays shared by all
// environments (L1/L2 resident).  State rows are [env][S] so that a team's loads and stores are contiguous.
// dg_render_kernel: one block per environment (or per group of its pixel tiles when the batch is small); visual shapes
// are staged in shared memory once per block, every tile is culled against them and every thread ray-casts its pixels
// (camera.py:58-92 of the reference, TinyRenderer replaced).
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/diygym_b200.h"
#include "dg_env.cuh"
#include "dg_ray.cuh"
#include "dg_dyn.cuh"
#include "dg_ik.cuh"

namespace dg {

struct LaunchArgs {
  float* state; float* param; const float* act; float* obs; float* rew; uint8_t* term;
  const uint8_t* mask; int n_envs; int mode; uint32_t seed; int env_off;
  unsigned long long opmask[2];
  float* gws;   // cold workspace: one slot of sc.g_total floats per resident team
  unsigned long long* dbg;   // phase-timing table or null (dg_debug_phase_cycles)
  unsigned* dropped;         // contacts lost to the max_contacts cap (one counter per world)
  // split schedule (mode 0 only): which stages of the step this launch runs (ST_*), the per-environment carry of the hot
  // workspace between launches, and the lists of environments left to the sweep kernel
  int stages; float* carry; int* rs_lists; int* rs_count; unsigned* rs_used; int no_hot;   // rs_lists: [RS_NCLS][n_envs]
};

template <int T>
__global__ void __launch_bounds__(256) dg_step_kernel(const __grid_constant__ DevScene sc, const LaunchArgs a) {
  extern __shared__ __align__(16) float smem[];
  // thread t = lane (t / E) of the block's environment (t % E): a warp holds one lane index of 32 environments
  const int E = blockDim.x / T;
  const int ei = threadIdx.x % E, ln = threadIdx.x / E;
  Env C;
  // the block's copy of the link tables sits behind the per-environment workspaces
  int* s_link_i = reinterpret_cast<int*>(smem + (size_t)E * sc.w_total);
  float* s_link_f = reinterpret_cast<float*>(s_link_i + ((DG_LINK_I_W * sc.nl + 3) & ~3));
  float* s_link_x = s_link_f + DG_LINK_F_W * sc.nl;
  for (int i = threadIdx.x; i < DG_LINK_I_W * sc.nl; i += blockDim.x) s_link_i[i] = sc.link_i[i];
  for (int i = threadIdx.x; i < DG_LINK_F_W * sc.nl; i += blockDim.x) s_link_f[i] = sc.link_f[i];
  for (int i = threadIdx.x; i < 16 * sc.nl; i += blockDim.x) s_link_x[i] = sc.link_x[i];
  __syncthreads();
  C.link_i = s_link_i; C.link_f = s_link_f; C.link_x = s_link_x;
  C.sc = &sc; C.ws = smem + (size_t)ei * sc.w_total; C.seed = a.seed;
  C.opmask[0] = a.opmask[0]; C.opmask[1] = a.opmask[1]; C.dbg = a.dbg; C.dropped = a.dropped;
  C.split = a.stages != ST_ALL ? 1 : 0; C.rs_lists = a.rs_lists; C.rs_stride = a.n_envs; C.rs_count = a.rs_count; C.rs_used = a.rs_used; C.no_hot = a.no_hot;
  { // environments that share a warp once the row-space sweeps remap the threads (thread t -> lane t % T of environment t / T)
    const int G = T >= 32 ? 1 : 32 / T, g0 = ei / G * G;
    C.grp0 = g0 - ei; C.grp1 = (g0 + G < E ? g0 + G : E) - ei;
  }
  // block-uniform trip count: every thread of the block walks the same number of environment groups
  for (int base = blockIdx.x * E; base < a.n_envs; base += gridDim.x * E) {
    const int e = base + ei;
    C.active = e < a.n_envs && (a.mask == nullptr || a.mask[e] != 0);
    const int ec = e < a.n_envs ? e : a.n_envs - 1;
    C.st = a.state + (size_t)ec * sc.S; C.pr = a.param + (size_t)ec * sc.P;
    C.act = a.act + (size_t)ec * sc.n_act; C.obs = a.obs + (size_t)ec * sc.n_obs; C.rew = a.rew + (size_t)ec * sc.n_rew;
    C.term = a.term + (size_t)ec * sc.n_term; C.env_id = a.env_off + ec; C.e_local = ec;
    C.wg = a.gws + (size_t)e * sc.g_total;   // the cold workspace is per environment (the allocation has slack for the tail slots)
    // masked launches (reset of finished episodes, issued every step without a host round trip): nothing to do for a block
    // whose environments are all unmasked
    if (a.mask != nullptr && !__syncthreads_or(C.active ? 1 : 0)) continue;
    // the hot workspaces of the block's environments are one contiguous piece of shared memory, their carry rows one
    // contiguous piece of global memory: copied by the whole block, 128 bits per thread
    const int ncarry = (a.n_envs - base < E ? a.n_envs - base : E) * sc.w_total;
    if (a.stages & ST_LOADC) {
      const float4* src = reinterpret_cast<const float4*>(a.carry + (size_t)base * sc.w_total); float4* dst = reinterpret_cast<float4*>(smem);
      for (int i = threadIdx.x; i < ncarry / 4; i += blockDim.x) dst[i] = src[i];
      __syncthreads();
    }
    if (a.stages != ST_ALL) run_env_step_stages(C, T, a.stages, ln);
    else if (a.mode == 0) run_env_step(C, T, ln); else if (a.mode == 1) run_env_reset(C, T, ln); else run_env_observe(C, T, ln);
    if (T > 1 || (a.stages & ST_SAVEC)) __syncthreads();
    if (a.stages & ST_SAVEC) {
      float4* dst = reinterpret_cast<float4*>(a.carry + (size_t)base * sc.w_total); const float4* src = reinterpret_cast<const float4*>(smem);
      for (int i = threadIdx.x; i < ncarry / 4; i += blockDim.x) dst[i] = src[i];
      __syncthreads();
    }
  }
}

// Build layout: this file is compiled once per team size with -DDG_STEP_T=<T> (that object holds only dg_step_kernel<T>
// and its two host wrappers) and once without (everything else); diy_gym_b200/build.py runs the compilations in
// parallel and links the objects into one library.
struct StepLaunch { int grid, block; size_t smem; cudaStream_t stream; };
template <int T> static cudaError_t step_configure_t(int block_threads, size_t smem, size_t smem_cap, int* occ) {
  // the attribute is per function, not per world: always allow the device maximum so that worlds of different sizes coexist
  cudaError_t e = cudaFuncSetAttribute(dg_step_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap);
  if (e != cudaSuccess) return e;
  // DG_CARVEOUT=<percent of the SM's shared memory>: preferred carve-out of the step kernel (the rest is L1); measurement aid
  if (const char* cv = getenv("DG_CARVEOUT")) {
    e = cudaFuncSetAttribute(dg_step_kernel<T>, cudaFuncAttributePreferredSharedMemoryCarveout, atoi(cv));
    if (e != cudaSuccess) return e;
  }
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, dg_step_kernel<T>, block_threads, smem);
}
template <int T> static cudaError_t step_launch_t(const DevScene& sc, const LaunchArgs& a, const StepLaunch& l) {
  dg_step_kernel<T><<<l.grid, l.block, l.smem, l.stream>>>(sc, a);
  return cudaGetLastError();
}
#define DG_DECLARE_STEP(T)                                                                              \
  cudaError_t dg_step_configure_##T(int block_threads, size_t smem, size_t smem_cap, int* occ);          \
  cudaError_t dg_step_launch_##T(const DevScene& sc, const LaunchArgs& a, const StepLaunch& l);
#define DG_DEFINE_STEP(T)                                                                               \
  cudaError_t dg_step_configure_##T(int block_threads, size_t smem, size_t smem_cap, int* occ) { return step_configure_t<T>(block_threads, smem, smem_cap, occ); } \
  cudaError_t dg_step_launch_##T(const DevScene& sc, const LaunchArgs& a, const StepLaunch& l) { return step_launch_t<T>(sc, a, l); }
DG_DECLARE_STEP(1) DG_DECLARE_STEP(2) DG_DECLARE_STEP(4) DG_DECLARE_STEP(8) DG_DECLARE_STEP(16) DG_DECLARE_STEP(32)
#if defined(DG_STEP_T)
#define DG_DEFINE_STEP_X(T) DG_DEFINE_STEP(T)
DG_DEFINE_STEP_X(DG_STEP_T)
#elif !defined(DG_SPLIT_BUILD)
#error "compile with -DDG_STEP_T=<team size> (one object per team size) or -DDG_SPLIT_BUILD (everything else): see diy_gym_b200/build.py"
#endif

#if !defined(DG_STEP_T)
// The contact sweeps of the environments a stage launch deferred: dg_solve_kernel<W, K>, one warp per block, W lanes per
// environment (32 / W environments per warp), lane l owns the K CONSECUTIVE positions K l .. K l + K - 1 of the padded layout
// (dg_env.cuh "row-space team solver") - classes 8 x 4 (<= 32 positions), 16 x 3 (<= 48), 32 x 2 (<= 64).  A lane holds, in
// registers, the right-hand sides, clamps and accumulated impulses of its rows and its K columns of A for EVERY row: the 150 sweeps
// of a sub-step touch no memory.  One step = the K rows of lane j: every lane evaluates the clamp of its first slot, the owner's
// change is broadcast by a shuffle; the owner folds it into its next row at once (its own registers), evaluates that clamp,
// broadcasts, ...; then every lane folds the K broadcasts into its K rows.  Only one update in K waits for a shuffle.
// Row order, clamps and friction bounds are those of the in-kernel team sweeps and of the oracle.  The environments of a warp run
// one instruction stream: their sections are laid out at common offsets (the largest of the section sizes; surplus positions are
// inert padding); if that common layout does not fit, the warp sweeps its environments one after the other.  Everything that
// steers the loops is read through block-uniform addresses, so the loop branches stay uniform (no divergence bookkeeping around
// the shuffles).
struct SolveArgs { float* carry; float* gws; const int* list; const int* count; };
template <int W, int K>
__global__ void __launch_bounds__(32, (K == 2 ? (W == 16 ? 16 : 12) : 8)) dg_solve_kernel(const __grid_constant__ DevScene sc, const SolveArgs a) {
  constexpr int G = 32 / W, RMAX = W * K;
  constexpr unsigned FULL = 0xffffffffu;
  const int count = *a.count, first = (int)blockIdx.x * G;
  if (first >= count) return;
  const int lane = threadIdx.x, half = lane / W, l = lane % W;
  // layouts of the environments of this warp (every lane reads all of them: uniform)
  RsLayout Ls[G]; int es[G];
  int P1w = 0, N2w = 0, N3w = 0;   // common section sizes
#pragma unroll
  for (int g = 0; g < G; g++) {
    es[g] = a.list[first + g < count ? first + g : first];
    const int* hdr = reinterpret_cast<const int*>(a.carry + (size_t)es[g] * sc.w_total) + sc.W_HDR;
    Ls[g] = rs_layout(K, hdr[WH_RS_NU], 6 * sc.ncons, hdr[WH_NCROW] / 3);
    if (first + g >= count) Ls[g] = rs_layout(K, 0, 0, 0);
    P1w = max(P1w, Ls[g].P1); N2w = max(N2w, Ls[g].P2 - Ls[g].P1); N3w = max(N3w, Ls[g].Rp - Ls[g].P2);
  }
  const bool together = P1w + N2w + N3w <= RMAX;   // else: one environment at a time, every group of the warp on the same one
  const int npass = (G > 1 && !together) ? G : 1;
  for (int pass = 0; pass < npass; pass++) {
    const int mine = npass > 1 ? pass : half;                       // which environment this lane works on
    const bool writer = npass > 1 ? half == 0 : true;               // (duplicated work: one group writes back)
    RsLayout L = Ls[0];
#pragma unroll
    for (int g = 1; g < G; g++) if (mine == g) L = Ls[g];
    // loop bounds from block-uniform values only (the layout of environment `pass`, not `mine`: the compiler must see that they are uniform)
    RsLayout Lu = Ls[0];
#pragma unroll
    for (int g = 1; g < G; g++) if (pass == g) Lu = Ls[g];
    const int P1 = npass > 1 ? Lu.P1 : P1w, P2 = P1 + (npass > 1 ? Lu.P2 - Lu.P1 : N2w), Rp = P2 + (npass > 1 ? Lu.Rp - Lu.P2 : N3w);
    const bool live = first + mine < count;
    int emine = es[0];
#pragma unroll
    for (int g = 1; g < G; g++) if (mine == g) emine = es[g];
    float* wg = a.gws + (size_t)emine * sc.g_total;
    float* REC = wg + sc.X_RSREC; float* A = wg + sc.X_RSA; const int cap = sc.rs_cap;
    // A[p][s] = J_s . (M^-1 J^T)_p, built HERE by the environment's W lanes (the stage launch leaves the dense row vectors of
    // phase_rs_setup in the cold workspace and skips phase_rs_build for deferred environments): lane per column s, only over the
    // support of J_s, the same four partial sums as phase_rs_build.  Rolled loops: the update sequence below is what must stay in
    // the instruction cache.
    {
      const int GV = sc.GV; const float* RSV = wg + sc.X_RSV;
#pragma unroll 1
      for (int s2 = l; s2 < L.Rp; s2 += W) {
        const bool rs2 = live && rs_real(L, s2);
        int c0 = 0, c1 = 0;
        if (rs2) { const int sup = float_as_int(REC[RR_W * s2 + RR_APPLIED]); c0 = sup & 0xffff; c1 = (sup >> 16) & 0xffff; if (c1 > GV) c1 = GV; }
        const float* Jd = RSV + (size_t)s2 * 2 * GV;
#pragma unroll 1
        for (int p = 0; p < L.Rp; p++) {
          float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
          if (rs2 && rs_real(L, p)) {
            const float* Md = RSV + (size_t)p * 2 * GV + GV;
#pragma unroll 2
            for (int c = c0; c < c1; c += 4) { const F4 jv = ld4(Jd + c), mv = ld4(Md + c); a0 = fmaf(jv.x, mv.x, a0); a1 = fmaf(jv.y, mv.y, a1); a2 = fmaf(jv.z, mv.z, a2); a3 = fmaf(jv.w, mv.w, a3); }
          }
          if (live) A[p * cap + s2] = (a0 + a1) + (a2 + a3);
        }
      }
      __syncwarp();
    }
    // warp position g -> position q in the environment's own layout (-1: padding)
    auto own_pos = [&](int g) {
      int q;
      if (g < P1) q = g < L.P1 ? g : -1;
      else if (g < P2) { q = L.P1 + (g - P1); q = q < L.P2 ? q : -1; }
      else { q = L.P2 + (g - P2); q = q < L.Rp ? q : -1; }
      return live ? q : -1;
    };
    // Per owned row the lane carries  v = rhs - dinv y  (the unclamped change of the impulse),  lo' = lo - ap, hi' = hi - ap, so that
    // one update is  d = min(max(v, lo'), hi')  - two dependent instructions - and folding a broadcast change d_p of row p is
    // v += g[p] d_p  with  g[p][r] = -dinv_r A[p][r]  (for r = p that is -1 up to rounding: the row's own change leaves v - d).
    // Mathematically the update of the team sweeps / the oracle  (ap' = clamp(ap + rhs - dinv y), d = ap' - ap);  only the
    // rounding differs.  lo', hi' are re-derived from the exact bounds once per section (no drift).
    float dinv[K], lo[K], hi[K], ap[K], v[K], lop[K], hip[K], mu[K]; int par[K], qown[K];
#pragma unroll
    for (int k = 0; k < K; k++) {
      v[k] = 0.f; dinv[k] = 0.f; lo[k] = 0.f; hi[k] = 0.f; ap[k] = 0.f; mu[k] = 0.f; par[k] = -1;
      const int q = own_pos(l * K + k); qown[k] = q;
      if (q >= 0) { const F4 r0 = ld4(REC + RR_W * q), r1 = ld4(REC + RR_W * q + 4); v[k] = r0.x; dinv[k] = r0.y; lo[k] = r0.z; hi[k] = r0.w; mu[k] = r1.x; par[k] = float_as_int(r1.y); }
      lop[k] = lo[k]; hip[k] = hi[k];   // ap = 0, y = 0 at the start
    }
    // The owner only CAPTURES its changes in the update sequence (chg); impulses and shifted bounds are brought up to date once
    // per section (DG_SETTLE) - a row is updated once per section, and nobody else reads them in between.
    float chg[K];
#pragma unroll
    for (int k = 0; k < K; k++) chg[k] = 0.f;
#define DG_SETTLE { _Pragma("unroll") for (int k = 0; k < K; k++) { ap[k] += chg[k]; chg[k] = 0.f; lop[k] = lo[k] - ap[k]; hip[k] = hi[k] - ap[k]; } }
    float g_[RMAX][K];   // g_[p][k] = -dinv[k] A[row at warp position p][this lane's slot k]
#pragma unroll
    for (int p = 0; p < RMAX; p++) {
      const int q = p < Rp ? own_pos(p) : -1;
#pragma unroll
      for (int k = 0; k < K; k++) g_[p][k] = (q >= 0 && qown[k] >= 0) ? -dinv[k] * A[q * cap + qown[k]] : 0.f;
    }
    const int nrm0 = P1 + 6 * sc.ncons;   // warp position of the normal row of contact 0
    // rows K j .. K j + K - 1 (lane j of each environment), ascending (FWD) or descending.  The owner folds its earlier changes into
    // its next row at once; the broadcast values are bit-identical to its own changes, so the folds at the end give it the same v.
#define DG_STEPK(j, FWD)                                                                                                      \
    {                                                                                                                           \
      float d_[K], b_[K];                                                                                                       \
      _Pragma("unroll") for (int t_ = 0; t_ < K; t_++) {                                                                        \
        const int k_ = (FWD) ? t_ : K - 1 - t_;                                                                                 \
        float vf_ = v[k_];                                                                                                      \
        _Pragma("unroll") for (int u_ = 0; u_ < t_; u_++) { const int ku_ = (FWD) ? u_ : K - 1 - u_; vf_ = fmaf(g_[K * (j) + ku_][k_], d_[ku_], vf_); } \
        d_[k_] = fminf(fmaxf(vf_, lop[k_]), hip[k_]);                                                                           \
        b_[k_] = __shfl_sync(FULL, d_[k_], (j), W);                                                                             \
        chg[k_] = (l == (j)) ? d_[k_] : chg[k_];                                                                                \
      }                                                                                                                         \
      _Pragma("unroll") for (int t_ = 0; t_ < K; t_++) {                                                                        \
        const int k_ = (FWD) ? t_ : K - 1 - t_;                                                                                 \
        _Pragma("unroll") for (int r_ = 0; r_ < K; r_++) v[r_] = fmaf(g_[K * (j) + k_][r_], b_[k_], v[r_]);                     \
      }                                                                                                                         \
    }
    // The sweeps enter the unrolled update sequence through a jump table (switch on a block-uniform index) instead of testing every
    // position: descending runs fall through to position 0 with no test at all, ascending runs test their end once per step.
    // ONE ascending sequence serves the three sections (the section loop is kept rolled: a third of the code, see no_inst stalls).
#define DG_ASC_(j) case (j): DG_STEPK((j), true) if ((j) + 1 >= e_) break;
#define DG_DSC_(j) case (j) + 1: DG_STEPK((j), false)
#define DG_ASC8_ DG_ASC_(0) DG_ASC_(1) DG_ASC_(2) DG_ASC_(3) DG_ASC_(4) DG_ASC_(5) DG_ASC_(6) DG_ASC_(7)
#define DG_ASC16_ DG_ASC8_ DG_ASC_(8) DG_ASC_(9) DG_ASC_(10) DG_ASC_(11) DG_ASC_(12) DG_ASC_(13) DG_ASC_(14) DG_ASC_(15)
#define DG_ASC32_ DG_ASC16_ DG_ASC_(16) DG_ASC_(17) DG_ASC_(18) DG_ASC_(19) DG_ASC_(20) DG_ASC_(21) DG_ASC_(22) DG_ASC_(23) DG_ASC_(24) DG_ASC_(25) DG_ASC_(26) DG_ASC_(27) DG_ASC_(28) DG_ASC_(29) DG_ASC_(30) DG_ASC_(31)
#define DG_DSC8_ DG_DSC_(7) DG_DSC_(6) DG_DSC_(5) DG_DSC_(4) DG_DSC_(3) DG_DSC_(2) DG_DSC_(1) DG_DSC_(0)
#define DG_DSC16_ DG_DSC_(15) DG_DSC_(14) DG_DSC_(13) DG_DSC_(12) DG_DSC_(11) DG_DSC_(10) DG_DSC_(9) DG_DSC_(8) DG_DSC8_
#define DG_DSC32_ DG_DSC_(31) DG_DSC_(30) DG_DSC_(29) DG_DSC_(28) DG_DSC_(27) DG_DSC_(26) DG_DSC_(25) DG_DSC_(24) DG_DSC_(23) DG_DSC_(22) DG_DSC_(21) DG_DSC_(20) DG_DSC_(19) DG_DSC_(18) DG_DSC_(17) DG_DSC_(16) DG_DSC16_
    const int n1 = (P1 + K - 1) / K, n2 = (P2 + K - 1) / K, n3 = (Rp + K - 1) / K;   // step index where a section ends
    for (int it = 0; it < sc.iters; it++) {
      const bool fwd1 = (it & 1) != 0;
      if (!fwd1) {
        if constexpr (W == 32) { switch (n1) { DG_DSC32_ default: break; } } else if constexpr (W == 16) { switch (n1) { DG_DSC16_ default: break; } } else { switch (n1) { DG_DSC8_ default: break; } }
        DG_SETTLE
      }
#pragma unroll 1
      for (int sec = fwd1 ? 0 : 1; sec < 3; sec++) {
        const int s_ = sec == 0 ? 0 : (sec == 1 ? n1 : n2), e_ = sec == 0 ? n1 : (sec == 1 ? n2 : n3);
        if (sec == 2) {
          // friction bounds from the normal impulses this sweep left (the normal of contact c sits at warp position nrm0 + c: slot
          // (nrm0 + c) % K of lane (nrm0 + c) / K)
#pragma unroll
          for (int k = 0; k < K; k++) {
            const int pn = par[k] >= 0 ? nrm0 + par[k] : 0;
            float vn = 0.f;
#pragma unroll
            for (int k2 = 0; k2 < K; k2++) { const float vk = __shfl_sync(FULL, ap[k2], pn / K, W); vn = (pn % K) == k2 ? vk : vn; }
            if (par[k] >= 0) { hi[k] = mu[k] * vn; lo[k] = -hi[k]; lop[k] = lo[k] - ap[k]; hip[k] = hi[k] - ap[k]; }
          }
        }
        if (s_ >= e_) continue;
        if constexpr (W == 32) { switch (s_) { DG_ASC32_ default: break; } } else if constexpr (W == 16) { switch (s_) { DG_ASC16_ default: break; } } else { switch (s_) { DG_ASC8_ default: break; } }
        DG_SETTLE
      }
    }
#undef DG_SETTLE
#undef DG_ASC_
#undef DG_DSC_
#undef DG_ASC8_
#undef DG_ASC16_
#undef DG_ASC32_
#undef DG_DSC8_
#undef DG_DSC16_
#undef DG_DSC32_
#undef DG_STEPK
    if (writer) {
#pragma unroll
      for (int k = 0; k < K; k++) if (qown[k] >= 0) REC[RR_W * qown[k] + RR_APPLIED] = ap[k];
    }
    __syncwarp();
    // ... and what phase_rs_finish would do in the next stage launch, with W lanes and the rows still in cache: dv of every
    // body from the accumulated impulses (dv = sum_rows (M^-1 J^T)_row x applied_row, rows in order - the same sums), motor /
    // limit impulses back into their unit-row records.  Both live in the hot workspace: written into the environment's carry row.
    if (writer && live) {
      const int GV = sc.GV; const float* RSV = wg + sc.X_RSV;
      float* hot = a.carry + (size_t)emine * sc.w_total;
#pragma unroll 1
      for (int i = l; i < GV; i += W) {
        float sum = 0.f;
#pragma unroll 1
        for (int p = 0; p < L.Rp; p++) if (rs_real(L, p)) sum = fmaf(RSV[(size_t)p * 2 * GV + GV + i], REC[RR_W * p + RR_APPLIED], sum);
        hot[sc.W_DV + i] = sum;
      }
#pragma unroll 1
      for (int r = l; r < L.nu; r += W) {
        const int id = float_as_int(REC[RR_W * r + RR_ID]); const int* bp = sc.body_plan + BP_W * sc.dyn_body[(id >> 16) & 0x3fff];
        hot[sc.X_UROW + UR_W * (bp[BP_UROW] + (id & 0xffff)) + UR_APPLIED] = REC[RR_W * r + RR_APPLIED];
      }
    }
  }
}
// class c of the scene (DevScene::rs_cls_k / rs_cls_r): the instantiation with W = positions / K lanes per environment
static cudaError_t solve_launch(int cls, const DevScene& sc, const SolveArgs& a, int n_envs, cudaStream_t s) {
  const int K = sc.rs_cls_k[cls], W = sc.rs_cls_r[cls] / std::max(K, 1);
  if (K == 4 && W == 8) dg_solve_kernel<8, 4><<<(n_envs + 3) / 4, 32, 0, s>>>(sc, a);
  else if (K == 3 && W == 16) dg_solve_kernel<16, 3><<<(n_envs + 1) / 2, 32, 0, s>>>(sc, a);
  else if (K == 2 && W == 16) dg_solve_kernel<16, 2><<<(n_envs + 1) / 2, 32, 0, s>>>(sc, a);
  else if (K == 2 && W == 32) dg_solve_kernel<32, 2><<<n_envs, 32, 0, s>>>(sc, a);
  else return cudaErrorInvalidValue;
  return cudaGetLastError();
}
#endif

#if !defined(DG_STEP_T)
__global__ void dg_init_kernel(const __grid_constant__ DevScene sc, float* state, float* param, int n_envs) {
  size_t total_s = (size_t)n_envs * sc.S, total_p = (size_t)n_envs * sc.P;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total_s; i += stride) state[i] = sc.state_def[i % sc.S];
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total_p; i += stride) param[i] = sc.param_def[i % sc.P];
}

// ---------------------------------------------------------------- camera ----------------------------------------
// (ray_shape, the exact ray-shape test, is in dg_ray.cuh)

// per visual shape in shared memory, in FRONT-TO-BACK order (by the nearest eye-space depth of its oriented bounding box):
//   R(9) p(3) dims(4) rgb(3) type(1) bound radius(1) | M = R_shape^T R_cam (9), ray origin in the shape frame (3),
//   |origin|^2 - radius^2 (1) | nearest depth zmin (1), screen rectangle x0 x1 y0 y1 of the box (4, pixels, inclusive), body id (1)
#define VS_W 40
#define VS_ZMIN 34
#define VS_RECT 35
#define VS_BODY 39
template <int NCW, int NH, bool U8>
__global__ void __launch_bounds__(256, 3) dg_render_kernel(const __grid_constant__ DevScene sc, const float* state, const float* param, int cam, float* rgb, float* depth,
                                                        float* seg, int tiles_x, int tiles_y, int groups) {
  // a block = one environment (or the `groups`-th part of its image).  Once per block: world pose, camera-relative constants,
  // screen rectangle and nearest depth of every visual shape, sorted front to back.  Then every warp renders 8 x 8 pixel patches (two rays per lane):
  // the shapes whose rectangle overlaps the patch (a bit per shape, in that order), per pixel the ray against those shapes,
  // nearest first, until the next shape's nearest depth is behind the hit already found; the patch is staged in shared memory
  // and written as whole 128-bit pieces of image rows.
  extern __shared__ __align__(16) float vs[];       // [nv][VS_W], then keys [nv], then the candidate bit set
  __shared__ float camRp[12];
  __shared__ __align__(16) float t_rgb[8 * 192];   // per warp: a patch of 64 pixels
  __shared__ __align__(16) float t_dep[8 * 64];
  __shared__ __align__(16) float t_seg[8 * 64];
  (void)tiles_x; (void)tiles_y;
  const int e = blockIdx.x / groups, grp = blockIdx.x % groups;
  const int* ci = sc.cam_i + DG_CAM_I_W * cam; const float* cf = sc.cam_f + DG_CAM_F_W * cam;
  const int width = ci[1], height = ci[2];
  float* key = vs + VS_W * sc.nv;
  Env C; C.sc = &sc; C.st = const_cast<float*>(state) + (size_t)e * sc.S; C.ws = nullptr; C.wg = nullptr; C.pr = nullptr; C.dbg = nullptr; C.dropped = nullptr; C.rs_used = nullptr; C.no_hot = 0;
  C.link_i = sc.link_i; C.link_f = sc.link_f; C.link_x = sc.link_x;
  const float fov = cf[7], nearp = cf[8], farp = cf[9];
  const float th = tanf(fov * kPi / 360.0f), aspect = (float)width / (float)height;
  if (threadIdx.x == 0) {
    float Rp[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, pp[3] = {0, 0, 0}, Rl[9], t[3];
    if (ci[0] >= 0) { float q[4]; frame_link_pose(C, ci[0], pp, q); q_to_mat(Rp, q); }
    q_to_mat(Rl, cf + 3); m_mul(camRp, Rp, Rl); m_vec(t, Rp, cf); v_add(camRp + 9, pp, t);
  }
  __syncthreads();
  // ---- per-shape records (registers), keys, ranks, records to their sorted slot --------------------------------------------------
  for (int s0 = 0; s0 < sc.nv; s0 += blockDim.x) {
    const int s = s0 + threadIdx.x; float o[VS_W];
    if (s < sc.nv) {
      const int* vi = sc.vis_i + DG_VIS_I_W * s; const float* vf = sc.vis_f + DG_VIS_F_W * s;
      if (vi[2]) { for (int i = 0; i < 12; i++) o[i] = sc.vis_wb[12 * s + i]; }
      else {
        float p[3], q[4], v[3], w[3], R[9], Rs[9], t[3];
        frame_com_state(C, vi[0], p, q, v, w); q_to_mat(R, q); q_to_mat(Rs, vf + 3); m_mul(o, R, Rs);
        m_vec(t, R, vf); v_add(o + 9, p, t);
      }
      for (int i = 0; i < 4; i++) o[12 + i] = vf[7 + i];
      for (int i = 0; i < 3; i++) o[16 + i] = param[(size_t)e * sc.P + DG_PO(&sc, P_COLOR) + 3 * s + i];   // per-environment colour (visual_randomizer)
      o[19] = int_as_float(vi[1]); o[20] = vf[15];
      const float r = o[20];
      float oc[3], ol[3]; v_sub(oc, camRp + 9, o + 9); mT_vec(ol, o, oc);
      mT_mul(o + 21, o, camRp);                                   // camera-space direction -> shape-frame direction
      o[30] = ol[0]; o[31] = ol[1]; o[32] = ol[2]; o[33] = v_dot(ol, ol) - r * r;
      // oriented bounding box of the shape -> nearest eye-space depth and screen rectangle (whole screen if it reaches behind the eye)
      const int type = vi[1]; const float* d = o + 12;
      float hx = d[0], hy = d[1], hz = d[2];
      if (type == SHAPE_SPHERE) { hy = d[0]; hz = d[0]; } else if (type == SHAPE_CAPSULE) { hy = d[0]; hz = d[1] + d[0]; } else if (type == SHAPE_CYLINDER) { hy = d[0]; hz = d[1]; }
      // corners in camera space; the part of the box in front of the eye plane z = -zc is what can be seen: its screen rectangle
      // comes from the corners in front and from the points where edges cross that plane
      const float zc = fmaxf(0.5f * nearp, 1e-4f);
      float ccx[8], ccy[8], ccd[8];
      float zmin = 1e30f, x0 = 1e30f, x1 = -1e30f, y0 = 1e30f, y1 = -1e30f;
      const float sx = 0.5f * width / (th * aspect), sy = 0.5f * height / th;
      auto add_pt = [&](float cx, float cy, float dep) {
        const float px = fminf(fmaxf(cx / dep * sx, -1e6f), 1e6f) + 0.5f * width - 0.5f, py = fminf(fmaxf(-cy / dep * sy, -1e6f), 1e6f) + 0.5f * height - 0.5f;
        x0 = fminf(x0, px); x1 = fmaxf(x1, px); y0 = fminf(y0, py); y1 = fmaxf(y1, py);
      };
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const float cl[3] = {(k & 1) ? hx : -hx, (k & 2) ? hy : -hy, (k & 4) ? hz : -hz};
        float cw[3], rel[3], cc[3]; m_vec(cw, o, cl); v_add(cw, cw, o + 9); v_sub(rel, cw, camRp + 9); mT_vec(cc, camRp, rel);
        ccx[k] = cc[0]; ccy[k] = cc[1]; ccd[k] = -cc[2];
        zmin = fminf(zmin, ccd[k]);
        if (ccd[k] > zc) add_pt(cc[0], cc[1], ccd[k]);
      }
#pragma unroll
      for (int k = 0; k < 8; k++) {
#pragma unroll
        for (int bit = 1; bit < 8; bit <<= 1) {
          if (k & bit) continue;
          const int k2 = k | bit;
          if ((ccd[k] > zc) == (ccd[k2] > zc)) continue;
          const float t = (zc - ccd[k]) / (ccd[k2] - ccd[k]);
          add_pt(ccx[k] + t * (ccx[k2] - ccx[k]), ccy[k] + t * (ccy[k2] - ccy[k]), zc);
        }
      }
      if (x1 < x0) { x0 = y0 = 1e9f; x1 = y1 = -1e9f; }   // nothing of the box in front of the eye: never a candidate
      zmin = fmaxf(zmin, 0.f);
      o[VS_ZMIN] = zmin;
      o[VS_RECT] = floorf(fmaxf(x0, -1e6f)) - 1.f; o[VS_RECT + 1] = ceilf(fminf(x1, 1e6f)) + 1.f;
      o[VS_RECT + 2] = floorf(fmaxf(y0, -1e6f)) - 1.f; o[VS_RECT + 3] = ceilf(fminf(y1, 1e6f)) + 1.f;
      o[VS_BODY] = (float)vi[3];
      key[s] = zmin;
    }
    __syncthreads();
    if (s < sc.nv) {
      int rank = 0; const float ks = key[s];
      for (int s2 = 0; s2 < sc.nv; s2++) { const float k2 = key[s2]; rank += (k2 < ks || (k2 == ks && s2 < s)) ? 1 : 0; }
      float* dst = vs + VS_W * rank;
#pragma unroll
      for (int i = 0; i < VS_W; i += 4) st4(dst + i, o[i], o[i + 1], o[i + 2], o[i + 3]);
    }
  }
  __syncthreads();
  const float light[3] = {0.4082482904638631f, 0.4082482904638631f, 0.8164965809277261f};
  const int npx = width * height;
  float* rgb_e = rgb + (size_t)e * npx * 3; float* dep_e = depth + (size_t)e * npx; float* seg_e = seg ? seg + (size_t)e * npx : nullptr;
  // U8: the colour image is [H][W][3] bytes, round(255 c) - what the reference's camera reads from the renderer before it divides by 255
  // (sensors/camera.py:76-78)
  unsigned char* rgb8_e = reinterpret_cast<unsigned char*>(rgb) + (size_t)e * npx * 3;
  auto to_u8 = [](float c) { return (unsigned char)__float2uint_rn(__saturatef(c) * 255.0f); };
  // Every WARP renders patches of MT_W x MT_H = 64 pixels on its own (no block barrier in this loop): the lanes test the shapes'
  // screen rectangles against the patch (ballots -> candidate bits in registers, front to back), every lane casts the ray of its
  // pixel, and the patch goes out as 128-bit pieces of image rows through the warp's slice of the staging buffers.
  constexpr int MT_W = 8, MT_H = 4 * NH;   // NH = 2: 8 x 8 patches, two rays per lane; NH = 1: 8 x 4, one ray (small images)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  const int mtx = (width + MT_W - 1) / MT_W, mty = (height + MT_H - 1) / MT_H, nmt = mtx * mty;
  const bool vec_ok = (width % (U8 ? 8 : 4)) == 0;   // image rows and patch offsets keep 16-byte (colour bytes: 8-byte) alignment
  float* w_rgb = t_rgb + 192 * warp; float* w_dep = t_dep + 64 * warp; float* w_seg = t_seg + 64 * warp;
  // NCW candidate words live in registers (32 NCW shapes; beyond 128: see below).  Lane l owns shapes l, 32 + l, ...: their screen
  // rectangles stay in its registers for the whole image, so the per-patch overlap test reads no memory.
  float rx0[NCW], rx1[NCW], ry0[NCW], ry1[NCW];
#pragma unroll
  for (int wd = 0; wd < NCW; wd++) {
    const int s = 32 * wd + lane; const bool in = s < sc.nv; const float* o = vs + VS_W * (in ? s : 0);
    rx0[wd] = in ? o[VS_RECT] : 1e9f; rx1[wd] = in ? o[VS_RECT + 1] : -1e9f; ry0[wd] = in ? o[VS_RECT + 2] : 1e9f; ry1[wd] = in ? o[VS_RECT + 3] : -1e9f;
  }
  // per-lane constants of the ray direction and of the staged stores.  A lane casts TWO rays per patch: pixels (li, lj) and
  // (li, lj + 4) of the 8 x 8 patch, so that the candidate ballots, the patch bookkeeping and the store addressing are paid once per
  // 64 pixels.  The patch leaves as 64 128-bit pieces (48 of colour, 16 of depth): two per lane.
  const int li = lane % MT_W, lj = lane / MT_W;
  const float kx = 2.0f * th * aspect / (float)width, ky = 2.0f * th / (float)height, cx0 = th * aspect, cy0 = th;
  // piece t of lane: index lane + 32 t.  NH = 2: < 48 colour (row idx / 6, float4 idx % 6), else depth (row (idx - 48) / 2, float4
  // (idx - 48) % 2), mask pieces on lanes 0..15.  NH = 1: one piece per lane, 0..23 colour, 24..31 depth and mask.
  const int row0 = NH == 2 ? lane / 6 : (lane < 24 ? lane / 6 : (lane - 24) / 2), c0 = NH == 2 ? lane % 6 : (lane < 24 ? lane % 6 : (lane - 24) % 2);
  const bool col0 = NH == 2 || lane < 24;
  const bool col1 = lane < 16;                                    // t = 1 (NH = 2 only): colour for lanes 0..15, depth for 16..31
  const int row1 = col1 ? (lane + 32) / 6 : (lane - 16) / 2, c1 = col1 ? (lane + 32) % 6 : (lane - 16) % 2;
  const int rows = NH == 2 ? lane / 2 : row0, cs = NH == 2 ? lane % 2 : c0;   // mask pieces
  const bool seg_lane = NH == 2 ? lane < 16 : lane >= 24;
  const unsigned off0 = col0 ? (unsigned)(row0 * width * 3 + 4 * c0) : (unsigned)(row0 * width + 4 * c0),
                 off1 = col1 ? (unsigned)(row1 * width * 3 + 4 * c1) : (unsigned)(row1 * width + 4 * c1), offs = (unsigned)(rows * width + 4 * cs);
  const float* src0 = col0 ? w_rgb + 24 * row0 + 4 * c0 : w_dep + 8 * row0 + 4 * c0;
  const float* src1 = col1 ? w_rgb + 24 * row1 + 4 * c1 : w_dep + 8 * row1 + 4 * c1;
  const float* srcs = w_seg + 8 * rows + 4 * cs;
  // U8: a patch row of colour is 24 bytes = three 64-bit pieces: lanes 0 .. 3 MT_H - 1; depth pieces (two float4 per row) on the next
  // 2 MT_H lanes (NH = 1) or in a second round on lanes 0..15 (NH = 2); mask pieces after them
  unsigned char* w8 = reinterpret_cast<unsigned char*>(w_rgb);
  const int b_row = lane / 3, b_c = lane % 3;
  const int d_lane = NH == 2 ? lane : lane - 12, s_lane = NH == 2 ? lane - 16 : lane - 20;
  const bool d_on = d_lane >= 0 && d_lane < 2 * MT_H, s_on = s_lane >= 0 && s_lane < 2 * MT_H;
  const unsigned b_off = (unsigned)(b_row * width * 3 + 8 * b_c), d_off = (unsigned)((d_lane / 2) * width + 4 * (d_lane % 2)), s_off = (unsigned)((s_lane / 2) * width + 4 * (s_lane % 2));
  // patches in row-major order, mt = grp nwarp + warp, then + groups nwarp: column / row kept incrementally (no division per patch)
  const int stride = groups * nwarp, dcol = stride % mtx, drow = stride / mtx;
  int mt = grp * nwarp + warp, pcol = mt % mtx, prow = mt / mtx;
  for (; mt < nmt; mt += stride, pcol += dcol, prow += drow) {
    if (pcol >= mtx) { pcol -= mtx; prow++; }
    const int px0 = pcol * MT_W, py0 = prow * MT_H;
    unsigned cw[NCW];
    {
      const float fx0 = (float)px0, fx1 = (float)(px0 + MT_W - 1), fy0 = (float)py0, fy1 = (float)(py0 + MT_H - 1);
#pragma unroll
      for (int wd = 0; wd < NCW; wd++) cw[wd] = __ballot_sync(0xffffffffu, rx0[wd] <= fx1 && rx1[wd] >= fx0 && ry0[wd] <= fy1 && ry1[wd] >= fy0);
    }
    const int wt = min(MT_W, width - px0), ht = min(MT_H, height - py0);
    const bool staged = vec_ok && wt == MT_W;
    const int i = px0 + li;
    if (staged) __syncwarp();                                      // the previous patch has left the staging buffers
#pragma unroll 1
    for (int half = 0; half < NH; half++) {
      const int j = py0 + lj + 4 * half, slot = lane + 32 * half;
      float r = 1.0f, g = 1.0f, bl = 1.0f, dz = -farp, sid = -1.0f;
      if (i < width && j < height) {
        const float dc[3] = {fmaf((float)i + 0.5f, kx, -cx0), fmaf((float)j + 0.5f, -ky, cy0), -1.0f};
        const float dd = v_dot(dc, dc);                            // rotations keep the length of the direction
        float best = farp; int hs = -1; float hnl[3] = {0, 0, 1};
        bool done = false;
        auto try_shape = [&](int s) {
          const float* o = vs + VS_W * s;
          // the ray parameter IS the eye-space depth (the camera-space direction has z = -1): nothing behind `best` can win
          if (o[VS_ZMIN] >= best) { done = true; return; }
          float dl[3]; m_vec(dl, o + 21, dc);
          const float b = v_dot(o + 30, dl), c2 = o[33];          // per-ray bounding-sphere reject, in the shape frame
          if (c2 > 0.f && (b > 0.f || b * b < c2 * dd)) return;
          float tt, nn[3];
          if (ray_shape(float_as_int(o[19]), o + 12, o + 30, dl, best, &tt, nn) && tt >= nearp) { best = tt; hs = s; v_cpy(hnl, nn); }
        };
#pragma unroll
        for (int wd = 0; wd < NCW; wd++) {
          unsigned bits = cw[wd];
          while (bits && !done) { const int s = 32 * wd + __ffs(bits) - 1; bits &= bits - 1; try_shape(s); }
        }
        if (NCW == 4) for (int s = 128; s < sc.nv && !done; s++) {  // scenes with more than 128 visual shapes: the rest one by one
          const float* o = vs + VS_W * s;
          if (o[VS_RECT] <= (float)i && o[VS_RECT + 1] >= (float)i && o[VS_RECT + 2] <= (float)j && o[VS_RECT + 3] >= (float)j) try_shape(s);
        }
        if (hs >= 0) {
          float hn[3]; m_vec(hn, vs + VS_W * hs, hnl);
          const float* col = vs + VS_W * hs + 16; const float nl = fmaxf(v_dot(hn, light), 0.f), sh = 0.4f + 0.6f * nl;
          r = col[0] * sh; g = col[1] * sh; bl = col[2] * sh; dz = -best; sid = vs[VS_W * hs + VS_BODY];
        }
        if (!staged) {
          const size_t px = (size_t)j * width + i;
          if (U8) { rgb8_e[3 * px] = to_u8(r); rgb8_e[3 * px + 1] = to_u8(g); rgb8_e[3 * px + 2] = to_u8(bl); }
          else { rgb_e[3 * px] = r; rgb_e[3 * px + 1] = g; rgb_e[3 * px + 2] = bl; }
          dep_e[px] = dz;
          if (seg_e) seg_e[px] = sid;
        }
      }
      if (staged) {
        if (U8) { w8[3 * slot] = to_u8(r); w8[3 * slot + 1] = to_u8(g); w8[3 * slot + 2] = to_u8(bl); }
        else { w_rgb[3 * slot] = r; w_rgb[3 * slot + 1] = g; w_rgb[3 * slot + 2] = bl; }
        w_dep[slot] = dz; w_seg[slot] = sid;
      }
    }
    if (staged && U8) {
      __syncwarp();
      const unsigned pb = (unsigned)(py0 * width + px0);
      if (lane < 3 * MT_H && b_row < ht) *reinterpret_cast<uint2*>(rgb8_e + 3u * pb + b_off) = *reinterpret_cast<const uint2*>(w8 + 24 * b_row + 8 * b_c);
      if (d_on && d_lane / 2 < ht) *reinterpret_cast<float4*>(dep_e + pb + d_off) = *reinterpret_cast<const float4*>(w_dep + 4 * d_lane);
      if (seg_e && s_on && s_lane / 2 < ht) *reinterpret_cast<float4*>(seg_e + pb + s_off) = *reinterpret_cast<const float4*>(w_seg + 4 * s_lane);
    } else if (staged) {
      __syncwarp();
      const unsigned pb = (unsigned)(py0 * width + px0);
      if (row0 < ht) {
        if (col0) *reinterpret_cast<float4*>(rgb_e + 3u * pb + off0) = *reinterpret_cast<const float4*>(src0);
        else *reinterpret_cast<float4*>(dep_e + pb + off0) = *reinterpret_cast<const float4*>(src0);
      }
      if (NH == 2 && row1 < ht) {
        if (col1) *reinterpret_cast<float4*>(rgb_e + 3u * pb + off1) = *reinterpret_cast<const float4*>(src1);
        else *reinterpret_cast<float4*>(dep_e + pb + off1) = *reinterpret_cast<const float4*>(src1);
      }
      if (seg_e && seg_lane && rows < ht) *reinterpret_cast<float4*>(seg_e + pb + offs) = *reinterpret_cast<const float4*>(srcs);
    }
  }
}

// ---------------------------------------------------------------- ray_sensor ------------------------------------
// dg_ray_kernel: every ray_sensor op of the scene (dg_ray.cuh) in one launch, one warp per environment.  The warp puts the world
// poses of the collision shapes that move (from the state row's link cache) into its slice of shared memory; baked shapes use the
// compiled world poses (DevScene::shape_wb, the same for every environment: L1 / L2 resident).  Lane l casts rays l, l + 32, ...
// against every shape (bounding-sphere rejection, then the exact test in the shape frame); consecutive lanes store consecutive
// floats of the op's slice of the observation row.
constexpr int kRayWarps = 4;   // environments per block
__global__ void __launch_bounds__(32 * kRayWarps) dg_ray_kernel(const __grid_constant__ DevScene sc, const float* state, float* obs, const uint8_t* mask, int n_envs) {
  extern __shared__ __align__(16) float ray_mov[];   // [kRayWarps][nshw][12]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * kRayWarps + warp;
  if (e >= n_envs || (mask != nullptr && mask[e] == 0)) return;   // (whole warps: no barrier below spans more than one)
  float* mov = ray_mov + (size_t)warp * 12 * sc.nshw;
  Env C; C.sc = &sc; C.st = const_cast<float*>(state) + (size_t)e * sc.S; C.obs = obs + (size_t)e * sc.n_obs;
  C.ws = nullptr; C.wg = nullptr; C.pr = nullptr; C.dbg = nullptr; C.dropped = nullptr; C.rs_used = nullptr; C.no_hot = 0;
  C.link_i = sc.link_i; C.link_f = sc.link_f; C.link_x = sc.link_x;
  ray_stage_shapes(C, mov, lane, 32);
  __syncwarp();
  ray_env(C, mov, lane, 32);
}

// ---------------------------------------------------------------- dynamics queries --------------------------------
// dg_dyn_kernel: Jacobian / mass matrix / inverse dynamics of one body (dg_dyn.cuh), one warp per environment.  Lane 0 walks the
// body's links once (poses, velocities, accelerations) into the warp's slice of shared memory; then the lanes split the links
// (world inertias, link wrenches) and the outputs (Jacobian columns, upper-triangle entries of M, generalized forces).
constexpr int kDynWarps = 4;   // environments per block
__global__ void __launch_bounds__(32 * kDynWarps) dg_dyn_kernel(const __grid_constant__ DevScene sc, const DynArgs a, const float* state, const float* param, int n_envs) {
  extern __shared__ __align__(16) float dyn_smem[];   // [kDynWarps][dyn_scratch_floats(nl, n)]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.x * kDynWarps + warp;
  if (e >= n_envs) return;   // (whole warps: no barrier below spans more than one)
  float* base = dyn_smem + (size_t)warp * dyn_scratch_floats(a.nl, a.n);
  unsigned long long* msk = reinterpret_cast<unsigned long long*>(base);
  float* L = base + 2 * a.nl; float* col = L + DL_W_ * a.nl; float* pt = col + DC_W_ * a.n;
  const float* pr = param + (size_t)e * sc.P;
  if (lane == 0) dyn_chain(sc, a, state + (size_t)e * sc.S, pr, e, msk, L, col);
  __syncwarp();
  dyn_links(sc, a, pr, L, pt, lane, 32);
  __syncwarp();
  dyn_outputs(a, e, msk, L, col, pt, lane, 32);
}

// ---------------------------------------------------------------- inverse-kinematics query -------------------------
// dg_ik_kernel: calculateInverseKinematics of one body (dg_ik.cuh), one lane per environment.  Every iteration of the solve walks
// the link chain serially, so a warp per environment would leave 31 lanes idle; small blocks spread the environments over the
// SMs.  The block first stages the link tables in shared memory, because ik_solve* and joint_xform read them through shc().
// MAXD > 0: ik_solve_fast<MAXD, M>, its scratch in a per-thread array; MAXD = 0: the generic ik_solve, its scratch in the world's
// IK buffer behind the seed record.
constexpr int kIkThreads = 64;
template <int MAXD, int M>
__global__ void __launch_bounds__(kIkThreads) dg_ik_kernel(const __grid_constant__ DevScene sc, const IkArgs a, const float* state, int n_envs) {
  extern __shared__ __align__(16) float ik_smem[];
  int* s_link_i = reinterpret_cast<int*>(ik_smem);
  float* s_link_f = reinterpret_cast<float*>(s_link_i + ((DG_LINK_I_W * sc.nl + 3) & ~3));
  float* s_link_x = s_link_f + DG_LINK_F_W * sc.nl;
  for (int i = threadIdx.x; i < DG_LINK_I_W * sc.nl; i += blockDim.x) s_link_i[i] = sc.link_i[i];
  for (int i = threadIdx.x; i < DG_LINK_F_W * sc.nl; i += blockDim.x) s_link_f[i] = sc.link_f[i];
  for (int i = threadIdx.x; i < 16 * sc.nl; i += blockDim.x) s_link_x[i] = sc.link_x[i];
  __syncthreads();
  const int e = blockIdx.x * kIkThreads + threadIdx.x;
  if (e >= n_envs) return;
  Env C;
  C.sc = &sc; C.link_i = s_link_i; C.link_f = s_link_f; C.link_x = s_link_x;
  C.st = a.rec + (size_t)e * a.rec_stride;
  float scr[IkFastScratch<MAXD>::floats];
  ik_env<MAXD, M>(C, a, state + (size_t)e * sc.S, e, scr);
}
template <int MAXD, int M>
static cudaError_t ik_launch(const DevScene& d, const IkArgs& a, const float* state, int n_envs, size_t smem, cudaStream_t stream) {
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(dg_ik_kernel<MAXD, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  dg_ik_kernel<MAXD, M><<<(n_envs + kIkThreads - 1) / kIkThreads, kIkThreads, smem, stream>>>(d, a, state, n_envs);
  return cudaGetLastError();
}

}  // namespace dg

// ---------------------------------------------------------------- C ABI ------------------------------------------
using namespace dg;

struct DgWorld {
  HostScene hs;
  DevScene dev;            // pointers re-targeted to device memory
  int* d_ints = nullptr; float* d_floats = nullptr;
  int n_envs = 0, device = 0, team = 1, block_threads = 64, grid = 1, sm_count = 148;
  size_t smem = 0, smem_cap = 0;
  DgBufferTable buf{};
  bool bound = false;
  uint32_t seed = 1234u; int env_off = 0;
  unsigned long long opmask[2] = {~0ull, ~0ull};
  float* gws = nullptr;
  unsigned long long* dbg = nullptr;   // [grid][64] phase-cycle sums while dg_debug_phase_cycles is on
  unsigned* dropped = nullptr;         // device counter of contacts lost to the max_contacts cap
  // split schedule: stage launches of the step kernel around the sweep kernel (see run_step_split)
  bool split = false;
  float* carry = nullptr;              // [n_envs + slack][w_total] hot workspaces between stage launches
  int* rs_lists = nullptr;             // [2][n_envs] environments deferred to the sweep kernel (K = 1 | K = 2)
  int* rs_counts = nullptr;            // [substeps][2]
  cudaStream_t aux = nullptr, aux2 = nullptr; cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_join2 = nullptr;   // the sweep classes run side by side
  // Which schedule a step takes is decided from how many environments actually needed the contact solver lately: the stage
  // launches + carry traffic cost ~0.3 ms per step, which only pays when a good share of the environments is in contact
  // (a drone in the air, an R2D2 still falling: fused launch).  The device counter is copied to pinned memory every
  // kAdaptPeriod steps, asynchronously, and read one period later - no host synchronisation on the step path.
  bool split_ok = false;               // the scene and team allow the split schedule at all
  int split_mode = -1;                 // DG_SPLIT: 0 never, 1 always, -1 adaptive
  unsigned* rs_used = nullptr; unsigned* h_rs_used = nullptr; cudaEvent_t ev_stat = nullptr;
  int steps_in_period = 0; bool stat_pending = false;
  // DG_GRAPH=1: the launch sequence of a split step (memset, 3 stage launches, 4 sweep launches, the fork / join events) replayed
  // as one CUDA graph, captured on `cap` when the launch arguments change (action mask, seed), launched on the caller's stream.
  // Off by default: measured no gain (r2d2_maze 1.99 vs 1.98 ms, drone_pilot 0.56 vs 0.53 ms per step) - launch overhead is not
  // what separates the step from the sum of its kernels
  int use_graph = 0; cudaStream_t cap = nullptr; cudaGraph_t graph = nullptr; cudaGraphExec_t graph_exec = nullptr;
  unsigned long long graph_key[4] = {0, 0, 0, 0}; bool graph_valid = false;
  // ray_sensor ops (dg_ray_kernel, launched after the step / reset / observe launches when the scene has any)
  std::vector<int> ray_ops; size_t ray_smem = 0;
  // dg_body_ik: [n_envs][seed record + ik_stride] (dg_ik.cuh), allocated by the first call
  float* ik_rec = nullptr;
  int64_t launches = 0;
  std::string err;
};
static std::string g_create_err;

// Every entry point runs on the world's own device, whatever the caller's current device is (two worlds on two GPUs in one
// process, or a torch current device different from the world's), and leaves the caller's device as it found it.
struct DeviceGuard {
  int prev = -1; bool ok = true;
  explicit DeviceGuard(int dev) { if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); } if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess; else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define CK(w, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { (w)->err = std::string(#call) + ": " + cudaGetErrorString(e_); return DG_E_CUDA; } } while (0)

static cudaError_t configure_any(DgWorld* w) {
  int occ = 0; cudaError_t e;
  switch (w->team) {
    case 1: e = dg_step_configure_1(w->block_threads, w->smem, w->smem_cap, &occ); break;
    case 2: e = dg_step_configure_2(w->block_threads, w->smem, w->smem_cap, &occ); break;
    case 4: e = dg_step_configure_4(w->block_threads, w->smem, w->smem_cap, &occ); break;
    case 8: e = dg_step_configure_8(w->block_threads, w->smem, w->smem_cap, &occ); break;
    case 16: e = dg_step_configure_16(w->block_threads, w->smem, w->smem_cap, &occ); break;
    default: e = dg_step_configure_32(w->block_threads, w->smem, w->smem_cap, &occ); break;
  }
  if (e != cudaSuccess) return e;
  if (occ < 1) occ = 1;
  int teams_per_block = w->block_threads / w->team;
  int need = (w->n_envs + teams_per_block - 1) / teams_per_block;
  w->grid = std::max(1, std::min(need, w->sm_count * occ));
  return cudaSuccess;
}
static cudaError_t launch_any(DgWorld* w, const LaunchArgs& a, cudaStream_t s) {
  w->launches++;
  const StepLaunch l{w->grid, w->block_threads, w->smem, s};
  switch (w->team) {
    case 1: return dg_step_launch_1(w->dev, a, l); case 2: return dg_step_launch_2(w->dev, a, l); case 4: return dg_step_launch_4(w->dev, a, l);
    case 8: return dg_step_launch_8(w->dev, a, l); case 16: return dg_step_launch_16(w->dev, a, l); default: return dg_step_launch_32(w->dev, a, l);
  }
}

extern "C" {

const char* dg_last_error(const DgWorld* w) { return w ? w->err.c_str() : g_create_err.c_str(); }

int dg_world_create(const int32_t* ibuf, int n_ibuf, const double* fbuf, int n_fbuf, int n_envs, int device, int team, DgWorld** out) {
  if (!ibuf || !fbuf || !out || n_envs < 1) { g_create_err = "dg_world_create: bad argument"; return DG_E_ARG; }
  if (team != 0 && team != 1 && team != 2 && team != 4 && team != 8 && team != 16 && team != 32) { g_create_err = "dg_world_create: team must be 0,1,2,4,8,16,32"; return DG_E_ARG; }
  DgWorld* w = new DgWorld();
  w->n_envs = n_envs; w->device = device;
  DeviceGuard guard(device);
  cudaError_t e = guard.ok ? cudaSuccess : cudaGetLastError();
  if (e != cudaSuccess || !guard.ok) { g_create_err = std::string("cudaSetDevice: ") + cudaGetErrorString(e); delete w; return DG_E_CUDA; }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) { g_create_err = std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e); delete w; return DG_E_CUDA; }
  w->sm_count = prop.multiProcessorCount;
  const size_t smem_cap = prop.sharedMemPerBlockOptin;
  w->smem_cap = smem_cap;
  if (team == 0) {
    // built-in choice (from the team-size sweeps in profiles/): 4 lanes per environment for small scenes (two lanes
    // carry the per-body phases of a two-arm scene, the others help in the per-column / per-pair / per-row phases),
    // 8 lanes when the bodies have more than 12 generalized coordinates in total; DG_TEAM overrides
    const char* env_team = getenv("DG_TEAM");
    if (env_team) team = atoi(env_team);
    else {
      const int32_t* bsec = ibuf + ibuf[2 + 3 * SEC_BODY_I + 1]; const int nb_ = ibuf[ibuf[2 + 3 * SEC_HDR_I + 1] + HI_nb];
      int coords = 0;
      for (int b = 0; b < nb_; b++) if (bsec[DG_BODY_I_W * b] != 0) coords += (bsec[DG_BODY_I_W * b] == 2 ? 6 : 0) + bsec[DG_BODY_I_W * b + 4];
      team = coords > 12 ? 8 : 4;
      // fixed constraints between models ride on the row-space team solver, whose row capacity grows with the team
      const int32_t* hsec = ibuf + ibuf[2 + 3 * SEC_HDR_I + 1];
      auto pad8 = [](int n) { return (n + RS_KMAX - 1) / RS_KMAX * RS_KMAX; };
      const int rows_pad = pad8(2 * hsec[HI_nd]) + pad8(hsec[HI_max_contacts] + 6 * hsec[HI_ncons]) + pad8(2 * hsec[HI_max_contacts]);
      while (hsec[HI_ncons] > 0 && team < 32 && RS_KMAX * team < rows_pad) team *= 2;
    }
    if (team != 1 && team != 2 && team != 4 && team != 8 && team != 16 && team != 32) team = 4;
  }
  // environments per block: 32 (one warp per lane index) unless the block would exceed 256 threads or the batch is
  // too small to give every SM a few blocks; DG_ENVS_PER_BLOCK overrides
  const char* env_e = getenv("DG_ENVS_PER_BLOCK");
  int epb = env_e ? atoi(env_e) : 32;
  if (!env_e) {
    // measured (profiles/r1_block_size_sweep.log): scenes of small teams with articulated bodies (ur_high_5) run best with
    // full 32-environment blocks as long as every SM gets ~1.5 of them; the others want at least 2 smaller blocks per SM
    const int nd_ = ibuf[ibuf[2 + 3 * SEC_HDR_I + 1] + HI_nd];
    const int num = (team <= 4 && nd_ >= 8) ? 3 : 4;   // blocks per SM x 2
    while (epb > 8 && 2 * ((n_envs + epb - 1) / epb) < num * w->sm_count) epb /= 2;
  }
  while (epb * team > 256) epb /= 2;
  if (epb < 1) epb = 1;
  int block = epb * team;
  // workspace placement (dg_scene.h): frames / joint transforms / articulated-body transients always live in the
  // L2-backed cold workspace and the solver state in shared memory; the contact arrays default to the cold workspace
  // too (mode 3: measured faster on every example scene because more environments stay resident per SM);
  // DG_WS_MODE=2 keeps them in shared memory.
  const char* env_mode = getenv("DG_WS_MODE");
  int ws_mode = env_mode ? atoi(env_mode) : 3;
  if (ws_mode != 2 && ws_mode != 3) ws_mode = 3;
  if (!w->hs.build(ibuf, n_ibuf, fbuf, n_fbuf, team, ws_mode)) { g_create_err = "scene: " + w->hs.error; delete w; return DG_E_SCENE; }
  // DG_SOLVER=0: coupled environments fall back to lock-step dv-space sweeps; DG_RS_MIN=<rows>: uncoupled environments with
  // at least that many contact rows are solved in row space too (both kept for A/B measurements)
  if (const char* env_solver = getenv("DG_SOLVER")) w->hs.dev.solver = atoi(env_solver) != 0;
  if (const char* env_min = getenv("DG_RS_MIN")) w->hs.dev.rs_min = atoi(env_min);
  // DG_SWEEP_CLASSES="K:R,K:R,K:R" (rows per lane : row positions; 0:0 = unused) replaces the sweep-kernel classes, e.g. "2:32,0:0,2:64"
  // = the two-rows-per-lane classes of the first split build (A/B measurements)
  if (const char* ec = getenv("DG_SWEEP_CLASSES")) {
    int k[RS_NCLS] = {0, 0, 0}, r[RS_NCLS] = {0, 0, 0};
    if (sscanf(ec, "%d:%d,%d:%d,%d:%d", &k[0], &r[0], &k[1], &r[1], &k[2], &r[2]) >= 2) {
      bool ok = true;
      for (int c = 0; c < RS_NCLS; c++) ok = ok && (r[c] == 0 || (k[c] == 4 && r[c] == 32) || (k[c] == 3 && r[c] == 48) || (k[c] == 2 && (r[c] == 32 || r[c] == 64)));
      if (ok) for (int c = 0; c < RS_NCLS; c++) { w->hs.dev.rs_cls_k[c] = k[c]; w->hs.dev.rs_cls_r[c] = r[c]; }
    }
  }
  if (const char* env_pr = getenv("DG_PRECISE")) w->hs.dev.precise = atoi(env_pr) != 0;   // A/B of the SFU sincos in FK / IK (tools/qd_probe.py)
  {
    size_t per_team = (size_t)w->hs.dev.w_total * sizeof(float);
    const int nl_ = w->hs.dev.nl;
    size_t tables = (size_t)(((DG_LINK_I_W * nl_ + 3) & ~3) + (DG_LINK_F_W + 16) * nl_ + 4) * sizeof(float);   // block-shared link tables
    int teams = block / team;
    while (teams > 1 && per_team * teams + tables > smem_cap) teams--;
    if (per_team * teams + tables > smem_cap) { g_create_err = "scene workspace (" + std::to_string(per_team) + " B per environment) exceeds shared memory"; delete w; return DG_E_NOMEM; }
    w->block_threads = teams * team; w->smem = per_team * teams + tables;
  }
  w->team = team;
  // upload the constant tables
  size_t nbi = w->hs.ints.size() * sizeof(int), nbf = w->hs.floats.size() * sizeof(float);
  if (cudaMalloc(&w->d_ints, nbi) != cudaSuccess || cudaMalloc(&w->d_floats, nbf) != cudaSuccess) { g_create_err = "cudaMalloc of scene tables failed"; cudaGetLastError(); dg_world_destroy(w); return DG_E_CUDA; }
  if (cudaMemcpy(w->d_ints, w->hs.ints.data(), nbi, cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(w->d_floats, w->hs.floats.data(), nbf, cudaMemcpyHostToDevice) != cudaSuccess) { g_create_err = "upload of scene tables failed"; cudaGetLastError(); dg_world_destroy(w); return DG_E_CUDA; }
  w->dev = w->hs.dev;
  w->hs.point(w->dev, w->d_ints, w->d_floats);
  e = configure_any(w);
  if (e != cudaSuccess) { g_create_err = std::string("kernel configuration: ") + cudaGetErrorString(e); dg_world_destroy(w); return DG_E_CUDA; }
  {
    // cold workspace: one slot per ENVIRONMENT (it travels between the stage launches of the split schedule), with slack for the
    // environment-less tail slots of the last block
    size_t slots = (size_t)w->n_envs + 256;
    size_t bytes = std::max<size_t>(slots * (size_t)w->hs.dev.g_total * sizeof(float), 16);
    if (cudaMalloc(&w->gws, bytes) != cudaSuccess) { g_create_err = "cudaMalloc of the cold workspace (" + std::to_string(bytes >> 20) + " MiB) failed"; cudaGetLastError(); dg_world_destroy(w); return DG_E_NOMEM; }
    w->dev.g_total = w->hs.dev.g_total;
  }
  {
    // split schedule: possible for every scene with contacts or welds and a team of >= 2 lanes (row-space solver); taken when
    // enough environments are in contact (adaptive, see DgWorld).  DG_SPLIT=0 / 1 forces never / always.
    w->split_ok = w->hs.dev.rs_cap > 0 && w->hs.dev.solver == 1 && (w->hs.dev.npair > 0 || w->hs.dev.ncons > 0);
    if (const char* env_split = getenv("DG_SPLIT")) w->split_mode = atoi(env_split) != 0 ? 1 : 0;
    if (w->split_mode == 0) w->split_ok = false;
    if (const char* env_graph = getenv("DG_GRAPH")) w->use_graph = atoi(env_graph) != 0;
    w->split = w->split_ok && (w->split_mode == 1 || w->hs.dev.ncons > 0);   // welded models always have rows; else start fused and adapt
    if (w->split_ok) {
      const size_t nc = ((size_t)w->n_envs + 256) * (size_t)w->hs.dev.w_total * sizeof(float);
      bool ok = cudaMalloc(&w->carry, nc) == cudaSuccess && cudaMalloc(&w->rs_lists, RS_NCLS * (size_t)w->n_envs * sizeof(int)) == cudaSuccess &&
                cudaMalloc(&w->rs_counts, RS_NCLS * (size_t)std::max(w->hs.dev.substeps, 1) * sizeof(int)) == cudaSuccess &&
                cudaStreamCreateWithFlags(&w->aux, cudaStreamNonBlocking) == cudaSuccess && cudaStreamCreateWithFlags(&w->aux2, cudaStreamNonBlocking) == cudaSuccess &&
                cudaStreamCreateWithFlags(&w->cap, cudaStreamNonBlocking) == cudaSuccess && cudaEventCreateWithFlags(&w->ev_join2, cudaEventDisableTiming) == cudaSuccess &&
                cudaEventCreateWithFlags(&w->ev_fork, cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&w->ev_join, cudaEventDisableTiming) == cudaSuccess &&
                cudaEventCreateWithFlags(&w->ev_stat, cudaEventDisableTiming) == cudaSuccess && cudaMalloc(&w->rs_used, sizeof(unsigned)) == cudaSuccess &&
                cudaMemset(w->rs_used, 0, sizeof(unsigned)) == cudaSuccess && cudaMallocHost(&w->h_rs_used, sizeof(unsigned)) == cudaSuccess;
      if (!ok) { g_create_err = "allocation of the split-schedule buffers failed"; cudaGetLastError(); dg_world_destroy(w); return DG_E_CUDA; }
    }
  }
  if (cudaMalloc(&w->dropped, sizeof(unsigned)) != cudaSuccess || cudaMemset(w->dropped, 0, sizeof(unsigned)) != cudaSuccess) { g_create_err = "cudaMalloc of the contact-drop counter failed"; cudaGetLastError(); dg_world_destroy(w); return DG_E_CUDA; }
  {
    // ray_sensor ops: which ops, and the shared memory of dg_ray_kernel (the world poses of the moving shapes, per warp)
    const DevScene& hd = w->hs.dev;   // (host pointers)
    for (int k = 0; k < hd.nop; k++) if (hd.op_i[DG_OP_I_W * k] == OP_RAY_SENSOR) w->ray_ops.push_back(k);
    w->ray_smem = (size_t)kRayWarps * 12 * hd.nshw * sizeof(float);
    if (!w->ray_ops.empty() && w->ray_smem > 48 * 1024) {
      if (w->ray_smem > smem_cap || cudaFuncSetAttribute(dg_ray_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)w->ray_smem) != cudaSuccess) {
        g_create_err = "ray_sensor: the moving collision shapes do not fit in shared memory"; cudaGetLastError(); dg_world_destroy(w); return DG_E_NOMEM;
      }
    }
  }
  *out = w;
  return DG_OK;
}

void dg_world_destroy(DgWorld* w) {
  if (!w) return;
  DeviceGuard guard(w->device);
  if (w->d_ints) cudaFree(w->d_ints);
  if (w->d_floats) cudaFree(w->d_floats);
  if (w->gws) cudaFree(w->gws);
  if (w->dbg) cudaFree(w->dbg);
  if (w->dropped) cudaFree(w->dropped);
  if (w->carry) cudaFree(w->carry);
  if (w->rs_lists) cudaFree(w->rs_lists);
  if (w->rs_counts) cudaFree(w->rs_counts);
  if (w->ik_rec) cudaFree(w->ik_rec);
  if (w->aux) cudaStreamDestroy(w->aux);
  if (w->aux2) cudaStreamDestroy(w->aux2);
  if (w->ev_join2) cudaEventDestroy(w->ev_join2);
  if (w->ev_fork) cudaEventDestroy(w->ev_fork);
  if (w->ev_join) cudaEventDestroy(w->ev_join);
  if (w->ev_stat) cudaEventDestroy(w->ev_stat);
  if (w->graph_exec) cudaGraphExecDestroy(w->graph_exec);
  if (w->graph) cudaGraphDestroy(w->graph);
  if (w->cap) cudaStreamDestroy(w->cap);
  if (w->rs_used) cudaFree(w->rs_used);
  if (w->h_rs_used) cudaFreeHost(w->h_rs_used);
  delete w;
}

int64_t dg_query(const DgWorld* w, int key) {
  if (!w) return -1;
  const DevScene& d = w->dev;
  switch (key) {
    case DG_Q_STATE_SIZE: return d.S; case DG_Q_PARAM_SIZE: return d.P; case DG_Q_N_ACT: return d.n_act; case DG_Q_N_OBS: return d.n_obs;
    case DG_Q_N_REW: return d.n_rew; case DG_Q_N_TERM: return d.n_term; case DG_Q_N_ENVS: return w->n_envs; case DG_Q_TEAM: return w->team;
    case DG_Q_BLOCK_THREADS: return w->block_threads; case DG_Q_GRID_BLOCKS: return w->grid; case DG_Q_SMEM_BYTES: return (int64_t)w->smem;
    case DG_Q_WS_FLOATS: return d.w_total; case DG_Q_N_CAMERAS: return d.ncam; case DG_Q_LAUNCHES: return w->launches;
    case DG_Q_RS_ASHARED: return d.rs_ashared; case DG_Q_SOLVER: return d.solver; case DG_Q_MAX_CONTACTS: return d.maxc; case DG_Q_SPLIT: return w->split ? 1 : 0;
    case DG_Q_CONTACTS_DROPPED: {   // synchronises the device
      DeviceGuard guard(w->device); unsigned v = 0;
      if (!w->dropped || cudaMemcpy(&v, w->dropped, sizeof(unsigned), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
      return (int64_t)v;
    }
  }
  return -1;
}

int dg_bind_buffers(DgWorld* w, const DgBufferTable* t) {
  if (!w || !t) return DG_E_ARG;
  const DevScene& d = w->dev;
  if (!t->state || !t->param || (d.n_act && !t->action) || (d.n_obs && !t->obs) || (d.n_rew && !t->reward) || (d.n_term && !t->term)) { w->err = "dg_bind_buffers: a required buffer is NULL"; return DG_E_ARG; }
  w->buf = *t; w->bound = true;
  return DG_OK;
}

int dg_set_seed(DgWorld* w, uint32_t seed, int env_id_offset) {
  if (!w) return DG_E_ARG;
  w->seed = seed; w->env_off = env_id_offset;
  return DG_OK;
}

int dg_set_action_mask(DgWorld* w, const uint8_t* op_enabled, int n_ops) {
  if (!w || (n_ops > 0 && !op_enabled)) return DG_E_ARG;
  w->opmask[0] = w->opmask[1] = ~0ull;
  for (int k = 0; k < n_ops; k++) if (!op_enabled[k]) {
    // the mask has 128 bits; an action op beyond them cannot be switched off (compiler/scene.py refuses such scenes)
    if (k >= 128) { w->err = "dg_set_action_mask: ops at index >= 128 cannot be masked"; return DG_E_ARG; }
    w->opmask[k >> 6] &= ~(1ull << (k & 63));
  }
  return DG_OK;
}

int dg_init_state(DgWorld* w, void* stream) {
  if (!w) return DG_E_ARG;
  if (!w->bound) { w->err = "dg_init_state: buffers not bound"; return DG_E_UNBOUND; }
  DeviceGuard guard(w->device);
  w->launches++;
  dg_init_kernel<<<w->sm_count * 4, 256, 0, (cudaStream_t)stream>>>(w->dev, w->buf.state, w->buf.param, w->n_envs);
  CK(w, cudaGetLastError());
  return DG_OK;
}

static int run_step(DgWorld* w, int mode, const uint8_t* mask, void* stream) {
  if (!w) return DG_E_ARG;
  if (!w->bound) { w->err = "buffers not bound"; return DG_E_UNBOUND; }
  DeviceGuard guard(w->device);
  if (!guard.ok) { w->err = "cudaSetDevice failed"; cudaGetLastError(); return DG_E_CUDA; }
  LaunchArgs a{w->buf.state, w->buf.param, w->buf.action, w->buf.obs, w->buf.reward, w->buf.term, mask, w->n_envs, mode, w->seed, w->env_off, {w->opmask[0], w->opmask[1]}, w->gws, w->dbg, w->dropped,
               ST_ALL, nullptr, nullptr, nullptr, mode == 0 ? w->rs_used : nullptr, 0};
  cudaStream_t s = (cudaStream_t)stream;
  if (mode == 0 && w->split_ok && w->split_mode < 0 && w->dev.ncons == 0) {
    // adaptive schedule: share of environment sub-steps that needed the contact solver over the last period
    constexpr int kAdaptPeriod = 16;
    const cudaError_t qe = w->stat_pending ? cudaEventQuery(w->ev_stat) : cudaErrorNotReady;
    if (qe != cudaSuccess) cudaGetLastError();   // (cudaErrorNotReady is no error: keep it out of the next launch check)
    if (w->stat_pending && qe == cudaSuccess) {
      const double share = (double)*w->h_rs_used / ((double)kAdaptPeriod * std::max(w->dev.substeps, 1) * w->n_envs);
      if (share > 0.30) w->split = true; else if (share < 0.15) w->split = false;
      w->stat_pending = false;
    }
    if (++w->steps_in_period >= kAdaptPeriod && !w->stat_pending) {
      CK(w, cudaMemcpyAsync(w->h_rs_used, w->rs_used, sizeof(unsigned), cudaMemcpyDeviceToHost, s));
      CK(w, cudaMemsetAsync(w->rs_used, 0, sizeof(unsigned), s));
      CK(w, cudaEventRecord(w->ev_stat, s));
      w->stat_pending = true; w->steps_in_period = 0;
    }
  }
  const int nhot = mode == 1 ? w->dev.hot_start : 1;
  if (mode == 2 || !w->split || nhot < 1) { CK(w, launch_any(w, a, s)); return DG_OK; }
  // Split schedule of one step with n sub-steps (2 for the reference's settings, diy_gym.py:76-79):
  //   stage launch [add-on update, load | sub-step 0 up to the row-space system] -> sweeps ->
  //   stage launch [impulses + integration of sub-step k-1 | sub-step k up to its system] -> sweeps -> ... ->
  //   stage launch [impulses + integration of the last sub-step | link cache, state rows, sensors / rewards / terminals]
  // The sweeps of one sub-step are one launch of the sweep kernel per class: environments with <= 32 row positions (four per warp) on this
  // stream, the other classes beside them on the world's auxiliary streams (the one-per-warp class takes longest, so it should not
  // queue behind the others).
  const int nsub = std::max(w->dev.substeps, 1);
  a.carry = w->carry; a.rs_lists = w->rs_lists;
  // (DIYGym.reset of the masked environments: reset hooks + link cache as one fused launch, then every hot-start step takes the
  // same cut as a step, without add-on update; blocks without a masked environment return at once, the sweep kernel only sees
  // the listed ones)
  auto issue = [&](cudaStream_t q) -> int {
    if (mode == 1) { a.stages = ST_ALL; a.no_hot = 1; CK(w, launch_any(w, a, q)); a.no_hot = 0; }   // reset hooks + link cache, one fused launch
    for (int hot = 0; hot < nhot; hot++)
    for (int sub = 0; sub <= nsub; sub++) {
      const int first = mode == 0 ? ST_ACT : ST_LOAD;
      a.stages = (sub == 0 ? first : (ST_LOADC | ST_POST)) | (sub < nsub ? (ST_PRE | ST_SAVEC) : ST_END);
      a.rs_count = w->rs_counts + RS_NCLS * std::min(sub, nsub - 1);
      if (sub == 0) CK(w, cudaMemsetAsync(w->rs_counts, 0, RS_NCLS * (size_t)nsub * sizeof(int), q));
      CK(w, launch_any(w, a, q));
      if (sub == nsub) break;
      // the sweep classes of this sub-step side by side: class 0 on this stream, the others on the world's auxiliary streams
      CK(w, cudaEventRecord(w->ev_fork, q));
      int nl = 0;
      for (int c = RS_NCLS - 1; c >= 0; c--) {
        if (w->dev.rs_cls_r[c] <= 0) continue;
        const int* list = w->rs_lists + (size_t)c * w->n_envs;
        const SolveArgs sa{w->carry, w->gws, list, a.rs_count + c};
        cudaStream_t sq = c == 0 ? q : (c == 1 ? w->aux : w->aux2);
        if (c > 0) CK(w, cudaStreamWaitEvent(sq, w->ev_fork, 0));
        CK(w, solve_launch(c, w->dev, sa, w->n_envs, sq));
        if (c > 0) CK(w, cudaEventRecord(c == 1 ? w->ev_join : w->ev_join2, sq));
        nl++;
      }
      for (int c = 1; c < RS_NCLS; c++) if (w->dev.rs_cls_r[c] > 0) CK(w, cudaStreamWaitEvent(q, c == 1 ? w->ev_join : w->ev_join2, 0));   // (after class 0 is in the queue)
      w->launches += nl;
    }
    return DG_OK;
  };
  if (mode != 0 || !w->use_graph || w->dbg != nullptr) return issue(s);
  // graph replay of the step's launch sequence; the key holds everything the launches take by value
  const unsigned long long key[4] = {w->opmask[0], w->opmask[1], ((unsigned long long)w->seed << 32) | (unsigned)w->env_off, (unsigned long long)(uintptr_t)w->buf.state ^ ((unsigned long long)(uintptr_t)w->buf.action << 1)};
  if (!w->graph_valid || memcmp(key, w->graph_key, sizeof(key)) != 0) {
    if (w->graph_exec) { cudaGraphExecDestroy(w->graph_exec); w->graph_exec = nullptr; }
    if (w->graph) { cudaGraphDestroy(w->graph); w->graph = nullptr; }
    const int64_t l0 = w->launches;
    CK(w, cudaStreamBeginCapture(w->cap, cudaStreamCaptureModeThreadLocal));
    const int rc = issue(w->cap);
    cudaError_t ce = cudaStreamEndCapture(w->cap, &w->graph);
    w->launches = l0;
    if (rc != DG_OK || ce != cudaSuccess) { cudaGetLastError(); w->use_graph = 0; w->graph = nullptr; return issue(s); }   // capture refused: plain launches from now on
    if (cudaGraphInstantiate(&w->graph_exec, w->graph, 0) != cudaSuccess) { cudaGetLastError(); w->use_graph = 0; return issue(s); }
    memcpy(w->graph_key, key, sizeof(key)); w->graph_valid = true;
  }
  CK(w, cudaGraphLaunch(w->graph_exec, s));
  { int ncl = 0; for (int c = 0; c < RS_NCLS; c++) ncl += w->dev.rs_cls_r[c] > 0; w->launches += (nsub + 1) + ncl * nsub; }
  return DG_OK;
}
// Measurement aid: with `enable`, thread 0 of every block of the step kernel accumulates the cycles of each phase (barrier
// included) into a [grid][64] table keyed by (source line of the phase in dg_env.cuh) & 63; dg_debug_read copies it out
// (out[block * 64 + key], n <= grid * 64 entries) and clears it.  tools/phase_probe.py prints it.
int dg_debug_phase_cycles(DgWorld* w, int enable) {
  if (!w) return DG_E_ARG;
  DeviceGuard guard(w->device);
  if (!enable) { if (w->dbg) { cudaDeviceSynchronize(); cudaFree(w->dbg); w->dbg = nullptr; } return DG_OK; }
  if (!w->dbg) CK(w, cudaMalloc(&w->dbg, (size_t)w->grid * 64 * sizeof(unsigned long long)));
  CK(w, cudaMemset(w->dbg, 0, (size_t)w->grid * 64 * sizeof(unsigned long long)));
  return DG_OK;
}
int dg_debug_read(DgWorld* w, unsigned long long* out, int n) {
  if (!w || !out || !w->dbg || n > w->grid * 64) return DG_E_ARG;
  DeviceGuard guard(w->device);
  CK(w, cudaDeviceSynchronize());
  CK(w, cudaMemcpy(out, w->dbg, (size_t)n * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  CK(w, cudaMemset(w->dbg, 0, (size_t)w->grid * 64 * sizeof(unsigned long long)));
  return DG_OK;
}
// The step / reset / observe launches, then the ray_sensor ops (one launch of dg_ray_kernel on the same stream, after whichever
// schedule the step took: it reads the link cache the step left in the state rows).  A reset only casts the masked environments' rays.
static int run(DgWorld* w, int mode, const uint8_t* mask, void* stream) {
  const int rc = run_step(w, mode, mask, stream);
  if (rc != DG_OK || w->ray_ops.empty()) return rc;
  DeviceGuard guard(w->device);
  w->launches++;
  dg_ray_kernel<<<(w->n_envs + kRayWarps - 1) / kRayWarps, 32 * kRayWarps, w->ray_smem, (cudaStream_t)stream>>>(w->dev, w->buf.state, w->buf.obs, mode == 1 ? mask : nullptr, w->n_envs);
  CK(w, cudaGetLastError());
  return DG_OK;
}
int dg_step(DgWorld* w, void* stream) { return run(w, 0, nullptr, stream); }

int dg_body_dynamics(DgWorld* w, int body, int link, const float point[3], const float* q_dev, const float* qd_dev, const float* qdd_dev,
                     float* jac_dev, float* mass_dev, float* tau_dev, void* stream) {
  if (!w) return DG_E_ARG;
  if (!w->bound) { w->err = "dg_body_dynamics: buffers not bound"; return DG_E_UNBOUND; }
  const DevScene& hd = w->hs.dev;   // (host pointers)
  if (body < 0 || body >= hd.nb) { w->err = "dg_body_dynamics: no such body"; return DG_E_ARG; }
  const int* bi = hd.body_i + DG_BODY_I_W * body;
  DynArgs a;
  a.body = body; a.link = link; a.n = (bi[0] == 2 ? 6 : 0) + bi[4]; a.nl = bi[2] + 1;
  if (bi[0] == 0 || a.n == 0) { w->err = "dg_body_dynamics: the body has no degrees of freedom"; return DG_E_ARG; }
  if (a.n > DG_DYN_MAXN) { w->err = "dg_body_dynamics: the body has " + std::to_string(a.n) + " generalized coordinates, more than " + std::to_string((int)DG_DYN_MAXN); return DG_E_ARG; }
  if (link < -1 || link >= bi[2]) { w->err = "dg_body_dynamics: no such link"; return DG_E_ARG; }
  for (int i = 0; i < 3; i++) a.point[i] = point ? point[i] : 0.f;
  a.q = q_dev; a.qd = qd_dev; a.qdd = qdd_dev; a.jac = jac_dev; a.mass = mass_dev; a.tau = tau_dev;
  if (!jac_dev && !mass_dev && !tau_dev) return DG_OK;
  DeviceGuard guard(w->device);
  const size_t smem = (size_t)kDynWarps * dyn_scratch_floats(a.nl, a.n) * sizeof(float);
  if (smem > 48 * 1024) CK(w, cudaFuncSetAttribute(dg_dyn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  w->launches++;
  dg_dyn_kernel<<<(w->n_envs + kDynWarps - 1) / kDynWarps, 32 * kDynWarps, smem, (cudaStream_t)stream>>>(w->dev, a, w->buf.state, w->buf.param, w->n_envs);
  CK(w, cudaGetLastError());
  return DG_OK;
}

int dg_body_ik(DgWorld* w, int body, int link, const float* target_pos_dev, const float* target_orn_dev, const float* q0_dev,
               const float* limits_dev, int max_iters, float threshold, float* q_out_dev, float* err_dev, void* stream) {
  if (!w) return DG_E_ARG;
  if (!w->bound) { w->err = "dg_body_ik: buffers not bound"; return DG_E_UNBOUND; }
  const DevScene& hd = w->hs.dev;   // (host pointers)
  if (body < 0 || body >= hd.nb) { w->err = "dg_body_ik: no such body"; return DG_E_ARG; }
  const int* bi = hd.body_i + DG_BODY_I_W * body;
  const int ndb = bi[4];
  if (bi[0] == 0 || ndb == 0) { w->err = "dg_body_ik: the body has no degrees of freedom"; return DG_E_ARG; }
  if (ndb > DG_IK_MAX_ND) { w->err = "dg_body_ik: the body has " + std::to_string(ndb) + " degrees of freedom, more than " + std::to_string((int)DG_IK_MAX_ND); return DG_E_ARG; }
  if (link < 0 || link >= bi[2]) { w->err = "dg_body_ik: no such link"; return DG_E_ARG; }
  if (max_iters < 1) { w->err = "dg_body_ik: max_iters must be at least 1"; return DG_E_ARG; }
  if (!(threshold >= 0.f)) { w->err = "dg_body_ik: threshold must be a number >= 0"; return DG_E_ARG; }
  if (!target_pos_dev || !q_out_dev) { w->err = "dg_body_ik: target_pos and q_out are required"; return DG_E_ARG; }
  DevScene d = w->dev;   // (device pointers)
  IkArgs a;
  a.body = body; a.link = bi[1] + link; a.use_orn = target_orn_dev != nullptr;
  a.s_q = DG_SO(&d, S_Q); a.s_bpos = DG_SO(&d, S_BPOS); a.s_bquat = DG_SO(&d, S_BQUAT);
  a.seed_floats = ik_scene(d, max_iters, threshold);
  a.rec_stride = a.seed_floats + d.ik_stride;
  a.tpos = target_pos_dev; a.torn = target_orn_dev; a.q0 = q0_dev; a.lim = limits_dev; a.q_out = q_out_dev; a.err = err_dev;
  DeviceGuard guard(w->device);
  if (!w->ik_rec) CK(w, cudaMalloc(&w->ik_rec, (size_t)w->n_envs * a.rec_stride * sizeof(float)));
  a.rec = w->ik_rec;
  const size_t smem = (size_t)(((DG_LINK_I_W * d.nl + 3) & ~3) + (DG_LINK_F_W + 16) * d.nl) * sizeof(float);
  const cudaStream_t s = (cudaStream_t)stream;
  // the split of ik_solve_any: register-resident solves up to 12 DoF, the generic one above
  auto launch = ndb <= 6 ? (a.use_orn ? ik_launch<6, 6> : ik_launch<6, 3>) : ndb <= 12 ? (a.use_orn ? ik_launch<12, 6> : ik_launch<12, 3>) : ik_launch<0, 0>;
  w->launches++;
  CK(w, launch(d, a, w->buf.state, w->n_envs, smem, s));
  return DG_OK;
}
int dg_reset(DgWorld* w, const uint8_t* mask_dev, void* stream) { return run(w, 1, mask_dev, stream); }
int dg_observe(DgWorld* w, void* stream) { return run(w, 2, nullptr, stream); }

static int render_any(DgWorld* w, int cam, void* rgb_dev, bool u8, float* depth_dev, float* seg_dev, void* stream) {
  if (!w || !rgb_dev || !depth_dev) return DG_E_ARG;
  if (!w->bound) { w->err = "dg_render: buffers not bound"; return DG_E_UNBOUND; }
  const DevScene& d = w->dev;
  if (cam < 0 || cam >= d.ncam) { w->err = "dg_render: no such camera"; return DG_E_ARG; }
  DeviceGuard guard(w->device);
  const int* ci = w->hs.dev.cam_i + DG_CAM_I_W * cam;
  // patches of 8 x 8 pixels (two rays per lane), one per warp at a time; images too small to give every warp of a block a dozen of
  // those take 8 x 4 patches (measured: 50 x 50 is 14 % slower with the large ones, 200 x 200 12 % faster)
  const int nh = ((ci[1] + 7) / 8) * ((ci[2] + 7) / 8) >= 96 ? 2 : 1;
  int tiles_x = (ci[1] + 7) / 8, tiles_y = (ci[2] + 4 * nh - 1) / (4 * nh);
  size_t smem = ((size_t)std::max(d.nv, 1) * VS_W + (size_t)((d.nv + 3) & ~3) + (size_t)(d.nv + 31) / 32 + 8) * sizeof(float);
  const int ncw = (d.nv + 31) / 32;   // candidate words per patch the kernel keeps in registers: 1, 2 or 4 (then a per-shape tail)
  // (compiled for 3 resident blocks per SM, 80 registers; 4 blocks / 64 registers spills in the per-block set-up and measured
  // slower: 1.10 vs 1.03 ms per 4096 x 200 x 200 render)
  using RenderFn = void (*)(DevScene, const float*, const float*, int, float*, float*, float*, int, int, int);
  static const RenderFn table[2][2][3] = {
      {{dg_render_kernel<1, 1, false>, dg_render_kernel<2, 1, false>, dg_render_kernel<4, 1, false>}, {dg_render_kernel<1, 2, false>, dg_render_kernel<2, 2, false>, dg_render_kernel<4, 2, false>}},
      {{dg_render_kernel<1, 1, true>, dg_render_kernel<2, 1, true>, dg_render_kernel<4, 1, true>}, {dg_render_kernel<1, 2, true>, dg_render_kernel<2, 2, true>, dg_render_kernel<4, 2, true>}}};
  RenderFn kern = table[u8 ? 1 : 0][nh - 1][ncw <= 1 ? 0 : (ncw == 2 ? 1 : 2)];
  if (smem > 48 * 1024) { CK(w, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)w->smem_cap)); }
  // blocks per environment: one when the batch alone fills the GPU a few times over, else enough groups of tiles to do so
  int groups = std::max(1, std::min((tiles_x * tiles_y + 7) / 8, (8 * w->sm_count + w->n_envs - 1) / w->n_envs));
  w->launches++;
  kern<<<w->n_envs * groups, 256, smem, (cudaStream_t)stream>>>(w->dev, w->buf.state, w->buf.param, cam, reinterpret_cast<float*>(rgb_dev), depth_dev, seg_dev, tiles_x, tiles_y, groups);
  CK(w, cudaGetLastError());
  return DG_OK;
}
int dg_render_seg(DgWorld* w, int cam, float* rgb_dev, float* depth_dev, float* seg_dev, void* stream) { return render_any(w, cam, rgb_dev, false, depth_dev, seg_dev, stream); }
int dg_render_u8(DgWorld* w, int cam, uint8_t* rgb_dev, float* depth_dev, float* seg_dev, void* stream) { return render_any(w, cam, rgb_dev, true, depth_dev, seg_dev, stream); }
int dg_render(DgWorld* w, int cam, float* rgb_dev, float* depth_dev, void* stream) { return dg_render_seg(w, cam, rgb_dev, depth_dev, nullptr, stream); }

int dg_step_host(DgWorld* w, const float* action_host, float* obs_host, float* reward_host, uint8_t* term_host, void* stream) {
  if (!w) return DG_E_ARG;
  if (!w->bound) { w->err = "dg_step_host: buffers not bound"; return DG_E_UNBOUND; }
  DeviceGuard guard(w->device);
  const DevScene& d = w->dev; cudaStream_t s = (cudaStream_t)stream; size_t n = (size_t)w->n_envs;
  if (d.n_act && action_host) CK(w, cudaMemcpyAsync(w->buf.action, action_host, n * d.n_act * sizeof(float), cudaMemcpyHostToDevice, s));
  int rc = dg_step(w, stream);
  if (rc != DG_OK) return rc;
  if (d.n_obs && obs_host) CK(w, cudaMemcpyAsync(obs_host, w->buf.obs, n * d.n_obs * sizeof(float), cudaMemcpyDeviceToHost, s));
  if (d.n_rew && reward_host) CK(w, cudaMemcpyAsync(reward_host, w->buf.reward, n * d.n_rew * sizeof(float), cudaMemcpyDeviceToHost, s));
  if (d.n_term && term_host) CK(w, cudaMemcpyAsync(term_host, w->buf.term, n * d.n_term, cudaMemcpyDeviceToHost, s));
  CK(w, cudaStreamSynchronize(s));
  return DG_OK;
}

}  // extern "C"

// ---------------------------------------------------------------- FP32 FMA peak (roofline denominator) ------------
namespace dg {
__global__ void dg_fma_peak_kernel(float* out, int iters) {
  float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f, a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
  const float b = 0.999f, c = 1e-4f;
  for (int i = 0; i < iters; i++) {
    a0 = fmaf(a0, b, c); a1 = fmaf(a1, b, c); a2 = fmaf(a2, b, c); a3 = fmaf(a3, b, c);
    a4 = fmaf(a4, b, c); a5 = fmaf(a5, b, c); a6 = fmaf(a6, b, c); a7 = fmaf(a7, b, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}
}  // namespace dg

extern "C" int dg_measure_fp32_peak(int device, double* tflops_out) {
  if (!tflops_out) return DG_E_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return DG_E_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return DG_E_CUDA;
  const int blocks = prop.multiProcessorCount * 8, threads = 512, iters = 1 << 14;
  float* out = nullptr;
  if (cudaMalloc(&out, (size_t)blocks * threads * sizeof(float)) != cudaSuccess) return DG_E_CUDA;
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 5; rep++) {
    cudaEventRecord(e0);
    dg::dg_fma_peak_kernel<<<blocks, threads>>>(out, iters);
    cudaEventRecord(e1);
    if (cudaEventSynchronize(e1) != cudaSuccess) { cudaFree(out); return DG_E_CUDA; }
    float ms = 0.f; cudaEventElapsedTime(&ms, e0, e1);
    double tf = 2.0 * 8.0 * (double)iters * blocks * threads / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
  *tflops_out = best;
  return DG_OK;
}
#else
}  // namespace dg
#endif  // !DG_STEP_T
