// kernels.cuh — hand-written sm_100a kernels of the PARSDMM iteration.
//
// Kernels by reference routine (all HBM-bandwidth bound; one pass over their operands):
//   k_spmv_tile       (spmv_tile.cuh) the same SpMV / CG prologue for 3-D stencils as a plane sweep with TMA-staged tiles
//   k_spmv            CDS_MVp_MT.jl:9-25 + Ax_CDS_MT (argmin_x.jl:72-78) [+ dot(p,Ap), cg.jl:88]; Q as CDS arrays
//                     or as verified stencil-class tables (k_class_extract / k_class_verify / k_class_axpy)
//   k_cg_init         argmin_x.jl:33-37 + cg.jl:47-76   (one SpMV instead of the reference's two)
//   k_cg_xr / k_cg_p  cg.jl:86-114
//   k_rhs             rhs_compose.jl:24-36 (+ the dual residual of the previous iteration, update_y_l.jl:82-84)
//   k_yl_multi, k_yl  update_y_l.jl:39-94 with the projector / prox fused in, the six reductions of
//                     adapt_rho_gamma.jl:41-53, the snapshots of PARSDMM.jl:164-207 and (distance term) the
//                     obj / evol_x sums of PARSDMM.jl:140-145
//   k_rdual, k_stop   stand-alone versions of the two fused reductions (Minkowski, feasibility_only, last iteration)
//   k_cds_axpy        CDS_scaled_add!.jl:16-22 / Q assembly PARSDMM_initialize.jl:223-229 (array form of Q)
//   k_sparse_*        custom_TD_OP (setup_constraints.jl:70-72): explicit sparse operators
//   k_l1_pass         project_l1_Duchi!.jl:33-46 replaced by a sort-free Newton (Michelot) threshold search
//   k_radix_hist/...  project_cardinality!.jl:18-19 replaced by a radix select with index-ordered ties
//   k_card_fiber_*    project_cardinality!.jl:23-113 (fiber modes);  k_resample_nn  PARSDMM_multi_level.jl:61-82
#pragma once
#include "common.cuh"
#include "ops.cuh"

namespace sipb {

constexpr int kMaxDiag = 32;   // max diagonals of Q handled by the SpMV kernels
constexpr int kMaxSets = 16;   // max terms (incl. the distance term) per problem

// =============================================================================================
// CDS SpMV
// =============================================================================================
template <typename T>
struct SpmvArgs {
  const T* R;        // [nd][ld] diagonals, row aligned (R[j*ld + r] = A[r, r+off_j]), zero padded
  i64 ld;            // leading dimension (multiple of 16 elements)
  int nd;
  i64 off[kMaxDiag]; // offsets in accumulation order (Q_offsets order of the reference)
  i64 N;             // local rows
  i64 row0;          // global index of local row 0 (slabs); 0 on a single GPU
  i64 Nglob;         // global rows
  const T* x;        // x[r + off] addresses local row r (+halo), same indexing as y
  T* y;
  const T* x_lo;     // slabs, peer path: the lower / upper neighbour's vector (owned start), read over NVLink
  const T* x_hi;     //   instead of a local halo copy; null => local halo planes
  i64 n_lo;          // rows owned by the lower neighbour
  // stencil-class form of the matrix (see RowClass below): tab[cls*nd + j] replaces R[j*ld + r]; null => R
  const T* tab;
  unsigned gn[3];    // grid
  unsigned npts;     // grid points (rows per Minkowski half)
  // host-prepared constants of the class-form fast path (spmv_rows): 32-bit offsets, which of them keep 16-byte
  // alignment, the widest offset, and multiply-shift constants for the divisions by gn[0], gn[1]
  int fast;                     // 1: available (class form, nd <= kFastDiag, offsets fit 31 bits)
  int off32[8];
  unsigned amask;               // bit j: off[j] % VW == 0
  i64 maxoff;
  unsigned div_m[2];
  int div_s[2];
};
// floor(n / d) for n < 2^31 by multiply-shift (Granlund & Montgomery: m = ceil(2^(31+l) / d), l = ceil(log2 d))
__device__ __forceinline__ unsigned fast_div31(unsigned n, unsigned m, int s) {
  return (unsigned)(((unsigned long long)n * m) >> s);
}

// ---------------------------------------------------------------------------------------------
// Stencil classes.  Every AtA the reference builds from its constant-coefficient difference operators
// (get_TD_operator.jl) — and therefore Q = sum rho_i AtA_i, which is updated row-uniformly
// (Q_update!.jl:45-49) — holds the same values on all rows that agree on {first, interior, last} along each
// grid axis (and on the Minkowski half): 27 (54) classes.  The solver VERIFIES this on the uploaded CDS arrays
// and then keeps one row per class instead of N: the SpMV streams x and y only ((nd+2) -> 2 words per row)
// and performs exactly the multiply-adds, in exactly the order, of the array form — bit-identical results.
// Matrices that fail the check (custom operators) stay in array form.
// ---------------------------------------------------------------------------------------------
constexpr int kMaxClasses = 54;
template <typename T> __device__ __forceinline__ unsigned long long value_bits(T v);
template <> __device__ __forceinline__ unsigned long long value_bits<float>(float v) { return __float_as_uint(v); }
template <> __device__ __forceinline__ unsigned long long value_bits<double>(double v) {
  return (unsigned long long)__double_as_longlong(v);
}
__device__ __forceinline__ unsigned axis_class(unsigned idx, unsigned n) {
  return idx == 0u ? 0u : (idx == n - 1u ? 2u : 1u);
}
// class of global row g
__device__ __forceinline__ unsigned row_class(i64 g, const unsigned (&n)[3], unsigned npts) {
  const unsigned half = g >= (i64)npts ? 1u : 0u;
  const unsigned c = (unsigned)(g - (i64)half * npts);
  const unsigned q = c / n[0];
  const unsigned i = c - q * n[0];
  const unsigned kk = q / n[1];
  const unsigned j = q - kk * n[1];
  return ((half * 3u + axis_class(kk, n[2])) * 3u + axis_class(j, n[1])) * 3u + axis_class(i, n[0]);
}
// classes of W consecutive global rows; returns true when all W are equal (=> cls[0])
template <int W>
__device__ __forceinline__ bool row_classes(i64 g, const unsigned (&n)[3], unsigned npts, unsigned (&cls)[W]) {
  const unsigned half = g >= (i64)npts ? 1u : 0u;
  const unsigned c = (unsigned)(g - (i64)half * npts);
  const unsigned q = c / n[0];
  const unsigned i = c - q * n[0];
  if (i + (unsigned)W <= n[0] && (half || c + (unsigned)W <= npts)) {
    const unsigned kk = q / n[1];
    const unsigned j = q - kk * n[1];
    const unsigned base = ((half * 3u + axis_class(kk, n[2])) * 3u + axis_class(j, n[1])) * 3u;
    bool same = true;
#pragma unroll
    for (int e = 0; e < W; ++e) {
      cls[e] = base + axis_class(i + e, n[0]);
      same = same && cls[e] == cls[0];
    }
    return same;
  }
#pragma unroll
  for (int e = 0; e < W; ++e) cls[e] = row_class(g + e, n, npts);
  return false;
}

// true when the calling block (grid-stride over vector groups of W rows) owns rows within `halo` rows of either
// end of the local slab — only those rows are read by the neighbours, so only these blocks need
// system-scope fences / version waits on the peer path
__device__ __forceinline__ void block_touches_ends(i64 N, i64 halo, int W, bool& lo, bool& hi) {
  const i64 first = (i64)blockIdx.x * blockDim.x * W;
  const i64 sweep = (i64)gridDim.x * blockDim.x * W;
  const i64 nsweeps = first < N ? (N - 1 - first) / sweep : 0;
  const i64 last = min(N, first + nsweeps * sweep + (i64)blockDim.x * W);
  lo = first < halo;
  hi = last > N - halo;
}

// element x[idx] for a local index that may fall into a neighbour's slab
template <typename T>
__device__ __forceinline__ T spmv_x(const SpmvArgs<T>& a, i64 idx) {
  if (idx < 0 && a.x_lo) return __ldcg(a.x_lo + (a.n_lo + idx));
  if (idx >= a.N && a.x_hi) return __ldcg(a.x_hi + (idx - a.N));
  return a.x[idx];
}

// acc[e] for VW consecutive rows starting at r (vector path; r % VW == 0, r + VW <= N)
// tab: the class table staged in shared memory (null => array form)
template <typename T>
__device__ __forceinline__ void spmv_rows_vec(const SpmvArgs<T>& a, const T* tab, i64 r, T (&acc)[Vec<T>::W]) {
  constexpr int VW = Vec<T>::W;
#pragma unroll
  for (int e = 0; e < VW; ++e) acc[e] = (T)0;
  const i64 g = a.row0 + r;
  unsigned cls[VW];
  bool same = false;
  if (tab) same = row_classes<VW>(g, a.gn, a.npts, cls);
#pragma unroll 4
  for (int j = 0; j < a.nd; ++j) {
    T rv[VW], xv[VW];
    if (tab) {
      if (same) {
        const T q = tab[cls[0] * a.nd + j];
#pragma unroll
        for (int e = 0; e < VW; ++e) rv[e] = q;
      } else {
#pragma unroll
        for (int e = 0; e < VW; ++e) rv[e] = tab[cls[e] * a.nd + j];
      }
    } else {
      vload_stream<T>(a.R + (i64)j * a.ld + r, rv);
    }
    const i64 o = a.off[j];
    const i64 gc = g + o;
    const i64 li = r + o;
    const bool local = (a.x_lo == nullptr && a.x_hi == nullptr) || (li >= 0 && li + VW <= a.N);
    if (gc >= 0 && gc + VW <= a.Nglob && local) {
      const T* xp = a.x + li;
      if ((o & (VW - 1)) == 0) {
        vload<T>(xp, xv);
      } else {
#pragma unroll
        for (int e = 0; e < VW; ++e) xv[e] = xp[e];
      }
    } else {
#pragma unroll
      for (int e = 0; e < VW; ++e) {
        const i64 ge = gc + e;
        xv[e] = (ge >= 0 && ge < a.Nglob) ? spmv_x<T>(a, li + e) : (T)0;
      }
    }
#pragma unroll
    for (int e = 0; e < VW; ++e) acc[e] = acc[e] + rv[e] * xv[e];
  }
}

template <typename T>
__device__ __forceinline__ T spmv_row_scalar(const SpmvArgs<T>& a, const T* tab, i64 r) {
  T acc = (T)0;
  const i64 g = a.row0 + r;
  const unsigned cls = tab ? row_class(g, a.gn, a.npts) : 0u;
  for (int j = 0; j < a.nd; ++j) {
    const i64 gc = g + a.off[j];
    if (gc >= 0 && gc < a.Nglob) {
      const T q = tab ? tab[cls * a.nd + j] : a.R[(i64)j * a.ld + r];
      acc = acc + q * spmv_x<T>(a, r + a.off[j]);
    }
  }
  return acc;
}

// stage the class table in shared memory (all threads of the block call this)
template <typename T>
__device__ __forceinline__ const T* spmv_stage_table(const SpmvArgs<T>& a, T* tab_s) {
  if (!a.tab) return nullptr;
  for (int q = threadIdx.x; q < kMaxClasses * a.nd; q += blockDim.x) tab_s[q] = a.tab[q];
  __syncthreads();
  return tab_s;
}

// Fast path of the class form: a group of VW rows whose stencil stays inside the vector (and inside the local
// slab on the peer path) needs no range checks: offsets live in registers (kFastDiag compile-time slots,
// 32-bit), the matrix values come from the shared-memory table (mostly broadcast loads) and the loop over the
// diagonals is fully unrolled.  The selection is warp-uniform except near the two ends of the vector (a
// per-class selection would split almost every warp: each grid line has two boundary groups).  Groups near
// the ends, and matrices with nd > kFastDiag, take the generic routine; both evaluate the same expression
// acc = acc + q_j * x[r + off_j], j = 0..nd-1.
constexpr int kFastDiag = 8;
template <typename T>
__device__ __forceinline__ void spmv_rows(const SpmvArgs<T>& a, const T* tab, i64 r, T (&acc)[Vec<T>::W]) {
  constexpr int VW = Vec<T>::W;
  if (a.fast) {
    const i64 g = a.row0 + r;
    const bool peer = a.x_lo != nullptr || a.x_hi != nullptr;
    const bool inside = g >= a.maxoff && g + VW + a.maxoff <= a.Nglob &&
                        (!peer || (r >= a.maxoff && r + VW + a.maxoff <= a.N));
    if (inside) {        // warp-uniform except in the first / last plane of the vector
      const unsigned n0 = a.gn[0], n1 = a.gn[1];
      const unsigned half = g >= (i64)a.npts ? 1u : 0u;
      const unsigned c = (unsigned)(g - (i64)half * a.npts);
      const unsigned q = fast_div31(c, a.div_m[0], a.div_s[0]);
      const unsigned i = c - q * n0;
      unsigned tq[VW];      // first table entry of each row's class
      if (i + (unsigned)VW <= n0 && (half || c + (unsigned)VW <= a.npts)) {     // the group stays on one grid line
        const unsigned kk = fast_div31(q, a.div_m[1], a.div_s[1]);
        const unsigned j = q - kk * n1;
        const unsigned base = ((half * 3u + axis_class(kk, a.gn[2])) * 3u + axis_class(j, n1)) * 3u;
#pragma unroll
        for (int e = 0; e < VW; ++e) tq[e] = (base + axis_class(i + e, n0)) * (unsigned)a.nd;
      } else {
#pragma unroll
        for (int e = 0; e < VW; ++e) tq[e] = row_class(g + e, a.gn, a.npts) * (unsigned)a.nd;
      }
      const T* xr = a.x + r;
#pragma unroll
      for (int e = 0; e < VW; ++e) acc[e] = (T)0;
#pragma unroll
      for (int j = 0; j < kFastDiag; ++j) {
        if (j < a.nd) {
          T xv[VW];
          const T* xp = xr + a.off32[j];
          if ((a.amask >> j) & 1u) {
            vload<T>(xp, xv);
          } else {
#pragma unroll
            for (int e = 0; e < VW; ++e) xv[e] = xp[e];
          }
#pragma unroll
          for (int e = 0; e < VW; ++e) acc[e] = acc[e] + tab[tq[e] + j] * xv[e];
        }
      }
      return;
    }
  }
  spmv_rows_vec<T>(a, tab, r, acc);
}

// y = A x  and (DOT) partial sum of x.*y  -> out_dot[0]
// cd.on: p's neighbour planes are read through peer pointers (after p_wait) and the partial of p.Ap is
// published to every rank's mailbox instead of being written to out_dot.
template <typename T, bool DOT>
__global__ void __launch_bounds__(kThreads, 6) k_spmv(SpmvArgs<T> a, RedScratch rs, double* out_dot,
                                                   const int* __restrict__ done_flag, const __grid_constant__ CommDev cd) {
  if (done_flag && *done_flag) return;
  constexpr int VW = Vec<T>::W;
  __shared__ T tab_s[kMaxClasses * kMaxDiag];
  const T* tab = spmv_stage_table<T>(a, tab_s);
  double d[1] = {0.0};
  const i64 nvec = a.N / VW;
  if (cd.on && (a.x_lo || a.x_hi)) {
    // rows within one plane (= max |offset|) of the slab ends read the neighbours' p: only the blocks that
    // own such rows wait for the neighbours' version flag
    i64 halo = 0;
    for (int j = 0; j < a.nd; ++j) halo = max(halo, a.off[j] < 0 ? -a.off[j] : a.off[j]);
    bool lo, hi;
    block_touches_ends(a.N, halo, VW, lo, hi);
    p_wait(cd, lo, hi);
  }
  for (i64 iv = (i64)blockIdx.x * blockDim.x + threadIdx.x; iv < nvec; iv += (i64)gridDim.x * blockDim.x) {
    const i64 r = iv * VW;
    T acc[VW];
    spmv_rows<T>(a, tab, r, acc);
    vstore<T>(a.y + r, acc);
    if (DOT) {
      T xc[VW];
      vload<T>(a.x + r, xc);
#pragma unroll
      for (int e = 0; e < VW; ++e) d[0] += (double)xc[e] * (double)acc[e];
    }
  }
  // tail rows
  for (i64 r = nvec * VW + (i64)blockIdx.x * blockDim.x + threadIdx.x; r < a.N; r += (i64)gridDim.x * blockDim.x) {
    const T acc = spmv_row_scalar<T>(a, tab, r);
    a.y[r] = acc;
    if (DOT) d[0] += (double)a.x[r] * (double)acc;
  }
  if (DOT) {
    if (grid_sum<1>(d, rs)) {
      if (cd.on) mail_allreduce<1>(cd, d, out_dot);      // the global p.Ap is in place when the kernel ends
      else if (threadIdx.x == 0) out_dot[0] = d[0];
    }
  }
}

// =============================================================================================
// CG (device-resident scalars; the host only polls `done`)
// =============================================================================================
struct CgState {
  double bb;        // sum b^2
  double rr;        // gamma = dot(r,r) of the current residual
  double pAp;
  double rr_new;
  double tol;       // value of a T
  double tol_prev;  // x_solve_tol_ref carried between PARSDMM iterations (argmin_x.jl:33-37)
  double relres;    // resvec[lastIter]
  int iter;         // lastIter
  int done;
  int flag;         // 0 / -1 / -2 / -9 as cg.jl:29-37
  int maxit;
  int parsdmm_it;   // i of PARSDMM.jl:97 (selects the i<3 tolerance rule); 0 => plain cg with tol given
  int loops;        // loop iterations actually executed (speculative launches after `done` return at once)
};

}  // namespace sipb
#include "spmv_tile.cuh"     // tiled, TMA-staged SpMV / CG prologue for 3-D stencils (uses SpmvArgs, CgState, CommDev)
namespace sipb {

// r = b - Q x ; p = r ; (x_old = x) ; sums bb, rr
template <typename T>
__global__ void __launch_bounds__(kThreads) k_cg_init(SpmvArgs<T> a, const T* __restrict__ b, T* __restrict__ r,
                                                      T* __restrict__ p, T* __restrict__ x_old, RedScratch rs,
                                                      CgState* st, const __grid_constant__ CommDev cd) {
  constexpr int VW = Vec<T>::W;
  __shared__ T tab_s[kMaxClasses * kMaxDiag];
  const T* tab = spmv_stage_table<T>(a, tab_s);
  double d[2] = {0.0, 0.0};
  const i64 nvec = a.N / VW;
  for (i64 iv = (i64)blockIdx.x * blockDim.x + threadIdx.x; iv < nvec; iv += (i64)gridDim.x * blockDim.x) {
    const i64 row = iv * VW;
    T acc[VW], bv[VW], rv[VW];
    spmv_rows<T>(a, tab, row, acc);
    vload_stream<T>(b + row, bv);
#pragma unroll
    for (int e = 0; e < VW; ++e) {
      rv[e] = bv[e] - acc[e];
      d[0] += (double)bv[e] * (double)bv[e];
      d[1] += (double)rv[e] * (double)rv[e];
    }
    vstore<T>(r + row, rv);
    vstore<T>(p + row, rv);
    if (x_old) {
      T xc[VW];
      vload<T>(a.x + row, xc);
      vstore<T>(x_old + row, xc);
    }
  }
  for (i64 row = nvec * VW + (i64)blockIdx.x * blockDim.x + threadIdx.x; row < a.N;
       row += (i64)gridDim.x * blockDim.x) {
    const T acc = spmv_row_scalar<T>(a, tab, row);
    const T bv = b[row];
    const T rv = bv - acc;
    d[0] += (double)bv * (double)bv;
    d[1] += (double)rv * (double)rv;
    r[row] = rv;
    p[row] = rv;
    if (x_old) x_old[row] = a.x[row];
  }
  bool sys = false;
  if (cd.on) {
    i64 halo = 0;
    for (int j = 0; j < a.nd; ++j) halo = max(halo, a.off[j] < 0 ? -a.off[j] : a.off[j]);
    bool lo, hi;
    block_touches_ends(a.N, halo, VW, lo, hi);
    sys = lo || hi;            // only boundary rows of p are read by the neighbours
  }
  if (grid_sum<2>(d, rs, sys)) {
    if (cd.on) {
      mail_publish<2>(cd, d);                   // (the boundary planes of r were fenced at system scope: k_p_halo_init reads them)
    } else if (threadIdx.x == 0) {
      st->bb = d[0];
      st->rr = d[1];
    }
  }
}

// one-thread collector of a peer-memory reduction (between the producing and the consuming kernel)
template <int K>
__global__ void k_mail_collect(const __grid_constant__ CommDev cd, double* dst, const int* done_flag) {
  if (done_flag && *done_flag) return;
  mail_collect<K>(cd, dst);
}

// scalar epilogue of the init (after the optional all-reduce of bb, rr): tolerance rule of
// argmin_x.jl:33-37 and the early exits of cg.jl:47,73-76
template <typename T>
__global__ void k_cg_init_fin(CgState* st, const __grid_constant__ CommDev cd, LoopCond lc) {
  if (cd.on) mail_collect<2>(cd, &st->bb);       // bb, rr are adjacent
  loop_set(lc, true);
  const T nb = (T)sqrt(st->bb);
  const T nr = (T)sqrt(st->rr);
  st->iter = 0;
  st->loops = 0;
  st->done = 0;
  st->flag = -1;
  st->relres = 0.0;
  if (st->parsdmm_it > 0) {
    // TF(max(0.1*norm(Qx-rhs)/norm(rhs), 10*eps(TF))) evaluated in Float64; Julia's max propagates NaN
    const double ratio = 0.1 * (double)nr / (double)nb;
    const double floor_ = (double)((T)10 * (T)Eps<T>::v);
    double cur = (ratio != ratio) ? ratio : (ratio > floor_ ? ratio : floor_);
    if (st->parsdmm_it >= 3) {
      const double prev = st->tol_prev;
      cur = (cur != cur || prev != prev) ? (cur != cur ? cur : prev) : (cur < prev ? cur : prev);
    }
    st->tol = (double)(T)cur;
    st->tol_prev = st->tol;
  }
  if (nb == (T)0) {            // cg.jl:47: rhs == 0 -> zeros, flag -9, iter 0 (x is zero-filled afterwards)
    st->flag = -9;
    st->done = 1;
    loop_set(lc, false);
    return;
  }
  if (nr / nb <= (T)st->tol) {  // cg.jl:73-76
    st->flag = 0;
    st->iter = 1;
    st->done = 1;
    loop_set(lc, false);
  }
  if (st->maxit < 1) {          // for iter = 1:maxIter never runs
    st->done = 1;
    loop_set(lc, false);
  }
}
// Slabs, peer path: p = r on the halo planes too (cg.jl:77 on the neighbours' rows): copies the neighbours' boundary
// planes of r into the local halo planes of p.  Runs after k_cg_init_fin, i.e. after every rank's prologue has
// published its partial sums — their r is complete and fenced.
template <typename T>
__global__ void __launch_bounds__(kThreads) k_p_halo_init(i64 N, i64 halo, T* __restrict__ p, const T* __restrict__ r_lo,
                                                          const T* __restrict__ r_hi, i64 n_lo) {
  for (i64 q = (i64)blockIdx.x * blockDim.x + threadIdx.x; q < halo; q += (i64)gridDim.x * blockDim.x) {
    if (r_lo) p[q - halo] = __ldcg(r_lo + (n_lo - halo + q));
    if (r_hi) p[N + q] = __ldcg(r_hi + q);
  }
}
// cg.jl:47: x = zeros when the right-hand side is zero (flag -9); runs after the loop, returns at once otherwise
template <typename T>
__global__ void __launch_bounds__(kThreads) k_cg_zero_x(i64 N, T* __restrict__ x, const CgState* st) {
  if (st->flag != -9) return;
  for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < N; r += (i64)gridDim.x * blockDim.x) x[r] = (T)0;
}

// x += alpha p ; r -= alpha Ap ; rr_new = dot(r,r)        (cg.jl:88-100)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_cg_xr(i64 N, T* __restrict__ x, T* __restrict__ r,
                                                    const T* __restrict__ p, const T* __restrict__ Ap,
                                                    RedScratch rs, CgState* st, const __grid_constant__ CommDev cd,
                                                    i64 halo) {
  if (st->done) return;
  constexpr int VW = Vec<T>::W;
  const double pAp = st->pAp;                         // peer path: all-reduced by the SpMV's last block

  const T gamma = (T)st->rr;
  const T alpha = gamma / (T)pAp;
  const bool bad = (alpha == (T)INFINITY) || (alpha < (T)0);   // cg.jl:91
  double d[1] = {0.0};
  if (!bad) {
    const i64 nvec = N / VW;
    for (i64 iv = (i64)blockIdx.x * blockDim.x + threadIdx.x; iv < nvec; iv += (i64)gridDim.x * blockDim.x) {
      const i64 row = iv * VW;
      T xv[VW], rv[VW], pv[VW], av[VW];
      vload<T>(x + row, xv);
      vload<T>(r + row, rv);
      vload<T>(p + row, pv);
      vload_stream<T>(Ap + row, av);
#pragma unroll
      for (int e = 0; e < VW; ++e) {
        xv[e] = xv[e] + alpha * pv[e];
        rv[e] = rv[e] - alpha * av[e];
        d[0] += (double)rv[e] * (double)rv[e];
      }
      vstore<T>(x + row, xv);
      vstore<T>(r + row, rv);
    }
    for (i64 row = nvec * VW + (i64)blockIdx.x * blockDim.x + threadIdx.x; row < N;
         row += (i64)gridDim.x * blockDim.x) {
      const T xv = x[row] + alpha * p[row];
      const T rv = r[row] - alpha * Ap[row];
      d[0] += (double)rv * (double)rv;
      x[row] = xv;
      r[row] = rv;
    }
  }
  bool sys = false;
  if (cd.on) {                 // the neighbours read the boundary planes of r (k_cg_p): those blocks fence at system scope
    bool lo, hi;
    block_touches_ends(N, halo, VW, lo, hi);
    sys = lo || hi;
  }
  if (grid_sum<1>(d, rs, sys)) {
    if (bad) {
      if (threadIdx.x == 0) {
        st->flag = -2;          // "Matrix A in cg has to be positive definite"
        st->iter = st->iter + 1;
        st->loops = st->loops + 1;
        st->relres = 0.0;       // resvec[lastIter] never written
        st->done = 1;
      }
    } else if (cd.on) {
      mail_allreduce<1>(cd, d, &st->rr_new);             // the global r.r is in place when the kernel ends
    } else if (threadIdx.x == 0) {
      st->rr_new = d[0];
    }
  }
}

// convergence test + p = r + beta p          (cg.jl:100-114); the last block advances the state
template <typename T>
__global__ void __launch_bounds__(kThreads) k_cg_p(i64 N, const T* __restrict__ r, T* __restrict__ p,
                                                   RedScratch rs, CgState* st, const __grid_constant__ CommDev cd,
                                                   i64 halo, LoopCond lc, const T* __restrict__ r_lo,
                                                   const T* __restrict__ r_hi, i64 n_lo) {
  if (st->done) {               // k_cg_xr found alpha < 0 / Inf (cg.jl:91): the loop ends here
    if (blockIdx.x == 0 && threadIdx.x == 0) loop_set(lc, false);
    return;
  }
  constexpr int VW = Vec<T>::W;
  const double rr_new = st->rr_new;                   // peer path: all-reduced by k_cg_xr's last block

  const T nb = (T)sqrt(st->bb);
  const T res = (T)sqrt(rr_new) / nb;
  const bool conv = res <= (T)st->tol;
  const int it = st->iter + 1;
  const bool last_it = it >= st->maxit;
  if (!conv && !last_it) {
    const T gamma = (T)st->rr;
    const T beta = (T)rr_new / gamma;
    const i64 nvec = N / VW;
    for (i64 iv = (i64)blockIdx.x * blockDim.x + threadIdx.x; iv < nvec; iv += (i64)gridDim.x * blockDim.x) {
      const i64 row = iv * VW;
      T rv[VW], pv[VW];
      vload<T>(r + row, rv);
      vload<T>(p + row, pv);
#pragma unroll
      for (int e = 0; e < VW; ++e) pv[e] = rv[e] + beta * pv[e];
      vstore<T>(p + row, pv);
    }
    for (i64 row = nvec * VW + (i64)blockIdx.x * blockDim.x + threadIdx.x; row < N;
         row += (i64)gridDim.x * blockDim.x)
      p[row] = r[row] + beta * p[row];
    // Slabs, peer path: the halo planes of p are updated HERE, redundantly, with the same expression — from the
    // neighbour's boundary plane of r (read over NVLink; complete on every rank once the r.r partials have been
    // collected above) and the local halo copy of the old p.  The SpMV then finds all of p in local memory: no
    // p-halo transfer, no version flag, one rendezvous less per CG iteration (bit-identical: same beta, same operands).
    if (r_lo)
      for (i64 q = (i64)blockIdx.x * blockDim.x + threadIdx.x; q < halo; q += (i64)gridDim.x * blockDim.x)
        p[q - halo] = __ldcg(r_lo + (n_lo - halo + q)) + beta * p[q - halo];
    if (r_hi)
      for (i64 q = (i64)blockIdx.x * blockDim.x + threadIdx.x; q < halo; q += (i64)gridDim.x * blockDim.x)
        p[N + q] = __ldcg(r_hi + q) + beta * p[N + q];
  }
  if (last_block_ticket(rs.counter, false) && threadIdx.x == 0) {
    st->iter = it;
    st->loops = st->loops + 1;
    st->relres = (double)res;
    if (conv) {
      st->flag = 0;
      st->done = 1;
    } else if (last_it) {
      st->flag = -1;
      st->done = 1;
    } else {
      st->rr = rr_new;
      st->rr_new = rr_new;
    }
    loop_set(lc, !(conv || last_it));
  }
}

// =============================================================================================
// rhs = sum_i A_i' (rho_i y_i + l_i)        (rhs_compose.jl:24-36)
// =============================================================================================
constexpr int kRdualSets = 8;   // the fused rhs + dual-residual kernel handles up to 8 terms
template <typename T>
struct SetRef {
  OpDev op;
  const T* y;
  const T* l;
  const T* y_old;
  T rho;
};
template <typename T>
struct RhsArgs {
  int nsets;
  unsigned n[3];
  i64 npts;
  i64 ncols;       // npts or 2*npts
  int accumulate;  // start from the rhs already in memory (sets processed in several launches) instead of zero
  T* rhs;
  SetRef<T> sets[kMaxSets];
};

// G consecutive columns per thread (two 16-byte vectors of Float32): the gathers of a group are
// independent, which puts G x (rows per column) loads in flight per thread and hides the DRAM latency that
// bounded the per-column version (ncu round 1: long-scoreboard stalls on the first FMUL/FADD after each
// gather); rhs is written with 16-byte stores.  Groups that wrap a grid line fall back to single points.
template <typename T, int G, typename F>
__device__ __forceinline__ void rhs_set(const OpDev& op, const GridIdx& g0, bool line, const F& f, unsigned npts,
                                        const unsigned (&n)[3], T (&t)[F::NV][G]) {
  if (line) {
    op_adjoint_line<T, G>(op, op.mode, g0, f, t);
  } else {
    GridIdx g = g0;
#pragma unroll
    for (int e = 0; e < G; ++e) {
      T one[F::NV];
      op_adjoint_pt<T>(op, op.mode, g, f, one);
#pragma unroll
      for (int q = 0; q < F::NV; ++q) t[q][e] = one[q];
      grid_next(g, npts, n);
    }
  }
}

template <typename T, int G, bool RDUAL>
__device__ __forceinline__ void rhs_cols(const RhsArgs<T>& a, i64 c0, T (&acc)[G], double* d) {
  GridIdx g0 = grid_decode(c0, a.npts, a.n);
  const bool line = (G == 1) || (g0.i + (unsigned)G <= a.n[0] && (g0.upper || c0 + G <= a.npts));
  if (a.accumulate) {
    load_any<T, G>(a.rhs + c0, acc);
  } else {
#pragma unroll
    for (int e = 0; e < G; ++e) acc[e] = (T)0;
  }
  for (int s = 0; s < a.nsets; ++s) {
    const SetRef<T>& S = a.sets[s];
    if (RDUAL) {
      // the dual residual of the PREVIOUS iteration, ||A'(y - y_old)||^2 (update_y_l.jl:82-84), rides on the
      // same gather (y is loaded once for both): y_old still holds y^{k-1} until the next y/l update
      T t[2][G];
      rhs_set<T, G>(S.op, g0, line, FetchAxpyDiff<T>{S.rho, S.y, S.l, S.y_old}, (unsigned)a.npts, a.n, t);
      double sq = 0.0;
#pragma unroll
      for (int e = 0; e < G; ++e) {
        acc[e] = acc[e] + t[0][e];
        sq += (double)t[1][e] * (double)t[1][e];
      }
      if (s < kRdualSets) d[s * kThreads] += sq;     // per-thread slot in shared memory (keeps 16 registers free)
    } else {
      T t[1][G];
      rhs_set<T, G>(S.op, g0, line, FetchAxpy<T>{S.rho, S.y, S.l}, (unsigned)a.npts, a.n, t);
#pragma unroll
      for (int e = 0; e < G; ++e) acc[e] = acc[e] + t[0][e];
    }
  }
}

// RDUAL: additionally reduce, per set s < kRdualSets, ||A_s'(y_s - y_old_s)||^2 -> out[s]
template <typename T, bool RDUAL>
__global__ void __launch_bounds__(kThreads, 4) k_rhs(const __grid_constant__ RhsArgs<T> a, RedScratch rs, double* out) {
  constexpr int VW = Vec<T>::W;
  __shared__ double dsh[RDUAL ? kRdualSets * kThreads : 1];
  double* d = dsh + (RDUAL ? threadIdx.x : 0);
  if (RDUAL) {
#pragma unroll
    for (int q = 0; q < kRdualSets; ++q) d[q * kThreads] = 0.0;
  }
  constexpr int G = 2 * VW;
  const i64 ngrp = a.ncols / G;
  for (i64 iv = (i64)blockIdx.x * blockDim.x + threadIdx.x; iv < ngrp; iv += (i64)gridDim.x * blockDim.x) {
    T acc[G];
    rhs_cols<T, G, RDUAL>(a, iv * G, acc, d);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      T part[VW];
#pragma unroll
      for (int e = 0; e < VW; ++e) part[e] = acc[h * VW + e];
      vstore<T>(a.rhs + iv * G + h * VW, part);
    }
  }
  for (i64 c = ngrp * G + (i64)blockIdx.x * blockDim.x + threadIdx.x; c < a.ncols; c += (i64)gridDim.x * blockDim.x) {
    T acc[1];
    rhs_cols<T, 1, RDUAL>(a, c, acc, d);
    a.rhs[c] = acc[0];
  }
  if (RDUAL) {
    double dr[kRdualSets];
#pragma unroll
    for (int q = 0; q < kRdualSets; ++q) dr[q] = d[q * kThreads];
    if (grid_sum<kRdualSets>(dr, rs) && threadIdx.x == 0) {
#pragma unroll
      for (int q = 0; q < kRdualSets; ++q) out[q] = dr[q];
    }
  }
}

// =============================================================================================
// explicit sparse operators (constraint.custom_TD_OP, setup_constraints.jl:70-72)
//
// The stencil operators above are matrix-free and fused into the y/l and rhs kernels.  A user-supplied sparse
// matrix gets its own small kernels instead (so the hot kernels carry no variable-length loops): s = A x is
// written to the set's s buffer and the fused y/l kernels then see the identity acting on that buffer;
// A'(rho y + l) is accumulated into rhs between the stencil sets in the reference's set order.  Folds follow
// SparseArrays: ascending column index inside a row, ascending row index inside a column, from zero.
// =============================================================================================
template <typename T>
struct SparseRef {
  const long long* rp; const int* ci; const T* va;     // CSR of A
  const long long* cp; const int* ri; const T* vt;     // CSC of A
  i64 rows, cols;
};
// s = A x                                                     (update_y_l.jl:43, PARSDMM_initialize.jl:97)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_sparse_forward(SparseRef<T> A, const T* __restrict__ x, T* __restrict__ s) {
  for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < A.rows; r += (i64)gridDim.x * blockDim.x) {
    T acc = (T)0;
    for (long long q = A.rp[r]; q < A.rp[r + 1]; ++q) acc = acc + A.va[q] * x[A.ci[q]];
    s[r] = acc;
  }
}
// t = [t +] A' v  with  v = rho*y + l  (l == null: v = y)          (rhs_compose.jl:28-30)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_sparse_adjoint(SparseRef<T> A, T rho, const T* __restrict__ y,
                                                             const T* __restrict__ l, T* __restrict__ t, int accumulate) {
  for (i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x; c < A.cols; c += (i64)gridDim.x * blockDim.x) {
    T acc = (T)0;
    for (long long q = A.cp[c]; q < A.cp[c + 1]; ++q) {
      const int r = A.ri[q];
      const T v = l ? rho * y[r] + l[r] : y[r];
      acc = acc + A.vt[q] * v;
    }
    t[c] = accumulate ? t[c] + acc : acc;
  }
}
// || A' (y - y_old) ||^2 -> out[0]                                 (update_y_l.jl:82-84)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_sparse_rdual(SparseRef<T> A, const T* __restrict__ y,
                                                           const T* __restrict__ y_old, RedScratch rs, double* out) {
  double d[1] = {0.0};
  for (i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x; c < A.cols; c += (i64)gridDim.x * blockDim.x) {
    T acc = (T)0;
    for (long long q = A.cp[c]; q < A.cp[c + 1]; ++q) {
      const int r = A.ri[q];
      acc = acc + A.vt[q] * (y[r] - y_old[r]);
    }
    d[0] += (double)acc * (double)acc;
  }
  if (grid_sum<1>(d, rs) && threadIdx.x == 0) out[0] = d[0];
}

// =============================================================================================
// projectors applied element-wise
// =============================================================================================
template <typename T>
struct ProjDev {
  int kind;          // SIPB_SET_*
  T lo, hi;          // scalar bounds / (annulus: sigma_min, sigma_max) / l1 tau, l2 sigma in hi
  const T* lo_vec;   // vector bounds
  const T* hi_vec;
  const T* m;        // distance term: the vector being projected
  unsigned td[3];    // fiber bounds: transform-domain grid (rank-local on slabs)
  unsigned td_kofs;  //   slabs: global index of local plane 0 (the bounds of a z fiber are indexed by the global plane)
  int fiber_axis;
  T rho;             // distance term / prox_l1: current rho
  // parameters produced by the reduction passes:
  T theta;           // l1 soft threshold (0 => identity)
  T scale;           // l2 / annulus scale factor (1 => identity)
  T fill;            // annulus zero-vector fill value (NaN => unused)
  unsigned long long key_thr;   // cardinality: smallest kept magnitude key
  int keep_all;      // cardinality: k >= M
  int keep_none;     // cardinality: k <= 0
  // cardinality, deferred tie handling (y/l pass 2 on a single GPU): entries equal to the threshold are zeroed here when
  // all ties of their row chunk lie beyond the quota (tie_base[chunk] >= quota); the one chunk the quota boundary
  // falls into was handled in place by k_tie_cross.  tie_base == null: ties were already zeroed in place.
  const unsigned long long* tie_base;
  long long tie_chunk;
  unsigned long long quota;
  int need_ties;
};

template <typename T> __device__ __forceinline__ unsigned long long mag_key(T v);
template <> __device__ __forceinline__ unsigned long long mag_key<float>(float v) {
  return (unsigned long long)(__float_as_uint(v) & 0x7fffffffu);
}
template <> __device__ __forceinline__ unsigned long long mag_key<double>(double v) {
  return (unsigned long long)(__double_as_longlong(v) & 0x7fffffffffffffffll);
}

template <typename T> __device__ __forceinline__ T t_abs(T v);
template <> __device__ __forceinline__ float t_abs<float>(float v) { return fabsf(v); }
template <> __device__ __forceinline__ double t_abs<double>(double v) { return fabs(v); }
template <typename T> __device__ __forceinline__ T t_sign(T v) {
  return v > (T)0 ? (T)1 : (v < (T)0 ? (T)-1 : v);   // sign(0)=0, sign(NaN)=NaN like Julia
}
template <typename T> __device__ __forceinline__ T t_max(T a, T b) {   // Julia max (NaN-propagating)
  return (a != a) ? a : ((b != b) ? b : (a > b ? a : b));
}
template <typename T> __device__ __forceinline__ T t_min(T a, T b) {
  return (a != a) ? a : ((b != b) ? b : (a < b ? a : b));
}

// P(v) for element r with all reduction-derived parameters already known
template <typename T, int PK = -1>
__device__ __forceinline__ T proj_apply(const ProjDev<T>& P, T v, i64 r) {
  // PK >= 0: the set kind is a compile-time constant (the hot y/l kernels dispatch once per thread instead of
  // once per element); PK < 0: read it from the descriptor
  switch (PK >= 0 ? PK : P.kind) {
    case SIPB_SET_BOUNDS_SCALAR:   // max(LB, min(x, UB))   project_bounds!.jl:9
      return t_max<T>(P.lo, t_min<T>(v, P.hi));
    case SIPB_SET_BOUNDS_VECTOR:   // min then max          project_bounds!.jl:21-22
      return t_max<T>(P.lo_vec[r], t_min<T>(v, P.hi_vec[r]));
    case SIPB_SET_BOUNDS_FIBER: {  // x[:,i] .= min.(max.(x[:,i],LB),UB): max first, bounds follow the fiber coordinate
      const unsigned q = (unsigned)r;
      unsigned c = q % P.td[0];
      if (P.fiber_axis == 1) c = (q / P.td[0]) % P.td[1];
      else if (P.fiber_axis == 2) c = q / (P.td[0] * P.td[1]) + P.td_kofs;
      return t_min<T>(t_max<T>(v, P.lo_vec[c]), P.hi_vec[c]);       // project_bounds!.jl:46,50,65-77
    }
    case SIPB_SET_CARD_SLICE:
    case SIPB_SET_CARD_FIBER:      // already projected in place by k_card_fiber_* (pass-through)
    case SIPB_SET_HISTOGRAM:       // already projected in place by k_hist_apply (pass-through)
      return v;
    case SIPB_SET_DISTANCE: {      // (x*rho + m) / (rho + 1.0) in Float64   prox_l2s!.jl:4
      const T num = v * P.rho + P.m[r];
      return (T)((double)num / ((double)P.rho + 1.0));
    }
    case SIPB_SET_PROX_L1: {       // sign(x) * max(0, abs(x) - 1/rho)       prox_l1!.jl:9
      const T thr = (T)1 / P.rho;
      return t_sign<T>(v) * t_max<T>((T)0, t_abs<T>(v) - thr);
    }
    case SIPB_SET_L1:              // sign(v) * max(abs(v) - theta, 0)       project_l1_Duchi!.jl:49
      if (P.theta < (T)0) return v;   // inside the ball: untouched
      return t_sign<T>(v) * t_max<T>(t_abs<T>(v) - P.theta, (T)0);
    case SIPB_SET_L2:
    case SIPB_SET_ANNULUS:         // rmul!(x, sigma/nl2)   project_l2!.jl:11, project_annulus!.jl:11-17
      if (P.fill == P.fill) return P.fill;
      return (P.scale == (T)1) ? v : v * P.scale;
    case SIPB_SET_CARDINALITY:     // zero everything below the k-th largest magnitude
      if (P.keep_all) return v;
      if (P.keep_none) return (T)0;
      {
        const unsigned long long key = mag_key<T>(v);
        if (key != P.key_thr) return (key > P.key_thr) ? v : (T)0;
        if (P.need_ties && P.tie_base && P.tie_base[r / P.tie_chunk] >= P.quota) return (T)0;
        return v;
      }
    default:
      return v;
  }
}

__host__ __device__ __forceinline__ bool proj_is_elementwise(int kind) {
  return kind == SIPB_SET_BOUNDS_SCALAR || kind == SIPB_SET_BOUNDS_VECTOR || kind == SIPB_SET_BOUNDS_FIBER ||
         kind == SIPB_SET_DISTANCE ||
         kind == SIPB_SET_PROX_L1;
}

// cardinality search (defined with the radix select below): digit histograms that pass 1 of the y/l update
// accumulates on the side while it produces v
constexpr int kSelBins = 2048;          // bins of one level (2^11)
constexpr int kSpecBits = 11;           // digit width of the speculative histograms built by pass 1 of the y/l update
constexpr int kSpecLevels = 3;          // levels covered speculatively (all of a Float32 key, the top 33 bits of a Float64 key)
struct SpecCtx {
  unsigned int* sh;               // shared-memory histograms of levels 1 .. kSpecLevels-1
  unsigned long long guess;       // threshold key of the previous PARSDMM iteration
  unsigned int g0;                // its top digit
  unsigned int above;             // this thread's count of keys whose top digit exceeds the guess's
};
template <typename T>
__device__ __forceinline__ void spec_hist_add(SpecCtx& sc, T v);

// =============================================================================================
// y / l update                               (update_y_l.jl:39-94)
// fused with the rho/gamma adaptation reductions and snapshots
//                                            (adapt_rho_gamma.jl:41-53, PARSDMM.jl:164-207)
// =============================================================================================
template <typename T>
struct ProjParams {       // device-resident projector parameters written by the parameter kernels
  T theta;
  T scale;
  T fill;
  unsigned long long key_thr;
  unsigned long long quota;
  unsigned long long count_eq;
  int keep_all, keep_none, need_ties;
};

template <typename T>
struct YlArgs {
  OpDev op;
  ProjDev<T> P;
  const ProjParams<T>* dyn;   // reduction-type projectors: parameters produced on the device
  const T* x;
  T* y;                       // y^{k+1} (output; MODE 1 parks v = x_hat - l/rho here for pass 2)
  T* l;
  const T* y_old;             // y^{k}: the host swaps the y / y_old buffers instead of copying (update_y_l.jl:64)
  T* s;                       // reduction-type projectors: s = A x is stored by pass 1 only when somebody reads it later
  int store_s;                //   (the feasibility check of every 10th iteration); pass 2 recomputes it from x
  int skip_v;                 // pass 1 of an l1 set: do not store v (pass 2 recomputes it; the threshold search only reads
                              //   v when the ball is active — a gated second launch of pass 1 then writes it)
  const double* gate;         // gated launch of pass 1: return at once when (T)gate[0] <= (T)gate_tau (sum|v| <= tau: the
  double gate_tau;            //   vector lies inside the l1 ball, project_l1_Duchi!.jl:23, nobody will read v)
  T* lhat0; T* s0; T* l0; T* y0;   // snapshots of the adaptation scheme
  T rho, gamma;
  const T* x_old;    // distance term only: also reduce the stop sums ||x-m||^2, ||x_old-x||^2, ||x||^2 (PARSDMM.jl:140-145)
  double* stop_out;  //   -> stop_out[0..2]; null => the separate k_stop pass does it
  int want_feas;     // also reduce ||P(s)-s||^2 and ||s||^2 (element-wise projectors only)
  int do_sums;       // the six adaptation reductions against the previous snapshots
  int do_snapshot;   // overwrite the snapshots (l_hat_0, y_0, s_0, l_0)
};

template <typename T, int W> __device__ __forceinline__ void load_n(const T* p, T (&v)[W]) {
  if constexpr (W == Vec<T>::W) vload<T>(p, v);
  else {
#pragma unroll
    for (int e = 0; e < W; ++e) v[e] = p[e];
  }
}
template <typename T, int W> __device__ __forceinline__ void store_n(T* p, const T (&v)[W]) {
  if constexpr (W == Vec<T>::W) vstore<T>(p, v);
  else {
#pragma unroll
    for (int e = 0; e < W; ++e) p[e] = v[e];
  }
}

// Processes W consecutive rows starting at r0.
// MODE 0: element-wise projector, everything in one pass.
// MODE 1: reduction-type projector, pass 1: y <- v = x_hat - l/rho, s stored.
// MODE 2: reduction-type projector, pass 2: y <- P(v), l update.
// d[]: MODE 0/2: [0] ||y-s||^2, [1] ||P(s)-s||^2, [2] ||s||^2 ; MODE 1: [0] sum|v|, [1] sum v^2, [2] nnz(v)
//      ADAPT   : [3] dot(dH,dlh) [4] ||dH||^2 [5] ||dlh||^2 [6] ||dl||^2 [7] ||dG||^2 [8] dot(dG,dl)
template <typename T, int MODE, bool ADAPT, int W, int PK>
__device__ __forceinline__ void yl_rows(const YlArgs<T>& a, const ProjDev<T>& P, i64 r0, double* d,
                                        SpecCtx* spec = nullptr) {
  const T rho = a.rho, gamma = a.gamma;
  const T rho1 = (T)1.0 / rho;                      // update_y_l.jl:34
  const bool relaxed = !(gamma == (T)1);
  T s[W], yo[W], lo[W], yn[W], ln[W];
  if (MODE == 0 || MODE == 1) {
    if (relaxed || ADAPT) load_n<T, W>(a.y_old + r0, yo);
    load_n<T, W>(a.l + r0, lo);
    op_forward_n<T, W>(a.op, (unsigned)r0, a.x, s);
#pragma unroll
    for (int e = 0; e < W; ++e) {
      T xh = s[e];
      if (relaxed) xh = gamma * s[e] + ((T)1.0 - gamma) * yo[e];     // :72
      const T v = xh - lo[e] * rho1;                                    // :67 / :74
      if (MODE == 0) {
        yn[e] = proj_apply<T, PK>(P, v, r0 + e);
        const T rp = -s[e] + yn[e];                                     // :69 / :76
        ln[e] = relaxed ? lo[e] + rho * (-xh + yn[e]) : lo[e] + rho * rp;
        d[0] += (double)rp * (double)rp;
        if (PK != SIPB_SET_DISTANCE && a.want_feas) {
          const T pf = proj_apply<T, PK>(P, s[e], r0 + e) - s[e];
          d[1] += (double)pf * (double)pf;
          d[2] += (double)s[e] * (double)s[e];
        }
      } else {
        yn[e] = v;
        d[0] += (double)t_abs<T>(v);
        d[1] += (double)v * (double)v;
        d[2] += (v != (T)0) ? 1.0 : 0.0;
        if (spec) spec_hist_add<T>(*spec, v);                      // k_yl_spec only
      }
    }
    if (MODE == 0 || !a.skip_v) store_n<T, W>(a.y + r0, yn);
    if (MODE == 0) store_n<T, W>(a.l + r0, ln);
    else if (a.store_s) store_n<T, W>(a.s + r0, s);
    if (MODE == 0 && PK == SIPB_SET_DISTANCE) {
      // the distance term holds s = x and m in registers: the stop / log sums of PARSDMM.jl:140-145 ride along
      // (same expressions as k_stop); slot layout: d[1] ||x_old-x||^2, d[2] ||x||^2, last slot ||x-m||^2
      if (a.stop_out) {
        T xo[W];
        load_n<T, W>(a.x_old + r0, xo);
#pragma unroll
        for (int e = 0; e < W; ++e) {
          const T xv = s[e];
          const T dx = xo[e] - xv;
          d[1] += (double)dx * (double)dx;
          d[2] += (double)xv * (double)xv;
          const T o = xv - P.m[r0 + e];
          d[ADAPT ? 9 : 3] += (double)o * (double)o;
        }
      }
    }
  } else {
    T v[W];
    // the l1 ball never changes v in place: pass 2 recomputes it like s (same expressions as pass 1, bit for bit)
    constexpr bool kRecomputeV = (PK == SIPB_SET_L1);
    if (!kRecomputeV) load_n<T, W>(a.y + r0, v);
    // s = A x again (the same left fold as in pass 1, bit for bit): a gather of N words from x instead of a stored
    // and re-read M-vector (M = 3N for the TV sets)
    op_forward_n<T, W>(a.op, (unsigned)r0, a.x, s);
    load_n<T, W>(a.l + r0, lo);
    if (relaxed || ADAPT) load_n<T, W>(a.y_old + r0, yo);
#pragma unroll
    for (int e = 0; e < W; ++e) {
      if (kRecomputeV) {
        T xh = s[e];
        if (relaxed) xh = gamma * s[e] + ((T)1.0 - gamma) * yo[e];     // update_y_l.jl:72
        v[e] = xh - lo[e] * rho1;                                         // :67 / :74
      }
      yn[e] = proj_apply<T, PK>(P, v[e], r0 + e);
      const T rp = -s[e] + yn[e];
      if (relaxed) {
        const T xh = gamma * s[e] + ((T)1.0 - gamma) * yo[e];
        ln[e] = lo[e] + rho * (-xh + yn[e]);
      } else {
        ln[e] = lo[e] + rho * rp;
      }
      d[0] += (double)rp * (double)rp;
    }
    store_n<T, W>(a.y + r0, yn);
    store_n<T, W>(a.l + r0, ln);
  }
  if (ADAPT && MODE != 1) {
    T lh[W];
#pragma unroll
    for (int e = 0; e < W; ++e) lh[e] = lo[e] + rho * (-s[e] + yo[e]);     // adapt_rho_gamma.jl:41
    if (a.do_sums) {
      T lh0[W], s0[W], l0[W], y0[W];
      load_n<T, W>(a.lhat0 + r0, lh0);
      load_n<T, W>(a.s0 + r0, s0);
      load_n<T, W>(a.l0 + r0, l0);
      load_n<T, W>(a.y0 + r0, y0);
#pragma unroll
      for (int e = 0; e < W; ++e) {
        const T dlh = lh[e] - lh0[e];
        const T dH = s[e] - s0[e];
        const T dl = ln[e] - l0[e];
        const T dG = -(yn[e] - y0[e]);
        d[3] += (double)dH * (double)dlh;
        d[4] += (double)dH * (double)dH;
        d[5] += (double)dlh * (double)dlh;
        d[6] += (double)dl * (double)dl;
        d[7] += (double)dG * (double)dG;
        d[8] += (double)dG * (double)dl;
      }
    }
    if (a.do_snapshot) {
      store_n<T, W>(a.lhat0 + r0, lh);
      store_n<T, W>(a.y0 + r0, yn);
      store_n<T, W>(a.s0 + r0, s);
      store_n<T, W>(a.l0 + r0, ln);
    }
  }
}

// out: [0..2] as d[0..2] (MODE 2 writes only [0]); ADAPT sums go to out[4..9]
// PK: compile-time set kind of the specialised instances (-1: read the kind from the descriptor)
template <typename T, int MODE, bool ADAPT, int PK>
__device__ __forceinline__ void yl_body(const YlArgs<T>& a, const RedScratch& rs, double* out, SpecCtx* spec = nullptr) {
  constexpr int VW = Vec<T>::W;
  constexpr int NR = (ADAPT ? 9 : 3) + (MODE == 0 ? 1 : 0);      // MODE 0: one more slot for the fused stop sums
  ProjDev<T> P = a.P;
  if (a.dyn) {
    P.theta = a.dyn->theta; P.scale = a.dyn->scale; P.fill = a.dyn->fill;
    P.key_thr = a.dyn->key_thr; P.keep_all = a.dyn->keep_all; P.keep_none = a.dyn->keep_none;
    P.quota = a.dyn->quota; P.need_ties = a.dyn->need_ties;
  }
  double d[NR];
#pragma unroll
  for (int i = 0; i < NR; ++i) d[i] = 0.0;
  const i64 M = a.op.rows;
  const i64 nvec = M / VW;
  for (i64 iv = (i64)blockIdx.x * blockDim.x + threadIdx.x; iv < nvec; iv += (i64)gridDim.x * blockDim.x)
    yl_rows<T, MODE, ADAPT, VW, PK>(a, P, iv * VW, d, spec);
  for (i64 r = nvec * VW + (i64)blockIdx.x * blockDim.x + threadIdx.x; r < M; r += (i64)gridDim.x * blockDim.x)
    yl_rows<T, MODE, ADAPT, 1, PK>(a, P, r, d, spec);
  if (grid_sum<NR>(d, rs) && threadIdx.x == 0) {
    out[0] = d[0];
    if (MODE != 2) {
      out[1] = d[1];
      out[2] = d[2];
    }
    if (ADAPT) {
#pragma unroll
      for (int i = 0; i < 6; ++i) out[4 + i] = d[3 + i];
    }
    if (MODE == 0 && PK == SIPB_SET_DISTANCE && a.stop_out) {
      a.stop_out[0] = d[NR - 1];
      a.stop_out[1] = d[1];
      a.stop_out[2] = d[2];
    }
  }
}

template <typename T, int MODE, bool ADAPT>
__global__ void __launch_bounds__(kThreads, 4) k_yl(const __grid_constant__ YlArgs<T> a, RedScratch rs, double* out) {
  if (MODE == 1 && a.gate && (T)a.gate[0] <= (T)a.gate_tau) return;      // gated pass 1: v is not needed
  // one dispatch on the set kind per block: the common kinds run fully specialised bodies
  if (MODE == 2 && a.P.kind == SIPB_SET_L1) yl_body<T, MODE, ADAPT, SIPB_SET_L1>(a, rs, out);
  else yl_body<T, MODE, ADAPT, -1>(a, rs, out);
}

// Pass 1 of a vector-mode cardinality set on a single GPU: as k_yl<T, 1, false>, and the first levels of the radix
// select ride along (spec_hist_add): a per-thread count and shared-memory histograms per block, flushed into
// SelState::spec_above / spec at the end.  `guess_pp` holds the threshold key of the previous iteration (any value is a
// valid guess).
template <typename T>
__global__ void __launch_bounds__(kThreads, 4) k_yl_spec(const __grid_constant__ YlArgs<T> a, RedScratch rs, double* out,
                                                         unsigned long long* __restrict__ spec_above,
                                                         unsigned long long* __restrict__ spec,
                                                         const ProjParams<T>* __restrict__ guess_pp) {
  constexpr int NB = (kSpecLevels - 1) * kSelBins;
  __shared__ unsigned int sh[NB];
  __shared__ unsigned int s_above[kThreads / 32];
  for (int t = threadIdx.x; t < NB; t += blockDim.x) sh[t] = 0u;
  __syncthreads();
  const unsigned long long guess = guess_pp->key_thr;
  SpecCtx sc{sh, guess, (unsigned)(guess >> ((int)sizeof(T) * 8 - kSpecBits)), 0u};
  yl_body<T, 1, false, -1>(a, rs, out, &sc);
  unsigned int ab = sc.above;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ab += __shfl_xor_sync(0xffffffffu, ab, o);
  if ((threadIdx.x & 31) == 0) s_above[threadIdx.x >> 5] = ab;
  __syncthreads();
  for (int t = threadIdx.x; t < NB; t += blockDim.x)
    if (sh[t]) atomicAdd(&spec[t], (unsigned long long)sh[t]);
  if (threadIdx.x == 0) {
    unsigned long long tot = 0ull;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += s_above[i];
    if (tot) atomicAdd(spec_above, tot);
  }
}

// All element-wise sets of one PARSDMM iteration in a single launch: blockIdx.y selects the set, every set
// reduces into its own scratch slice / ticket.  One launch instead of one per set removes the per-kernel
// ramp, tail and last-block latency (~8 us each at 200^3, most of the time at 256^2) and lets the tail of
// one set overlap the head of the next.
constexpr int kYlMulti = 8;
template <typename T>
struct YlMultiArgs {
  YlArgs<T> a[kYlMulti];
  double* out[kYlMulti];
};
template <typename T, bool ADAPT>
__global__ void __launch_bounds__(kThreads, 4) k_yl_multi(const __grid_constant__ YlMultiArgs<T> m, RedScratch rs) {
  const RedScratch mine{rs.partials + (size_t)blockIdx.y * kMaxRed * kMaxBlocks, rs.counter + blockIdx.y};
  const YlArgs<T>& a = m.a[blockIdx.y];
  switch (a.P.kind) {       // one dispatch per block: fully specialised bodies for the common set kinds
    case SIPB_SET_BOUNDS_SCALAR: yl_body<T, 0, ADAPT, SIPB_SET_BOUNDS_SCALAR>(a, mine, m.out[blockIdx.y]); break;
    case SIPB_SET_DISTANCE: yl_body<T, 0, ADAPT, SIPB_SET_DISTANCE>(a, mine, m.out[blockIdx.y]); break;
    default: yl_body<T, 0, ADAPT, -1>(a, mine, m.out[blockIdx.y]);
  }
}

// forward operator only: s = A x      (initial feasibility, PARSDMM_initialize.jl:97-99; unit tests)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_op_forward(const __grid_constant__ OpDev op, const T* __restrict__ x,
                                                         T* __restrict__ s) {
  for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < op.rows; r += (i64)gridDim.x * blockDim.x)
    s[r] = op_forward<T>(op, r, x);
}

// adjoint only: t = A' v (unit tests / sipb_op_apply)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_op_adjoint(const __grid_constant__ OpDev op, const T* __restrict__ v,
                                                         T* __restrict__ t) {
  for (i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x; c < op.cols; c += (i64)gridDim.x * blockDim.x) {
    const GridIdx g = grid_decode(c, op.npts, op.n);
    T one[1];
    op_adjoint_pt<T>(op, op.mode, g, FetchPlain<T>{v}, one);
    t[c] = one[0];
  }
}

// sums of a stored vector: [0] sum|v|, [1] sum v^2, [2] count(v != 0)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_vec_stats(i64 M, const T* __restrict__ v, RedScratch rs, double* out) {
  double d[3] = {0.0, 0.0, 0.0};
  for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < M; r += (i64)gridDim.x * blockDim.x) {
    const T t = v[r];
    d[0] += (double)t_abs<T>(t);
    d[1] += (double)t * (double)t;
    d[2] += (t != (T)0) ? 1.0 : 0.0;
  }
  if (grid_sum<3>(d, rs) && threadIdx.x == 0) {
    out[0] = d[0];
    out[1] = d[1];
    out[2] = d[2];
  }
}

// feasibility of a stored s w.r.t. a projector with known parameters: [0] ||P(s)-s||^2, [1] ||s||^2
// (update_y_l.jl:92-94).  `apply` != 0 writes P(s) back (sipb_project / initial feasibility).
template <typename T>
__global__ void __launch_bounds__(kThreads) k_feas(i64 M, T* __restrict__ s, const __grid_constant__ ProjDev<T> P,
                                                   int apply, RedScratch rs, double* out) {
  double d[2] = {0.0, 0.0};
  for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < M; r += (i64)gridDim.x * blockDim.x) {
    const T t = s[r];
    const T pt = proj_apply<T>(P, t, r);
    const T pf = pt - t;
    d[0] += (double)pf * (double)pf;
    d[1] += (double)t * (double)t;
    if (apply) s[r] = pt;
  }
  if (grid_sum<2>(d, rs) && threadIdx.x == 0) {
    out[0] = d[0];
    out[1] = d[1];
  }
}

// =============================================================================================
// dual residual: || A' (y - y_old) ||^2      (update_y_l.jl:82-84)
// =============================================================================================
template <typename T, int W>
__device__ __forceinline__ void rdual_cols(const OpDev& op, const T* __restrict__ y, const T* __restrict__ y_old,
                                           i64 c0, double* d) {
  // the dual residual runs over one N-block only: evaluate the operator as if it were un-blocked
  GridIdx g = grid_decode(c0, op.npts, op.n);
  const FetchDiff<T> fd{y, y_old};
  T t[1][W];
  if (W == 1 || g.i + (unsigned)W <= op.n[0]) {
    op_adjoint_line<T, W>(op, SIPB_BLOCK_PLAIN, g, fd, t);
  } else {
#pragma unroll
    for (int e = 0; e < W; ++e) {
      T one[1];
      op_adjoint_pt<T>(op, SIPB_BLOCK_PLAIN, g, fd, one);
      t[0][e] = one[0];
      grid_next(g, 0xffffffffu, op.n);
    }
  }
#pragma unroll
  for (int e = 0; e < W; ++e) d[0] += (double)t[0][e] * (double)t[0][e];
}

template <typename T>
__global__ void __launch_bounds__(kThreads) k_rdual(const __grid_constant__ OpDev op, const T* __restrict__ y,
                                                    const T* __restrict__ y_old, RedScratch rs, double* out) {
  constexpr int VW = Vec<T>::W;
  double d[1] = {0.0};
  const i64 nvec = op.npts / VW;
  for (i64 iv = (i64)blockIdx.x * blockDim.x + threadIdx.x; iv < nvec; iv += (i64)gridDim.x * blockDim.x)
    rdual_cols<T, VW>(op, y, y_old, iv * VW, d);
  for (i64 cc = nvec * VW + (i64)blockIdx.x * blockDim.x + threadIdx.x; cc < op.npts; cc += (i64)gridDim.x * blockDim.x)
    rdual_cols<T, 1>(op, y, y_old, cc, d);
  if (grid_sum<1>(d, rs) && threadIdx.x == 0)
    out[0] = (op.mode == SIPB_BLOCK_BOTH) ? 2.0 * d[0] : d[0];   // [A A]' v = [A'v; A'v]
}

// =============================================================================================
// objective / evolution reductions              (PARSDMM.jl:139-145)
// out: [0] ||x - m||^2 (or ||x1 + x2 - m||^2 for Minkowski)  [1] ||x_old - x||^2  [2] ||x||^2
// =============================================================================================
template <typename T>
__global__ void __launch_bounds__(kThreads) k_stop(i64 N, i64 npts, int minkowski, const T* __restrict__ x,
                                                   const T* __restrict__ x_old, const T* __restrict__ m,
                                                   RedScratch rs, double* out) {
  double d[3] = {0.0, 0.0, 0.0};
  constexpr int VW = Vec<T>::W;
  const i64 nvec = minkowski ? 0 : N / VW;       // plain problems: 16-byte loads; Minkowski / tail: one row at a time
  for (i64 iv = (i64)blockIdx.x * blockDim.x + threadIdx.x; iv < nvec; iv += (i64)gridDim.x * blockDim.x) {
    T xv[VW], xo[VW], mv[VW];
    vload<T>(x + iv * VW, xv);
    vload<T>(x_old + iv * VW, xo);
    vload<T>(m + iv * VW, mv);
#pragma unroll
    for (int e = 0; e < VW; ++e) {
      const T dx = xo[e] - xv[e];
      d[1] += (double)dx * (double)dx;
      d[2] += (double)xv[e] * (double)xv[e];
      const T o = xv[e] - mv[e];
      d[0] += (double)o * (double)o;
    }
  }
  for (i64 r = nvec * VW + (i64)blockIdx.x * blockDim.x + threadIdx.x; r < N; r += (i64)gridDim.x * blockDim.x) {
    const T xv = x[r];
    const T e = x_old[r] - xv;
    d[1] += (double)e * (double)e;
    d[2] += (double)xv * (double)xv;
    if (!minkowski) {
      const T o = xv - m[r];
      d[0] += (double)o * (double)o;
    } else if (r < npts) {
      const T sx = ((T)0 + xv) + x[r + npts];     // TD_OP[end]*x with TD_OP[end] = [I I]
      const T o = sx - m[r];
      d[0] += (double)o * (double)o;
    }
  }
  if (grid_sum<3>(d, rs) && threadIdx.x == 0) {
    out[0] = d[0];
    out[1] = d[1];
    out[2] = d[2];
  }
}

// =============================================================================================
// A[:,col] += alpha * B[:,k]                  (CDS_scaled_add!.jl:22; Q assembly)
// =============================================================================================
template <typename T>
__global__ void __launch_bounds__(kThreads) k_cds_axpy(i64 N, T* __restrict__ A, const T* __restrict__ B, T alpha) {
  constexpr int VW = Vec<T>::W;
  const i64 nvec = N / VW;
  for (i64 iv = (i64)blockIdx.x * blockDim.x + threadIdx.x; iv < nvec; iv += (i64)gridDim.x * blockDim.x) {
    const i64 r = iv * VW;
    T av[VW], bv[VW];
    vload<T>(A + r, av);
    vload_stream<T>(B + r, bv);
#pragma unroll
    for (int e = 0; e < VW; ++e) av[e] = av[e] + alpha * bv[e];
    vstore<T>(A + r, av);
  }
  for (i64 r = nvec * VW + (i64)blockIdx.x * blockDim.x + threadIdx.x; r < N; r += (i64)gridDim.x * blockDim.x)
    A[r] = A[r] + alpha * B[r];
}

// ---- stencil-class tables (see RowClass above) ------------------------------------------------------------
struct ClassGeom {
  unsigned n[3];
  unsigned npts;
  int nhalf;         // 1, or 2 for Minkowski
  unsigned kofs;     // slabs: global plane number of the first local plane
  unsigned nz_loc;   // local planes
};
// representative LOCAL row of class `cls`, or -1 when the class has no local row
__device__ __forceinline__ i64 class_local_row(const ClassGeom& g, unsigned cls) {
  const unsigned ci = cls % 3u, cj = (cls / 3u) % 3u, ck = (cls / 9u) % 3u, half = cls / 27u;
  if ((int)half >= g.nhalf) return -1;
  auto rep = [](unsigned c, unsigned n, unsigned lo, unsigned cnt, bool& ok) -> unsigned {
    // an index in [lo, lo+cnt) with axis_class == c
    unsigned idx;
    if (c == 0u) idx = 0u;
    else if (c == 2u) idx = n - 1u;
    else idx = lo > 1u ? lo : 1u;
    ok = ok && idx >= lo && idx < lo + cnt && axis_class(idx, n) == c;
    return idx;
  };
  bool ok = true;
  const unsigned i = rep(ci, g.n[0], 0u, g.n[0], ok);
  const unsigned j = rep(cj, g.n[1], 0u, g.n[1], ok);
  const unsigned kk = rep(ck, g.n[2], g.kofs, g.nz_loc, ok);
  if (!ok) return -1;
  const i64 plane = (i64)g.n[0] * g.n[1];
  return (i64)half * g.npts + (i64)(kk - g.kofs) * plane + (i64)j * g.n[0] + i;
}
// tab[cls*nd + j] = R[j*ld + representative row]   (0 for classes without a local row)
template <typename T>
__global__ void k_class_extract(const T* __restrict__ R, i64 ld, int nd, ClassGeom g, T* __restrict__ tab) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= kMaxClasses * nd) return;
  const unsigned cls = q / nd;
  const int j = q - cls * nd;
  const i64 r = class_local_row(g, cls);
  tab[q] = r >= 0 ? R[(i64)j * ld + r] : (T)0;
}
// bad[0] != 0 when some local entry differs (bitwise) from its class value
template <typename T>
__global__ void __launch_bounds__(kThreads) k_class_verify(const T* __restrict__ R, i64 ld, int nd, i64 N, i64 row0,
                                                           ClassGeom g, const T* __restrict__ tab, int* bad) {
  __shared__ T tab_s[kMaxClasses * kMaxDiag];
  for (int q = threadIdx.x; q < kMaxClasses * nd; q += blockDim.x) tab_s[q] = tab[q];
  __syncthreads();
  bool mismatch = false;
  for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < N; r += (i64)gridDim.x * blockDim.x) {
    const unsigned cls = row_class(row0 + r, g.n, g.npts);
    for (int j = 0; j < nd; ++j) {
      const T v = R[(i64)j * ld + r];
      const T t = tab_s[cls * nd + j];
      mismatch = mismatch || value_bits<T>(v) != value_bits<T>(t);
    }
  }
  if (mismatch) atomicExch(bad, 1);
}
// Q_tab[cls*nq + qcol[j]] += alpha * A_tab[cls*nd + j]      (CDS_scaled_add!.jl:22 on one row per class)
struct QCols { int c[kMaxDiag]; };
template <typename T>
__global__ void k_class_axpy(T* __restrict__ Qt, int nq, const T* __restrict__ At, int nd, QCols qc, T alpha) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= kMaxClasses * nd) return;
  const int cls = q / nd;
  const int j = q - cls * nd;
  T* dst = Qt + cls * nq + qc.c[j];
  *dst = *dst + alpha * At[q];
}

// =============================================================================================
// l1-ball threshold: sort-free Newton / Michelot iteration on
//     f(theta) = sum max(|v| - theta, 0) - tau            (project_l1_Duchi!.jl:33-46)
// Each pass reduces count and sum of the entries above the current theta; the last block performs
// the Newton step theta <- (S - tau)/C.  From any start the first step lands left of the root
// (f is convex), afterwards the iterates increase monotonically and reach the exact root of the
// piecewise-linear f in finitely many steps (the fix point is detected bit-exactly because the
// reductions are deterministic).
// =============================================================================================
struct L1State {
  double C, S;       // count and sum of the entries above theta (adjacent: one 2-double all-reduce with slabs)
  double theta;      // current iterate
  double tau;
  double S1;         // sum |v|
  double M;          // number of elements
  int on_left;       // iterate known to be <= root
  int done;
  int passes;
  int failed;        // sticky: a search hit the pass limit without reaching its fix point
};

// Newton step theta <- (S - tau)/C with the restart / fix-point logic
__device__ __forceinline__ void l1_newton_step(L1State* st, double C, double S) {
  const double theta = st->theta;
  st->passes += 1;
  st->C = C;                 // kept for the host: C == M at the fix point triggers the reference's lv-1 cap (k_l1_cap)
  st->S = S;
  if (C == 0.0) {            // theta at/above max|v|: restart from the left end
    st->theta = 0.0;
    st->on_left = 1;
    if (theta == 0.0) st->done = 1;   // all-zero vector
  } else {
    double tn = (S - st->tau) / C;
    if (tn < 0.0) tn = 0.0;
    if (st->on_left && tn <= theta) {
      st->done = 1;          // fix point: theta is the exact root
    } else {
      st->theta = tn;
      st->on_left = 1;
    }
  }
  if (st->passes >= 200 && !st->done) { st->done = 1; st->failed = 1; }     // no fix point: reported by the host
}

// fused != 0: the last block performs the Newton step (single GPU); otherwise it only publishes the
// rank-local (C, S) and k_l1_step runs after the all-reduce.
template <typename T>
__global__ void __launch_bounds__(kThreads) k_l1_pass(i64 M, const T* __restrict__ v, RedScratch rs, L1State* st,
                                                      int fused, const __grid_constant__ CommDev cd, LoopCond lc) {
  if (st->done) {
    if (blockIdx.x == 0 && threadIdx.x == 0) loop_set(lc, false);
    return;
  }
  const double theta = st->theta;
  double d[2] = {0.0, 0.0};
  constexpr int VW = Vec<T>::W;
  const i64 nvec = M / VW;
  for (i64 iv = (i64)blockIdx.x * blockDim.x + threadIdx.x; iv < nvec; iv += (i64)gridDim.x * blockDim.x) {
    T t[VW];
    vload<T>(v + iv * VW, t);
#pragma unroll
    for (int e = 0; e < VW; ++e) {
      const double a = (double)t_abs<T>(t[e]);
      if (a > theta) { d[0] += 1.0; d[1] += a; }
    }
  }
  for (i64 r = nvec * VW + (i64)blockIdx.x * blockDim.x + threadIdx.x; r < M; r += (i64)gridDim.x * blockDim.x) {
    const double a = (double)t_abs<T>(v[r]);
    if (a > theta) { d[0] += 1.0; d[1] += a; }
  }
  if (grid_sum<2>(d, rs)) {
    if (cd.on) mail_publish<2>(cd, d);          // slabs, peer path: partial (C, S) to every rank's mailbox
    else if (threadIdx.x == 0) {
      if (fused) {
        l1_newton_step(st, d[0], d[1]);
        loop_set(lc, !st->done);
      } else { st->C = d[0]; st->S = d[1]; }
    }
  }
}
// one thread; peer path: first sums the ranks' (C, S) partials from the mailbox (C and S are adjacent)
__global__ void k_l1_step(L1State* st, const __grid_constant__ CommDev cd, LoopCond lc) {
  if (st->done) { loop_set(lc, false); return; }
  if (cd.on) mail_collect<2>(cd, &st->C);
  l1_newton_step(st, st->C, st->S);
  loop_set(lc, !st->done);
}

// min |v| as an order-preserving magnitude key -> atomicMin on out[0] (initialised to ~0ull by the host).
// Only needed when EVERY entry stays above the l1 threshold: the reference's scan stops at lv-1
// (project_l1_Duchi!.jl:42-46), so its theta then comes from the lv-1 largest entries (see k_l1_cap).
template <typename T>
__global__ void __launch_bounds__(kThreads) k_absmin_key(i64 M, const T* __restrict__ v, unsigned long long* out,
                                                         const L1State* st) {
  if (st && !(st->theta >= 0.0 && st->C == st->M && st->M >= 2.0)) return;     // the cap applies to all-active vectors only
  unsigned long long k = ~0ull;
  for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < M; r += (i64)gridDim.x * blockDim.x) {
    const unsigned long long q = mag_key<T>(v[r]);
    k = q < k ? q : k;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long q = __shfl_xor_sync(0xffffffffu, k, o);
    k = q < k ? q : k;
  }
  if ((threadIdx.x & 31) == 0 && k != ~0ull) atomicMin(out, k);
}

// =============================================================================================
// cardinality: radix select of the k-th largest magnitude key (MSB-first digits of `dbits` bits:
// 11 on a single GPU — 3 levels for Float32 keys —, 8 on slabs where every level's histogram is all-reduced)
// =============================================================================================
struct SelState {
  unsigned long long prefix;      // digits decided so far (high bits)
  unsigned long long k_rem;       // rank still to locate inside the current prefix bucket (1-based)
  unsigned long long count_eq;    // elements whose key == final threshold
  unsigned long long hist[kSelBins];
  unsigned long long spec_above;                     // speculation (k_yl_spec): keys whose top digit exceeds the guess's,
  unsigned long long spec[(kSpecLevels - 1) * kSelBins];   //   histograms of levels 1.. ; consumed and cleared by k_sel_begin
  int bits_left;                  // undecided low bits of the key; <= 0 when finished
  int key_bits;
  int dbits;                      // digit width of this search
  int table_valid;                // the last level's per-block histograms are in the tie table (single GPU)
  int levels_run;                 // k_radix_hist launches of this search that histogrammed a level (the rest were decided
                                  //   by the speculation and returned at once); read by the select probe
};

// Choose the digit bucket that contains the k_rem-th largest key among the current prefix bucket, from the level
// histogram `h` (cleared on the way).  Called by all 256 threads of a block: every thread takes 2^w / 256 consecutive
// bins from the top down, a block-wide scan finds the thread whose bins hold the k-th largest key.
__device__ __forceinline__ void radix_pick_block(SelState* st, unsigned long long* h) {
  __shared__ unsigned long long s_wsum[8];
  __shared__ int s_bl;
  const int t = threadIdx.x;                       // blockDim.x == 256
  if (t == 0) s_bl = st->bits_left;
  __syncthreads();
  const int bl = s_bl;
  if (bl <= 0) return;                             // block-uniform
  const int w = min(st->dbits, bl);                // 8 <= w <= 11
  const int per = (1 << w) >> 8;                   // bins per thread: 1, 2, 4 or 8
  const unsigned long long k = st->k_rem;
  const int top = (1 << w) - 1 - t * per;
  unsigned long long c[8];
  unsigned long long sum = 0ull;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    c[j] = 0ull;
    if (j < per) {
      c[j] = h[top - j];
      h[top - j] = 0ull;
      sum += c[j];
    }
  }
  unsigned long long incl = sum;                   // inclusive scan over t (bins from the top down)
  const int lane = t & 31, wp = t >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long up = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += up;
  }
  if (lane == 31) s_wsum[wp] = incl;
  __syncthreads();                                 // (also orders every thread's read of k_rem before the winner's write)
  unsigned long long base = 0ull;
  for (int q = 0; q < wp; ++q) base += s_wsum[q];
  incl += base;
  const unsigned long long excl = incl - sum;      // keys in strictly higher bins than this thread's
  if (incl >= k && excl < k) {                     // exactly one thread
    unsigned long long cum = excl;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j < per) {
        if (cum + c[j] >= k) {
          st->k_rem = k - cum;
          st->count_eq = c[j];
          st->prefix = (st->prefix << w) | (unsigned long long)(top - j);
          st->bits_left = bl - w;
          break;
        }
        cum += c[j];
      }
    }
  }
  __syncthreads();                                 // the state and the scratch may be reused by a following call
}

// One level of the search: histogram of the next digit over the keys that match the decided prefix.
// chunk > 0 (single GPU): block b owns rows [b*chunk, (b+1)*chunk) — the partition of the tie kernels —, and the last
//   level leaves its per-block histogram in `table[b][*]`: the per-block tie counts are then a look-up (k_tie_count_p).
// chunk == 0 (slabs): grid-stride.
// fused != 0: the last block also picks the digit (single GPU); with slabs the histogram is all-reduced
// first and k_radix_pick runs afterwards.
template <typename T>
__global__ void __launch_bounds__(kThreads) k_radix_hist(i64 M, const T* __restrict__ v, SelState* st,
                                                         unsigned int* counter, int fused, i64 chunk,
                                                         unsigned int* __restrict__ table) {
  __shared__ unsigned int sh[kSelBins];
  const int bl = st->bits_left;
  if (bl <= 0) return;
  const int w = min(st->dbits, bl), shift = bl - w, nb = 1 << w;
  const unsigned long long mask = (unsigned long long)(nb - 1);
  const unsigned long long prefix = st->prefix;
  const bool all_match = bl >= st->key_bits;
  if (blockIdx.x == 0 && threadIdx.x == 0) st->levels_run += 1;
  for (int t = threadIdx.x; t < nb; t += blockDim.x) sh[t] = 0u;
  __syncthreads();
  // rows [lo, hi) of this block, visited with stride `step` after the block's / grid's first pass (chunk > 0: the block's
  // own contiguous chunk; else grid-stride over all rows); 16-byte loads when the vector is aligned (a chunk starts on a
  // multiple of 256 rows)
  i64 lo = 0, hi = M, first = (i64)blockIdx.x * blockDim.x + threadIdx.x, step = (i64)gridDim.x * blockDim.x;
  if (chunk > 0) {
    lo = (i64)blockIdx.x * chunk;
    hi = min(M, lo + chunk);
    first = threadIdx.x;
    step = blockDim.x;
  }
  auto add = [&](T val) {
    const unsigned long long key = mag_key<T>(val);
    const bool match = all_match ? true : ((key >> bl) == prefix);
    if (match) atomicAdd(&sh[(unsigned)((key >> shift) & mask)], 1u);
  };
  if (hi > lo) {
    if ((reinterpret_cast<unsigned long long>(v) & 15ull) == 0ull) {
      constexpr int VW = Vec<T>::W;
      const i64 nv = (hi - lo) / VW;
      for (i64 iv = first; iv < nv; iv += step) {
        T x4[VW];
        vload<T>(v + lo + iv * VW, x4);
#pragma unroll
        for (int e = 0; e < VW; ++e) add(x4[e]);
      }
      for (i64 r = lo + nv * VW + first; r < hi; r += step) add(v[r]);
    } else {
      for (i64 r = lo + first; r < hi; r += step) add(v[r]);
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < nb; t += blockDim.x)
    if (sh[t]) atomicAdd(&st->hist[t], (unsigned long long)sh[t]);
  const bool keep = table != nullptr && chunk > 0 && shift == 0;
  if (keep)
    for (int t = threadIdx.x; t < nb; t += blockDim.x) table[(size_t)blockIdx.x * kSelBins + t] = sh[t];
  if (fused) {
    if (last_block_ticket(counter)) {
      __threadfence();
      if (keep && threadIdx.x == 0) st->table_valid = 1;
      radix_pick_block(st, st->hist);
    }
  }
}
__global__ void __launch_bounds__(256) k_radix_pick(SelState* st) { radix_pick_block(st, st->hist); }

// Speculative levels of the cardinality search, accumulated by pass 1 of the y/l update while it produces v (k_yl_spec),
// around `guess` = the previous PARSDMM iteration's threshold.  Level 0 is not histogrammed at all (one shared-memory
// atomic per row, mostly on a handful of bins, cost 0.2 ms per 512^3 pass): the rows whose top digit EXCEEDS the guess's
// are counted in a register, and level j > 0 histograms digit j of the keys whose higher digits equal the guess's — a
// few per cent of the rows.  The threshold lies in the guess's top-digit bucket iff  above < k <= above + |bucket|
// (|bucket| = the total of the level-1 histogram); k_sel_begin then walks the levels for as long as the digits it
// decides agree with the guess, and the remaining levels run as ordinary k_radix_hist passes.  Exactness does not depend
// on the guess: a wrong guess only costs the passes it was meant to save.
template <typename T> struct NativeKey { typedef unsigned long long type; };
template <> struct NativeKey<float> { typedef unsigned int type; };       // Float32 keys: 32-bit integer arithmetic
template <typename T>
__device__ __forceinline__ void spec_hist_add(SpecCtx& sc, T v) {
  typedef typename NativeKey<T>::type K;
  constexpr int KB = (int)sizeof(T) * 8;
  const K key = (K)mag_key<T>(v), guess = (K)sc.guess;
  const unsigned d0 = (unsigned)(key >> (KB - kSpecBits));
  sc.above += (d0 > sc.g0) ? 1u : 0u;
  if (d0 == sc.g0) {
#pragma unroll
    for (int lv = 1; lv < kSpecLevels; ++lv) {
      const int bl = KB - kSpecBits * lv;                       // bits left at this level (> 0 for both key widths)
      const int w = bl < kSpecBits ? bl : kSpecBits;
      if (lv == 1 || (key >> bl) == (guess >> bl))
        atomicAdd(&sc.sh[(lv - 1) * kSelBins + (unsigned)((key >> (bl - w)) & (K)((1 << w) - 1))], 1u);
    }
  }
}

// nearest-neighbour resampling of a column-major box (multilevel warm starts): sample k of an axis reads source
// index floor(pos + 1/2) - 1 with pos = 1 + k (ns-1)/(nd-1), evaluated in exact integer arithmetic.
// Only the destination elements [q0, q1) of the box are written, to dst[0 .. q1-q0) (slabs: the rows a rank stores);
// the source is the whole box.
__device__ __forceinline__ long long nn_src_index(long long k, long long ns, long long nd) {
  if (nd <= 1) return 0;
  return (3 * (nd - 1) + 2 * k * (ns - 1)) / (2 * (nd - 1)) - 1;
}
template <typename T>
__global__ void __launch_bounds__(kThreads) k_resample_nn(const T* __restrict__ src, T* __restrict__ dst, i64 ns0,
                                                          i64 ns1, i64 ns2, i64 nd0, i64 nd1, i64 nd2, i64 q0, i64 q1) {
  for (i64 q = q0 + (i64)blockIdx.x * blockDim.x + threadIdx.x; q < q1; q += (i64)gridDim.x * blockDim.x) {
    const i64 i = q % nd0, t = q / nd0, j = t % nd1, kk = t / nd1;
    const i64 si = nn_src_index(i, ns0, nd0), sj = nn_src_index(j, ns1, nd1), sk = nn_src_index(kk, ns2, nd2);
    dst[q - q0] = src[si + ns0 * (sj + ns1 * sk)];
  }
}

// =============================================================================================
// per-fiber cardinality (project_cardinality!.jl:23-113, fiber modes): in every fiber of the
// transform-domain grid keep the k largest magnitudes (stable sortperm: among equal magnitudes the lower
// index inside the fiber wins) and zero the rest — a bit-serial radix select, in place.
// =============================================================================================
template <typename T> struct KeyBits;
template <> struct KeyBits<float> { static constexpr int n = 31; };
template <> struct KeyBits<double> { static constexpr int n = 63; };

// fibers along the fastest axis are contiguous: one warp per fiber, lanes strided over the fiber
template <typename T>
__global__ void __launch_bounds__(kThreads) k_card_fiber_contig(T* __restrict__ v, i64 nfib, unsigned L, long long k) {
  const int lane = threadIdx.x & 31;
  const i64 wpg = (i64)gridDim.x * (blockDim.x >> 5);
  for (i64 f = (i64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); f < nfib; f += wpg) {
    T* fib = v + f * (i64)L;
    if (k >= (long long)L) continue;
    if (k <= 0) {
      for (unsigned e = lane; e < L; e += 32) fib[e] = (T)0;
      continue;
    }
    unsigned long long prefix = 0ull;          // decided high bits of the k-th largest key
    unsigned long long need = (unsigned long long)k;   // rank still to locate among the keys matching the prefix
    for (int b = KeyBits<T>::n - 1; b >= 0; --b) {
      unsigned cnt = 0;
      for (unsigned e = lane; e < L; e += 32) {
        const unsigned long long key = mag_key<T>(fib[e]);
        cnt += ((key >> b) == ((prefix << 1) | 1ull)) ? 1u : 0u;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
      if ((unsigned long long)cnt >= need) prefix = (prefix << 1) | 1ull;
      else { need -= cnt; prefix = prefix << 1; }
    }
    // prefix = threshold key; `need` = how many of the ties survive (lowest indices first)
    unsigned long long seen = 0ull;
    for (unsigned e0 = 0; e0 < L; e0 += 32) {
      const unsigned e = e0 + lane;
      const unsigned long long key = e < L ? mag_key<T>(fib[e]) : 0ull;
      const bool tie = e < L && key == prefix;
      const unsigned bal = __ballot_sync(0xffffffffu, tie);
      const unsigned before = __popc(bal & ((1u << lane) - 1u));
      if (e < L && (key < prefix || (tie && seen + before >= need))) fib[e] = (T)0;
      seen += __popc(bal);
    }
  }
}

// slice modes (project_cardinality!.jl:122-129,138-145): permutedims + reshape so that every slice orthogonal to
// `axis` becomes one contiguous column, in the reference's element order inside the slice
//   axis 0: dst[(j + d1*k) + d1*d2*i]   axis 1: dst[(i + d0*k) + d0*d2*j]   (inverse != 0: the way back)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_slice_permute(const T* __restrict__ src, T* __restrict__ dst, unsigned d0,
                                                            unsigned d1, unsigned d2, int axis, int inverse) {
  const i64 n = (i64)d0 * d1 * d2;
  for (i64 q = (i64)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (i64)gridDim.x * blockDim.x) {
    const unsigned i = (unsigned)(q % d0);
    const unsigned j = (unsigned)((q / d0) % d1);
    const unsigned kk = (unsigned)(q / ((i64)d0 * d1));
    const i64 t = axis == 0 ? ((i64)j + (i64)d1 * kk) + (i64)d1 * d2 * i : ((i64)i + (i64)d0 * kk) + (i64)d0 * d2 * j;
    if (inverse) dst[q] = src[t];
    else dst[t] = src[q];
  }
}

// fibers along a slower axis: one thread per fiber, so that the lanes of a warp (neighbouring fibers) read
// neighbouring addresses at every step of the walk along the fiber
template <typename T>
__global__ void __launch_bounds__(kThreads) k_card_fiber_strided(T* __restrict__ v, unsigned d0, unsigned d1, unsigned d2,
                                                                 int axis, long long k) {
  const unsigned L = axis == 1 ? d1 : d2;
  const i64 stride = axis == 1 ? (i64)d0 : (i64)d0 * d1;
  const i64 nfib = axis == 1 ? (i64)d0 * d2 : (i64)d0 * d1;
  for (i64 f = (i64)blockIdx.x * blockDim.x + threadIdx.x; f < nfib; f += (i64)gridDim.x * blockDim.x) {
    T* fib = axis == 1 ? v + (f % d0) + (i64)d0 * d1 * (f / d0) : v + f;
    if (k >= (long long)L) continue;
    if (k <= 0) {
      for (unsigned e = 0; e < L; ++e) fib[e * stride] = (T)0;
      continue;
    }
    unsigned long long prefix = 0ull, need = (unsigned long long)k;
    for (int b = KeyBits<T>::n - 1; b >= 0; --b) {
      unsigned cnt = 0;
      for (unsigned e = 0; e < L; ++e) cnt += ((mag_key<T>(fib[e * stride]) >> b) == ((prefix << 1) | 1ull)) ? 1u : 0u;
      if ((unsigned long long)cnt >= need) prefix = (prefix << 1) | 1ull;
      else { need -= cnt; prefix = prefix << 1; }
    }
    unsigned long long seen = 0ull;
    for (unsigned e = 0; e < L; ++e) {
      const unsigned long long key = mag_key<T>(fib[e * stride]);
      if (key < prefix) fib[e * stride] = (T)0;
      else if (key == prefix) {
        if (seen >= need) fib[e * stride] = (T)0;
        ++seen;
      }
    }
  }
}

// =============================================================================================
// relaxed histogram projection (project_histogram_relaxed.jl:9-26): sort_ind = sortperm(x) — a stable sort in
// Julia's isless order (-0.0 < 0.0, NaN last) — then x[sort_ind[j]] = max(LB[j], min(x[sort_ind[j]], UB[j])).
// The permutation comes from a stable LSD radix sort of order-preserving integer keys (cub::DeviceRadixSort, library
// code) with the row index as payload; the two kernels here build the keys and apply the bounds through it.
// =============================================================================================
template <typename T> struct SortKey;
template <> struct SortKey<float> { typedef unsigned int type; };
template <> struct SortKey<double> { typedef unsigned long long type; };
template <typename T> __device__ __forceinline__ typename SortKey<T>::type isless_key(T v);
template <> __device__ __forceinline__ unsigned int isless_key<float>(float v) {
  if (v != v) return 0xffffffffu;
  const unsigned int u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
template <> __device__ __forceinline__ unsigned long long isless_key<double>(double v) {
  if (v != v) return ~0ull;
  const unsigned long long u = (unsigned long long)__double_as_longlong(v);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
template <typename T>
__global__ void __launch_bounds__(kThreads) k_hist_keys(i64 M, const T* __restrict__ v,
                                                        typename SortKey<T>::type* __restrict__ keys,
                                                        unsigned int* __restrict__ idx) {
  for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < M; r += (i64)gridDim.x * blockDim.x) {
    keys[r] = isless_key<T>(v[r]);
    idx[r] = (unsigned int)r;
  }
}
template <typename T>
__global__ void __launch_bounds__(kThreads) k_hist_apply(i64 M, T* __restrict__ v, const unsigned int* __restrict__ sorted_idx,
                                                         const T* __restrict__ lb, const T* __restrict__ ub) {
  for (i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x; j < M; j += (i64)gridDim.x * blockDim.x) {
    const unsigned int r = sorted_idx[j];
    T t = v[r];
    t = t_min<T>(t, ub[j]);          // x[j] = min(x[j], UB[j])     :15
    t = t_max<T>(lb[j], t);          // x[j] = max(LB[j], x[j])     :16
    v[r] = t;
  }
}

// fill helper
template <typename T>
__global__ void __launch_bounds__(kThreads) k_fill(i64 N, T* __restrict__ x, T val) {
  for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < N; r += (i64)gridDim.x * blockDim.x) x[r] = val;
}

}  // namespace sipb
