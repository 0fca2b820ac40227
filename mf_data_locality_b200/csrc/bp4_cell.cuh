// bp4_cell.cuh -- per-cell sum-factorisation phases of the BP4 vector-Laplace operator
// for one Q_p hexahedron with tri-linear geometry evaluated on the fly.
//
// Replaces the CPU SIMD kernels K1-K5 of the reference (SURVEY 2a):
//   read_dof_values_compressed        vector_access_reduced.h:51-283
//   LaplaceOperator::local_apply      poisson_operator.h:429-685 (3-D branch :534-666)
//   distribute_local_to_global_compr. vector_access_reduced.h:287-531
// It is NOT a translation of that code: the reference keeps one cell per SIMD lane and
// sweeps z-layers; here a thread block owns CPB cells and the work is cut into three
// register-blocked phases that each do two or three 1-D contractions per shared-memory
// round trip (B200 has 64 FP64 FMA/clk/SM but only 128 B/clk/SM of shared-memory
// bandwidth, so a line-per-thread scheme with one contraction per round trip would be
// shared-memory bound):
//
//   phase 1  item (comp c, node-row j)   : x-interp, z-interp, d/dzeta, d/dxi   -> smem
//   phase 2  item (qx, qz), all 3 comps  : y-interp, d/deta, Jacobian, G = w/det K^T K,
//                                          flux, d/deta^T, y-back-interp       -> smem
//   phase 3  item (comp c, node-row j)   : d/dxi^T, d/dzeta^T, z- and x-back-interp
//
// d/dxi and d/dzeta are taken *before* the y-interpolation (they commute with it), so
// phase 2 only ever needs y-lines and the three components of one quadrature point
// meet in one thread for the geometry.
//
// The same source is compiled by g++ for tests/emu (a CPU emulation of the thread loops
// used to check indexing without a GPU); the product never runs it on the CPU.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#  define BP4_HD __host__ __device__ __forceinline__
#  define BP4_UNROLL _Pragma("unroll")
#else
#  define BP4_HD inline
#  define BP4_UNROLL
#endif

namespace bp4
{
  // 1 / x without control flow: MUFU.RCP64H seed (~20 bits) + two Newton steps (-> < 1 ulp for
  // the well-scaled Jacobian determinants met here).  The IEEE division the compiler emits
  // carries a slow-path branch and convergence barriers per use, which keeps ptxas from
  // interleaving the Q independent quadrature points of a line.
  BP4_HD double rcp_nobranch(const double x)
  {
#ifdef __CUDA_ARCH__
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r        = fma(r, e, r);
    e        = fma(-x, r, 1.0);
    return fma(r, e, r);
#else
    return 1.0 / x;
#endif
  }
  // the FP32 form: MUFU.RCP seed (~23 bits with .ftz) + one Newton step
  BP4_HD float rcp_nobranch(const float x)
  {
#ifdef __CUDA_ARCH__
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    const float e = fmaf(-x, r, 1.0f);
    return fmaf(r, e, r);
#else
    return 1.0f / x;
#endif
  }

  // T = float: the same tables rounded to float, for the FP32 cell kernel
  template <int P, typename T = double>
  struct Tab
  {
    static constexpr int N = P + 1; // nodes per direction (GLL)
    static constexpr int Q = P + 2; // Gauss points per direction
    T S[N][Q];                      // S[i][q]  = l_i^GLL(x_q)            (shape_values)
    T Dn[N][Q];                     // Dn[i][q] = d/dx l_i^GLL(x_q)       (= S * D)
    T D[Q][Q];                      // D[i][q]  = d/dx l_i^Gauss(x_q)     (collocation gradient)
    T xq[Q];                        // Gauss points on [0,1]
    T wq[Q];                        // Gauss weights
    // even-odd halves (the role of deal.II's shape_values_eo / shape_gradients_collocation_eo,
    // poisson_operator.h:461-463): S[i][q] = S[N-1-i][Q-1-q], D and Dn change sign under the
    // same reflection.  Xf* pair the FIRST index (used when it is contracted), Xs* the SECOND:
    //   Xfp[i][q] = (X[i][q] + X[n-1-i][q]) / 2,  Xfm[i][q] = (X[i][q] - X[n-1-i][q]) / 2
    //   Xsp[i][q] = (X[i][q] + X[i][m-1-q]) / 2,  Xsm[i][q] = (X[i][q] - X[i][m-1-q]) / 2
    T Sfp[N][Q], Sfm[N][Q], Ssp[N][Q], Ssm[N][Q];
    T Dnfp[N][Q], Dnfm[N][Q], Dnsp[N][Q], Dnsm[N][Q];
    T Dfp[Q][Q], Dfm[Q][Q], Dsp[Q][Q], Dsm[Q][Q];
  };

  // ---------------------------------------------------------------------------------------
  // even-odd 1-D contractions on register arrays.  SG = +1: M[i][q] = M[NI-1-i][NO-1-q] (values),
  // SG = -1: M[i][q] = -M[NI-1-i][NO-1-q] (derivatives).  About half the multiplications of the
  // plain form: sums/differences of mirrored inputs meet the even/odd halves of the matrix, and
  // mirrored outputs are E + O and SG (E - O).
  // ---------------------------------------------------------------------------------------
  // out[q] = sum_i M[i][q] in[i]   (first index contracted; Mp/Mm = M's "f" halves)
  template <int NI, int NO, int SG, typename T>
  BP4_HD void eo_first(const T (&Mp)[NI][NO], const T (&Mm)[NI][NO], const T (&M)[NI][NO], const T (&in)[NI],
                       T (&out)[NO])
  {
    constexpr int HI = NI / 2, HO = NO / 2;
    T        e[HI > 0 ? HI : 1], o[HI > 0 ? HI : 1];
    BP4_UNROLL
    for (int i = 0; i < HI; ++i)
      {
        e[i] = in[i] + in[NI - 1 - i];
        o[i] = in[i] - in[NI - 1 - i];
      }
    BP4_UNROLL
    for (int q = 0; q < HO; ++q)
      {
        T E = Mp[0][q] * e[0], O = Mm[0][q] * o[0];
        BP4_UNROLL
        for (int i = 1; i < HI; ++i)
          {
            E += Mp[i][q] * e[i];
            O += Mm[i][q] * o[i];
          }
        if (NI % 2)
          E += M[HI][q] * in[HI];
        out[q]          = E + O;
        out[NO - 1 - q] = SG > 0 ? E - O : O - E;
      }
    if (NO % 2) // the middle output is its own mirror image: only one half contributes
      {
        T s;
        if (SG > 0)
          {
            s = Mp[0][HO] * e[0];
            BP4_UNROLL
            for (int i = 1; i < HI; ++i)
              s += Mp[i][HO] * e[i];
            if (NI % 2)
              s += M[HI][HO] * in[HI];
          }
        else
          {
            s = Mm[0][HO] * o[0];
            BP4_UNROLL
            for (int i = 1; i < HI; ++i)
              s += Mm[i][HO] * o[i];
          }
        out[HO] = s;
      }
  }

  // out[i] = sum_q M[i][q] in[q]   (second index contracted; Mp/Mm = M's "s" halves)
  template <int NI, int NO, int SG, typename T>
  BP4_HD void eo_second(const T (&Mp)[NI][NO], const T (&Mm)[NI][NO], const T (&M)[NI][NO], const T (&in)[NO],
                        T (&out)[NI])
  {
    constexpr int HI = NI / 2, HO = NO / 2;
    T        e[HO > 0 ? HO : 1], o[HO > 0 ? HO : 1];
    BP4_UNROLL
    for (int q = 0; q < HO; ++q)
      {
        e[q] = in[q] + in[NO - 1 - q];
        o[q] = in[q] - in[NO - 1 - q];
      }
    BP4_UNROLL
    for (int i = 0; i < HI; ++i)
      {
        T E = Mp[i][0] * e[0], O = Mm[i][0] * o[0];
        BP4_UNROLL
        for (int q = 1; q < HO; ++q)
          {
            E += Mp[i][q] * e[q];
            O += Mm[i][q] * o[q];
          }
        if (NO % 2)
          E += M[i][HO] * in[HO];
        out[i]          = E + O;
        out[NI - 1 - i] = SG > 0 ? E - O : O - E;
      }
    if (NI % 2)
      {
        T s;
        if (SG > 0)
          {
            s = Mp[HI][0] * e[0];
            BP4_UNROLL
            for (int q = 1; q < HO; ++q)
              s += Mp[HI][q] * e[q];
            if (NO % 2)
              s += M[HI][HO] * in[HO];
          }
        else
          {
            s = Mm[HI][0] * o[0];
            BP4_UNROLL
            for (int q = 1; q < HO; ++q)
              s += Mm[HI][q] * o[q];
          }
        out[HI] = s;
      }
  }

  template <int P>
  struct Geom // sizes and shared-memory strides of one cell slot
  {
    static constexpr int N   = P + 1;
    static constexpr int Q   = P + 2;
    static constexpr int N3  = N * N * N;
    static constexpr int ROWS = 3 * N;             // rows (c, j) per cell = phase 1/3 items
    // Both staging arrays are organised as one row per phase-1/3 item (cell, c, j) with an
    // ODD row stride: consecutive lanes of phase 1/3 then hit an arithmetic progression with
    // odd stride (a bijection modulo the 16 eight-byte banks) and the (qz, qx) lanes of
    // phase 2 hit consecutive addresses -> no shared-memory bank conflicts inside a cell (ncu:
    // none in phases 1 and 3; in phase 2 the warps that straddle two cells lose a wavefront,
    // the table-driven gather/scatter addresses conflict - DESIGN.md section 6).
    //   dofs[row][k][i]            staged cell DoFs
    //   work[row][a][qz][qx]       a = 0 value, 1 xi-derivative/flux, 2 zeta-derivative/flux
    static constexpr int RD  = (N * N) | 1;
    static constexpr int RW  = (3 * Q * Q) | 1;
    static constexpr int DOF = 3 * N3;             // DoFs of a cell
    static constexpr int DOFS = ROWS * RD;         // doubles of the dofs staging per cell
    static constexpr int WORK = ROWS * RW;         // doubles of the work staging per cell
    static constexpr int ITEMS13 = ROWS;           // phase 1/3 items per cell
    static constexpr int ITEMS2  = Q * Q;          // phase 2 items per cell
  };

  // entity code of a node coordinate: 0 left vertex, 1 interior, 2 right vertex
  template <int P>
  BP4_HD int ecode(int i)
  {
    return i == 0 ? 0 : (i == P ? 2 : 1);
  }

  // w-th node of a cell in entity-major order (entity a = ex + 3 ey + 9 ez ascending, nodes
  // lexicographic inside the entity: vector_access_reduced.h:176-258 addresses node `pos` of
  // entity a at idx[a] + 3 * pos + component), packed as
  //   bits 0-6  k*N+i (position inside the staging row) | bits 7-10 j (row) |
  //   bits 11-15 entity | bits 16-31 pos
  template <int P>
  inline void build_walk(uint32_t *walk)
  {
    constexpr int N = P + 1;
    int w = 0;
    for (int a = 0; a < 27; ++a)
      {
        const int e[3] = {a % 3, (a / 3) % 3, a / 9};
        int lo[3], hi[3];
        for (int d = 0; d < 3; ++d)
          {
            lo[d] = e[d] == 0 ? 0 : (e[d] == 1 ? 1 : P);
            hi[d] = e[d] == 0 ? 1 : (e[d] == 1 ? P : P + 1);
          }
        int pos = 0;
        for (int k = lo[2]; k < hi[2]; ++k)
          for (int j = lo[1]; j < hi[1]; ++j)
            for (int i = lo[0]; i < hi[0]; ++i, ++pos, ++w)
              walk[w] = uint32_t(k * N + i) | (uint32_t(j) << 7) | (uint32_t(a) << 11) | (uint32_t(pos) << 16);
      }
  }
  BP4_HD uint32_t walk_inrow(uint32_t pk) { return pk & 127u; }
  BP4_HD uint32_t walk_j(uint32_t pk) { return (pk >> 7) & 15u; }
  BP4_HD uint32_t walk_ent(uint32_t pk) { return (pk >> 11) & 31u; }
  BP4_HD uint32_t walk_pos(uint32_t pk) { return pk >> 16; }
  // staging offset of (component c, walk entry pk) inside a cell's dofs block
  template <int P>
  BP4_HD uint32_t dofs_offset(uint32_t pk, int c)
  {
    return (uint32_t(c) * Geom<P>::N + walk_j(pk)) * Geom<P>::RD + walk_inrow(pk);
  }

  // per-DoF gather/scatter table of a cell, r = 3 w + c in entity-major order (consecutive r
  // = consecutive addresses inside an entity's segment):
  //   bits 0-6 k*N+i (position in the staging row) | bits 7-11 row c*N+j | bits 12-16 entity |
  //   bits 17-31 3*pos + c (offset from the entity's first DoF)
  template <int P>
  inline void build_dof_table(uint32_t *tab)
  {
    uint32_t walk[Geom<P>::N3];
    build_walk<P>(walk);
    for (int w = 0; w < Geom<P>::N3; ++w)
      for (int c = 0; c < 3; ++c)
        tab[3 * w + c] = walk_inrow(walk[w]) | ((uint32_t(c) * Geom<P>::N + walk_j(walk[w])) << 7) |
                         (walk_ent(walk[w]) << 12) | ((3u * walk_pos(walk[w]) + c) << 17);
  }
  BP4_HD uint32_t dtab_inrow(uint32_t t) { return t & 127u; }
  BP4_HD uint32_t dtab_row(uint32_t t) { return (t >> 7) & 31u; }
  BP4_HD uint32_t dtab_ent(uint32_t t) { return (t >> 12) & 31u; }
  BP4_HD uint32_t dtab_rel(uint32_t t) { return t >> 17; }
  // offset inside a cell's dofs staging block (row stride RD) ...
  template <int P>
  BP4_HD uint32_t dtab_off(uint32_t t)
  {
    return dtab_row(t) * Geom<P>::RD + dtab_inrow(t);
  }
  // ... and inside its work block (row stride RW), where phase 3 may leave its result in place
  template <int P>
  BP4_HD uint32_t dtab_off_work(uint32_t t)
  {
    return dtab_row(t) * Geom<P>::RW + dtab_inrow(t);
  }

  // ---------------------------------------------------------------------------------------
  // phase 1: item = row (c, j).  dofs_row[k][i] -> work_row[{0,1,2}][qz][qx]
  // ---------------------------------------------------------------------------------------
  template <typename T>
  struct RowIn // staged DoFs of one row, dofs_row[k*N + i]
  {
    const T *p;
    BP4_HD T operator()(const int kk) const { return p[kk]; }
  };
  template <typename T>
  struct RowOut
  {
    T *p;
    BP4_HD void operator()(const int kk, const T v) const { p[kk] = v; }
  };
  template <int P, typename In, typename T>
  BP4_HD void phase1_io(const Tab<P, T> &tb, const In in, T *out)
  {
    using G         = Geom<P>;
    constexpr int N = G::N, Q = G::Q, HN = N / 2, HQ = Q / 2;
    T        t[N][Q];
    BP4_UNROLL
    for (int k = 0; k < N; ++k)
      {
        T r[N];
        BP4_UNROLL
        for (int i = 0; i < N; ++i)
          r[i] = in(k * N + i);
        eo_first<N, Q, 1>(tb.Sfp, tb.Sfm, tb.S, r, t[k]);
      }
    // z direction: rows k and N-1-k of t become their sum and difference, then every pair of
    // output layers (qz, Q-1-qz) shares the even and odd partial sums
    BP4_UNROLL
    for (int k = 0; k < HN; ++k)
      BP4_UNROLL
    for (int q = 0; q < Q; ++q)
      {
        const T e = t[k][q] + t[N - 1 - k][q], o = t[k][q] - t[N - 1 - k][q];
        t[k][q]         = e;
        t[N - 1 - k][q] = o;
      }
    BP4_UNROLL
    for (int qz = 0; qz < (Q + 1) / 2; ++qz)
      {
        const bool mid = (Q % 2) && qz == HQ; // the middle layer is its own mirror image
        T     uA[Q], uB[Q], zA[Q], zB[Q], sA[Q], sB[Q];
        BP4_UNROLL
        for (int q = 0; q < Q; ++q)
          {
            T Eu = tb.Sfp[0][qz] * t[0][q], Ou = tb.Sfm[0][qz] * t[N - 1][q];
            T Ez = tb.Dnfp[0][qz] * t[0][q], Oz = tb.Dnfm[0][qz] * t[N - 1][q];
            BP4_UNROLL
            for (int k = 1; k < HN; ++k)
              {
                Eu += tb.Sfp[k][qz] * t[k][q];
                Ou += tb.Sfm[k][qz] * t[N - 1 - k][q];
                Ez += tb.Dnfp[k][qz] * t[k][q];
                Oz += tb.Dnfm[k][qz] * t[N - 1 - k][q];
              }
            if (N % 2)
              {
                Eu += tb.S[HN][qz] * t[HN][q];
                Ez += tb.Dn[HN][qz] * t[HN][q];
              }
            if (mid)
              {
                uA[q] = Eu;
                zA[q] = Oz;
              }
            else
              {
                uA[q] = Eu + Ou;
                uB[q] = Eu - Ou;
                zA[q] = Ez + Oz;
                zB[q] = Oz - Ez;
              }
          }
        eo_first<Q, Q, -1>(tb.Dfp, tb.Dfm, tb.D, uA, sA);
        BP4_UNROLL
        for (int q = 0; q < Q; ++q)
          {
            out[0 * Q * Q + qz * Q + q] = uA[q];
            out[1 * Q * Q + qz * Q + q] = sA[q];
            out[2 * Q * Q + qz * Q + q] = zA[q];
          }
        if (!mid)
          {
            eo_first<Q, Q, -1>(tb.Dfp, tb.Dfm, tb.D, uB, sB);
            BP4_UNROLL
            for (int q = 0; q < Q; ++q)
              {
                out[0 * Q * Q + (Q - 1 - qz) * Q + q] = uB[q];
                out[1 * Q * Q + (Q - 1 - qz) * Q + q] = sB[q];
                out[2 * Q * Q + (Q - 1 - qz) * Q + q] = zB[q];
              }
          }
      }
  }

  // ---------------------------------------------------------------------------------------
  // fine-grained phases 1 and 3 for the high degrees.  With few cells per block the 3N rows
  // (c, j) of a cell are too few items for 128 threads (Q8: 27), and one row's t[N][Q] no longer
  // fits the register file.  Here every 1-D contraction is its own sweep with a block barrier
  // in between, one line per item, in place in the row:
  //   1a (row, k ): dofs[k][:]            -> t[k][:]      kept in the d/dzeta slots
  //   1b (row, qx): t[:][qx]              -> u[:][qx], d/dzeta[:][qx]   (own column, in place)
  //   1c (row, qz): u[qz][:]              -> d/dxi[qz][:]
  //   3a (row, qz): v[qz][:], fx[qz][:]   -> v[qz][:] += D fx
  //   3b (row, qx): v[:][qx], fz[:][qx]   -> t[:][qx]     (own column of the d/dzeta slots)
  //   3c (row, k ): t[k][:]               -> result[k][:]
  // Same FMAs as phase1/phase3, (N + Q) registers of data per item, Q or N independent chains.
  // The matrix entries stay compile-time constant-bank operands: the line index only selects data.
  // ---------------------------------------------------------------------------------------
  template <int P, typename T>
  BP4_HD void phase1a(const Tab<P, T> &tb, T *row, const int k)
  {
    constexpr int N = Geom<P>::N, Q = Geom<P>::Q;
    T        r[N];
    BP4_UNROLL
    for (int i = 0; i < N; ++i)
      r[i] = row[k * N + i];
    T o[Q];
    eo_first<N, Q, 1>(tb.Sfp, tb.Sfm, tb.S, r, o);
    BP4_UNROLL
    for (int q = 0; q < Q; ++q)
      row[2 * Q * Q + k * Q + q] = o[q];
  }

  template <int P, typename T>
  BP4_HD void phase1b(const Tab<P, T> &tb, T *row, const int qx)
  {
    constexpr int N = Geom<P>::N, Q = Geom<P>::Q;
    T        t[N];
    BP4_UNROLL
    for (int k = 0; k < N; ++k)
      t[k] = row[2 * Q * Q + k * Q + qx];
    T su[Q], sz[Q];
    eo_first<N, Q, 1>(tb.Sfp, tb.Sfm, tb.S, t, su);
    eo_first<N, Q, -1>(tb.Dnfp, tb.Dnfm, tb.Dn, t, sz);
    BP4_UNROLL
    for (int qz = 0; qz < Q; ++qz)
      {
        row[0 * Q * Q + qz * Q + qx] = su[qz];
        row[2 * Q * Q + qz * Q + qx] = sz[qz];
      }
  }

  template <int P, typename T>
  BP4_HD void phase1c(const Tab<P, T> &tb, T *row, const int qz)
  {
    constexpr int Q = Geom<P>::Q;
    T        u[Q];
    BP4_UNROLL
    for (int i = 0; i < Q; ++i)
      u[i] = row[qz * Q + i];
    T sx[Q];
    eo_first<Q, Q, -1>(tb.Dfp, tb.Dfm, tb.D, u, sx);
    BP4_UNROLL
    for (int q = 0; q < Q; ++q)
      row[1 * Q * Q + qz * Q + q] = sx[q];
  }

  template <int P, typename T>
  BP4_HD void phase3a(const Tab<P, T> &tb, T *row, const int qz)
  {
    constexpr int Q = Geom<P>::Q;
    T        fx[Q];
    BP4_UNROLL
    for (int q = 0; q < Q; ++q)
      fx[q] = row[1 * Q * Q + qz * Q + q];
    T d[Q];
    eo_second<Q, Q, -1>(tb.Dsp, tb.Dsm, tb.D, fx, d);
    BP4_UNROLL
    for (int i = 0; i < Q; ++i)
      row[qz * Q + i] += d[i];
  }

  template <int P, typename T>
  BP4_HD void phase3b(const Tab<P, T> &tb, T *row, const int qx)
  {
    constexpr int N = Geom<P>::N, Q = Geom<P>::Q;
    T        v[Q], fz[Q];
    BP4_UNROLL
    for (int qz = 0; qz < Q; ++qz)
      {
        v[qz]  = row[0 * Q * Q + qz * Q + qx];
        fz[qz] = row[2 * Q * Q + qz * Q + qx];
      }
    T sv[N], sf[N];
    eo_second<N, Q, 1>(tb.Ssp, tb.Ssm, tb.S, v, sv);
    eo_second<N, Q, -1>(tb.Dnsp, tb.Dnsm, tb.Dn, fz, sf);
    BP4_UNROLL
    for (int k = 0; k < N; ++k)
      row[2 * Q * Q + k * Q + qx] = sv[k] + sf[k];
  }

  template <int P, typename T>
  BP4_HD void phase3c(const Tab<P, T> &tb, T *row, const int k)
  {
    constexpr int N = Geom<P>::N, Q = Geom<P>::Q;
    T        t[Q];
    BP4_UNROLL
    for (int q = 0; q < Q; ++q)
      t[q] = row[2 * Q * Q + k * Q + q];
    T o[N];
    eo_second<N, Q, 1>(tb.Ssp, tb.Ssm, tb.S, t, o);
    BP4_UNROLL
    for (int i = 0; i < N; ++i)
      row[k * N + i] = o[i];
  }

  // ---------------------------------------------------------------------------------------
  // phase 2: item = (qx, qz), all three components, one y-line of quadrature points.
  // QUAD = false: cf = tri-linear coefficients [8][3] in the order v0,v1,v3,v4,v9,v10,v12,v13
  // (the ones LaplaceOperator::initialize fills, poisson_operator.h:165-177);
  // QUAD = true : cf = all 27 coefficients [27][3] of X = sum v_{a+3b+9c} xi^a eta^b zeta^c, the
  // form local_apply evaluates (poisson_operator.h:577-602).
  // x = xq[qx], z = xq[qz], wxz = wq[qx]*wq[qz].
  // ---------------------------------------------------------------------------------------
  template <int P, bool QUAD = false, typename T = double>
  BP4_HD void phase2(const Tab<P, T> &tb, const T *cf, T *work, const int qx, const int qz,
                     const T x, const T z, const T wxz)
  {
    using G         = Geom<P>;
    constexpr int N = G::N, Q = G::Q;
    // --- geometry of the whole y-line first: G = (w / det) K^T K, six entries per point.
    // rows of dX/dxi_e; along the line they are polynomials in y whose coefficients are
    // collapsed in zeta and xi once per line:
    //   tri-linear: r0 = dX/dxi   = (v1 + z v10) + y (v4 + z v13)
    //               r1 = dX/deta  = (v3 + z v12) + x (v4 + z v13)      (constant along the line)
    //               r2 = dX/dzeta = (v9 + x v10) + y (v12 + x v13)
    //   quadratic : r0, r2 quadratic and r1 linear in y (same collapse order as the reference:
    //               xi_i = v_i + z (v_{9+i} + z v_{18+i}), di_i = v_{9+i} + 2 z v_{18+i})
    T g00[Q], g01[Q], g02[Q], g11[Q], g12[Q], g22[Q];
    {
      constexpr int NB = QUAD ? 3 : 2; // coefficients in y of r0 and r2
      T        A[NB][3], Cc[NB][3], R1[2][3];
      BP4_UNROLL
      for (int d = 0; d < 3; ++d)
        {
          if constexpr (!QUAD)
            {
              const T v1 = cf[3 + d], v3 = cf[6 + d], v4 = cf[9 + d], v9 = cf[12 + d],
                           v10 = cf[15 + d], v12 = cf[18 + d], v13 = cf[21 + d];
              A[0][d]  = v1 + z * v10;
              A[1][d]  = v4 + z * v13;
              R1[0][d] = (v3 + z * v12) + x * A[1][d];
              R1[1][d] = T(0);
              Cc[0][d] = v9 + x * v10;
              Cc[1][d] = v12 + x * v13;
            }
          else
            {
              T xi[9], di[9];
              BP4_UNROLL
              for (int i = 0; i < 9; ++i)
                {
                  xi[i] = cf[3 * i + d] + z * (cf[3 * (9 + i) + d] + z * cf[3 * (18 + i) + d]);
                  di[i] = cf[3 * (9 + i) + d] + (z + z) * cf[3 * (18 + i) + d];
                }
              BP4_UNROLL
              for (int b = 0; b < 3; ++b)
                {
                  A[b][d]  = xi[1 + 3 * b] + (x + x) * xi[2 + 3 * b];
                  Cc[b][d] = di[3 * b] + x * (di[3 * b + 1] + x * di[3 * b + 2]);
                }
              R1[0][d] = xi[3] + x * (xi[4] + x * xi[5]);
              R1[1][d] = xi[6] + x * (xi[7] + x * xi[8]);
            }
        }
      BP4_UNROLL
      for (int q = 0; q < Q; ++q)
        {
          const T y = tb.xq[q];
          T       r0[3], r1[3], r2[3];
          BP4_UNROLL
          for (int d = 0; d < 3; ++d)
            {
              if constexpr (!QUAD)
                {
                  r0[d] = A[0][d] + y * A[1][d];
                  r1[d] = R1[0][d];
                  r2[d] = Cc[0][d] + y * Cc[1][d];
                }
              else
                {
                  r0[d] = A[0][d] + y * (A[1][d] + y * A[NB - 1][d]);
                  r1[d] = R1[0][d] + (y + y) * R1[1][d];
                  r2[d] = Cc[0][d] + y * (Cc[1][d] + y * Cc[NB - 1][d]);
                }
            }
          // columns of adj: k0 = r1 x r2, k1 = r2 x r0, k2 = r0 x r1;  det = r0 . k0
          // (the cofactor inverse of poisson_operator.h:41-63 without the division)
          T k0[3], k1[3], k2[3];
          k0[0] = r1[1] * r2[2] - r1[2] * r2[1];
          k0[1] = r1[2] * r2[0] - r1[0] * r2[2];
          k0[2] = r1[0] * r2[1] - r1[1] * r2[0];
          k1[0] = r2[1] * r0[2] - r2[2] * r0[1];
          k1[1] = r2[2] * r0[0] - r2[0] * r0[2];
          k1[2] = r2[0] * r0[1] - r2[1] * r0[0];
          k2[0] = r0[1] * r1[2] - r0[2] * r1[1];
          k2[1] = r0[2] * r1[0] - r0[0] * r1[2];
          k2[2] = r0[0] * r1[1] - r0[1] * r1[0];
          const T det = r0[0] * k0[0] + r0[1] * k0[1] + r0[2] * k0[2];
          // == det * w * J^-1 J^-T  (poisson_operator.h:604-625)
          const T sc = (wxz * tb.wq[q]) * rcp_nobranch(det);
          g00[q]          = sc * (k0[0] * k0[0] + k0[1] * k0[1] + k0[2] * k0[2]);
          g01[q]          = sc * (k0[0] * k1[0] + k0[1] * k1[1] + k0[2] * k1[2]);
          g02[q]          = sc * (k0[0] * k2[0] + k0[1] * k2[1] + k0[2] * k2[2]);
          g11[q]          = sc * (k1[0] * k1[0] + k1[1] * k1[1] + k1[2] * k1[2]);
          g12[q]          = sc * (k1[0] * k2[0] + k1[1] * k2[1] + k1[2] * k2[2]);
          g22[q]          = sc * (k2[0] * k2[0] + k2[1] * k2[1] + k2[2] * k2[2]);
        }
    }
    // --- the three components one after the other (a rolled loop: the unrolled body of one
    // component is ~1/3 of the instruction footprint, which matters with two warps per
    // scheduler and a 32 KB instruction cache)
#ifdef __CUDACC__
#  pragma unroll 1
#endif
    for (int c = 0; c < 3; ++c)
      {
        T *base = work + (c * N) * G::RW + qz * Q + qx; // rows (c, j), j = 0..N-1
        T  gx[Q], gy[Q], gz[Q], v[Q], a0[N], a1[N], a2[N];
        BP4_UNROLL
        for (int j = 0; j < N; ++j)
          {
            a0[j] = base[j * G::RW];
            a1[j] = base[j * G::RW + Q * Q];
            a2[j] = base[j * G::RW + 2 * Q * Q];
          }
        // y-interpolation of value, xi-derivative and zeta-derivative lines, then d/deta
        eo_first<N, Q, 1>(tb.Sfp, tb.Sfm, tb.S, a0, v);
        eo_first<N, Q, 1>(tb.Sfp, tb.Sfm, tb.S, a1, gx);
        eo_first<N, Q, 1>(tb.Sfp, tb.Sfm, tb.S, a2, gz);
        eo_first<Q, Q, -1>(tb.Dfp, tb.Dfm, tb.D, v, gy);
        // flux = G grad
        BP4_UNROLL
        for (int q = 0; q < Q; ++q)
          {
            const T a = gx[q], b = gy[q], e = gz[q];
            gx[q] = g00[q] * a + g01[q] * b + g02[q] * e;
            gy[q] = g01[q] * a + g11[q] * b + g12[q] * e;
            gz[q] = g02[q] * a + g12[q] * b + g22[q] * e;
          }
        // d/deta^T on the eta-flux -> value-like line, then y-back-interpolation of the three lines
        eo_second<Q, Q, -1>(tb.Dsp, tb.Dsm, tb.D, gy, v);
        eo_second<N, Q, 1>(tb.Ssp, tb.Ssm, tb.S, v, a0);
        eo_second<N, Q, 1>(tb.Ssp, tb.Ssm, tb.S, gx, a1);
        eo_second<N, Q, 1>(tb.Ssp, tb.Ssm, tb.S, gz, a2);
        BP4_UNROLL
        for (int j = 0; j < N; ++j)
          {
            base[j * G::RW]             = a0[j];
            base[j * G::RW + Q * Q]     = a1[j];
            base[j * G::RW + 2 * Q * Q] = a2[j];
          }
      }
  }

  // ---------------------------------------------------------------------------------------
  // phase 3: item = row (c, j).  work_row[{0,1,2}][qz][qx] -> dofs_row[k][i]
  // ---------------------------------------------------------------------------------------
  template <int P, typename T>
  BP4_HD void phase1(const Tab<P, T> &tb, const T *in, T *out)
  {
    phase1_io<P>(tb, RowIn<T>{in}, out);
  }

  template <int P, typename Out, typename T>
  BP4_HD void phase3_io(const Tab<P, T> &tb, const T *in, const Out out)
  {
    using G         = Geom<P>;
    constexpr int N = G::N, Q = G::Q, HN = N / 2, HQ = Q / 2;
    // X = (even part of S^T v) + (odd part of Dn^T fz), Y = (odd of S^T v) + (even of Dn^T fz):
    // t[k] = X[k] + Y[k], t[N-1-k] = X[k] - Y[k]
    T X[(N + 1) / 2][Q], Y[HN > 0 ? HN : 1][Q];
    BP4_UNROLL
    for (int qz = 0; qz < (Q + 1) / 2; ++qz)
      {
        const bool mid = (Q % 2) && qz == HQ;
        T     vA[Q], fA[Q], zA[Q], vB[Q], fB[Q], zB[Q], d[Q];
        BP4_UNROLL
        for (int q = 0; q < Q; ++q)
          {
            vA[q] = in[0 * Q * Q + qz * Q + q];
            fA[q] = in[1 * Q * Q + qz * Q + q];
            zA[q] = in[2 * Q * Q + qz * Q + q];
          }
        eo_second<Q, Q, -1>(tb.Dsp, tb.Dsm, tb.D, fA, d);
        BP4_UNROLL
        for (int q = 0; q < Q; ++q)
          vA[q] += d[q];
        if (!mid)
          {
            BP4_UNROLL
            for (int q = 0; q < Q; ++q)
              {
                vB[q] = in[0 * Q * Q + (Q - 1 - qz) * Q + q];
                fB[q] = in[1 * Q * Q + (Q - 1 - qz) * Q + q];
                zB[q] = in[2 * Q * Q + (Q - 1 - qz) * Q + q];
              }
            eo_second<Q, Q, -1>(tb.Dsp, tb.Dsm, tb.D, fB, d);
            BP4_UNROLL
            for (int q = 0; q < Q; ++q)
              {
                const T vb = vB[q] + d[q];
                const T ev = vA[q] + vb, ov = vA[q] - vb, ef = zA[q] + zB[q], of = zA[q] - zB[q];
                BP4_UNROLL
                for (int k = 0; k < (N + 1) / 2; ++k)
                  {
                    const T x = tb.Ssp[k][qz] * ev + tb.Dnsm[k][qz] * of;
                    X[k][q]        = qz == 0 ? x : X[k][q] + x;
                  }
                BP4_UNROLL
                for (int k = 0; k < HN; ++k)
                  {
                    const T y = tb.Ssm[k][qz] * ov + tb.Dnsp[k][qz] * ef;
                    Y[k][q]        = qz == 0 ? y : Y[k][q] + y;
                  }
              }
          }
        else
          {
            BP4_UNROLL
            for (int q = 0; q < Q; ++q)
              {
                BP4_UNROLL
                for (int k = 0; k < (N + 1) / 2; ++k)
                  X[k][q] += tb.S[k][qz] * vA[q];
                BP4_UNROLL
                for (int k = 0; k < HN; ++k)
                  Y[k][q] += tb.Dn[k][qz] * zA[q];
              }
          }
      }
    BP4_UNROLL
    for (int k = 0; k < (N + 1) / 2; ++k)
      {
        T tA[Q], tB[Q], o[N];
        BP4_UNROLL
        for (int q = 0; q < Q; ++q)
          {
            tA[q] = k < HN ? X[k][q] + Y[k < HN ? k : 0][q] : X[k][q];
            tB[q] = k < HN ? X[k][q] - Y[k < HN ? k : 0][q] : T(0);
          }
        eo_second<N, Q, 1>(tb.Ssp, tb.Ssm, tb.S, tA, o);
        BP4_UNROLL
        for (int i = 0; i < N; ++i)
          out(k * N + i, o[i]);
        if (k < HN)
          {
            eo_second<N, Q, 1>(tb.Ssp, tb.Ssm, tb.S, tB, o);
            BP4_UNROLL
            for (int i = 0; i < N; ++i)
              out((N - 1 - k) * N + i, o[i]);
          }
      }
  }

  template <int P, typename T>
  BP4_HD void phase3(const Tab<P, T> &tb, const T *in, T *out)
  {
    phase3_io<P>(tb, in, RowOut<T>{out});
  }
} // namespace bp4
