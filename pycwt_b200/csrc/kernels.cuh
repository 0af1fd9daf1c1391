// Kernel bodies of the CWT engine.  Every kernel is a `Body` struct with
//   Args, NPHASE, SMEM (bytes), and  template<int PH> phase(args, bx, by, tid, smem)
// Phases are separated by a CTA barrier.  The generic __global__ wrapper lives in
// engine.cu; tests/emu runs the same phases sequentially on the CPU.
#pragma once
#include <math.h>
#include "fft_tile.cuh"

namespace cwtb {

// ---- per-scale descriptor (host-planned, read by the kernels) -------------------
struct ScaleDesc {
  double s;        // scale s_j
  double amp;      // sqrt(s*w1*Np) * family constant / Np
  int row;         // output row of W (after NaN-row removal, done by the host)
  int k_lo, k_hi;  // signed band limits (inclusive) outside which psi_ft is treated as 0
  int log2K;       // pruned transform length K' = 1 << log2K  (K' == Np: dense)
  int rsplit;      // residue r >= rsplit  <->  signed bin k = r - K'
  int trow;        // row in the caller's psi_ft table (CWTB_TABLE family)
  int chan;        // channel of a batched transform: spectrum at spec + chan*Np
  int pad_;
  long long boff;  // offset of this scale's band product B[] in the band buffer
  // ---- band-limited expansion path (ip_log2Nc > 0; see ExpandBody) ----
  int ip_log2Nc;   // coarse grid length Nc = 1 << ip_log2Nc  (0: exact pruned-transform path)
  int ip_kc;       // centre bin of the band (signed): the coarse grid holds the band shifted to 0
  int ip_w;        // taps of the interpolation kernel
  int ip_pad_;
  long long ip_coff;   // offset of this row's Nc coarse samples in the coarse buffers
  long long ip_woff;   // offset of the [taps][R] weight table of this row's class
  double ip_beta;      // Kaiser-Bessel shape parameter
  double ip_dc;        // I0(beta) / taps: 1 / (transform of the kernel) = ip_dc * z / sinh(z)
};

struct Fam {
  int family;      // 0 Morlet, 1 Paul, 2 DOG, 3 table
  int m;           // order (Paul, DOG)
  int unit;        // multiply by i^unit  (conj(-(1j**m)) for DOG)
  int pad_;
  double f0;       // Morlet wavenumber
  double dw;       // 1 / (Np * dt)   (numpy fftfreq's `val`)
  const double2 *table;  // [S][Np] complex128: sqrt(s*w1*Np)*conj(psi_ft)  (family 3)
  long long tpitch;
};

HD double ipow(double f, int m) {
  double r = 1.0, b = f;
  int e = m < 0 ? -m : m;
  while (e) { if (e & 1) r *= b; b *= b; e >>= 1; }
  return m < 0 ? 1.0 / r : r;
}

// |conj(psi_ft(s*w_k))| without the family constant; pycwt/mothers.py:26-28,118-122,170-173.
// w_k is formed as numpy does: 2*pi * (k * (1/(Np*dt))).
HD double amp_eval(const Fam &fp, double s, int k) {
  const double w = 6.283185307179586 * ((double)k * fp.dw);
  const double f = s * w;
  if (fp.family == 0) {
    const double d = f - fp.f0;
    return exp(-0.5 * d * d);
  } else if (fp.family == 1) {
    return f > 0.0 ? ipow(f, fp.m) * exp(-f) : 0.0;
  } else {
    return ipow(f, fp.m) * exp(-0.5 * f * f);
  }
}

// the same in the engine's arithmetic: the fp32 engine forms f = s*w in double (w spans 2^18 bins)
// and evaluates the power and the exponential in float (the caller keeps orders above 8 in double:
// their powers overflow float).  fp64 instructions run at half the fp32 rate on B200: one double exp per band product made
// the band-product launches and the generating first kernel fp64-pipe bound in the fp32 engine.
template <typename T> HD T amp_eval_t(const Fam &fp, double s, int k) {
  if constexpr (sizeof(T) == 8) {
    return amp_eval(fp, s, k);
  } else {
    const double w = 6.283185307179586 * ((double)k * fp.dw);
    const double f = s * w;
    if (fp.family == 0) {
      const float d = (float)(f - fp.f0);
      return expf(-0.5f * d * d);
    }
    const float ff = (float)f;
    float r = 1.0f, b = ff;
    for (int e = fp.m; e; e >>= 1) { if (e & 1) r *= b; b *= b; }
    if (fp.family == 1) return ff > 0.0f ? r * expf(-ff) : 0.0f;
    return r * expf(-0.5f * ff * ff);
  }
}

template <typename T> HD cx<T> rot_unit(cx<T> v, int unit) {
  switch (unit & 3) {
    case 1: return mk<T>(-v.y, v.x);
    case 2: return mk<T>(-v.x, -v.y);
    case 3: return mk<T>(v.y, -v.x);
    default: return v;
  }
}

// value of x^[bin] * conj(psi_ft)(s, k) * norm / Np  for one scale
template <typename T>
HD cx<T> band_value(const Fam &fp, const ScaleDesc &d, const cx<T> *spec, unsigned bin, int k, unsigned N) {
  cx<T> v = ldg(&spec[(size_t)d.chan * N + bin]);
  if (fp.family == 3) {
    double2 t = ldg(&fp.table[(size_t)d.trow * fp.tpitch + bin]);
    cx<T> tt = mk<T>((T)(t.x * d.amp), (T)(t.y * d.amp));
    return cmul(v, tt);
  }
  // (orders above 8: value and normalisation only combine to a float-range number in double)
  const T a = (sizeof(T) == 8 || (fp.family != 0 && fp.m > 8)) ? (T)(amp_eval(fp, d.s, k) * d.amp)
                                                               : (T)(amp_eval_t<T>(fp, d.s, k) * (T)d.amp);
  return rot_unit<T>(cscale(v, a), fp.unit);
}

// ---- storers -------------------------------------------------------------------
// final output: out[row][u + q*U], u = u0 + b, trimmed to n < nout.
// Epilogues fused into the store:
//   EPI_STORE      out = x
//   EPI_MULCONJ    out = out * conj(x)          (cross-wavelet: second transform of xwt)
//   EPI_GAUSS      out = x * exp(g * k_n^2) * post, k_n = 2 pi fftfreq(nfreq)[n]
//                  (time-smoothing filter of Morlet.smooth applied to a forward transform)
enum { EPI_STORE = 0, EPI_MULCONJ = 1, EPI_GAUSS = 2 };
template <typename T> struct Epilogue {
  int mode;
  double g;        // EPI_GAUSS: -0.5 * (s/dt)^2 of this row
  double invn;     // 1 / nfreq
  double post;     // extra real factor (1/npad of the following inverse transform)
  long long nfreq;
  HD cx<T> apply(cx<T> x, cx<T> old, long long n) const {
    if (mode == EPI_MULCONJ) return cmul(old, cconj(x));
    if (mode == EPI_GAUSS) {
      const long long qs = n < nfreq / 2 ? n : n - nfreq;   // numpy fftfreq ordering
      const double k = 6.283185307179586 * ((double)qs * invn);
      const T f = (T)(exp(g * (k * k)) * post);
      return cscale(x, f);
    }
    return x;
  }
};
template <typename T> struct OutStorer {
  using V = cx<T>;
  V *row;          // out + row*pitch
  long long nout;  // keep final index < nout
  int u0, U;
  Epilogue<T> epi;
  int ostride = 1, ooff = 0;   // final index = n*ostride + ooff (interleaved sub-transforms, Np > 2^20)
  template <int R> HD void store(int b, int ql, int qs, V (&x)[R]) const {
    const int u = u0 + b;
    if (u >= U) return;
    size_t step = (size_t)qs * (size_t)U;
    size_t n = (size_t)u + (size_t)ql * (size_t)U;
    if (ostride != 1) { n = n * (size_t)ostride + (size_t)ooff; step *= (size_t)ostride; }
    if (epi.mode == EPI_STORE && (long long)(n + (R - 1) * step) < nout) {
      // common case: every output of this butterfly is kept -> pointer walk, no per-element test
      V *p = row + n;
#pragma unroll
      for (int c = 0; c < R; ++c) { st_stream(p, x[c]); p += step; }
      return;
    }
#pragma unroll
    for (int c = 0; c < R; ++c, n += step) {
      if ((long long)n < nout) {
        if (epi.mode == EPI_STORE) st_stream(&row[n], x[c]);
        else row[n] = epi.apply(x[c], epi.mode == EPI_MULCONJ ? row[n] : x[c], (long long)n);
      }
    }
  }
};

// first-kernel output: Z[(p + q*M)*K2 + r2] = x_q * e^{SIGN 2 pi i r2 (p+qM)/N}
template <typename T, int SIGN> struct ZStorer {
  using V = cx<T>;
  V *Z;
  NTab nt;
  int p, M, r20, bmax;
  unsigned K2 = K2C;   // row length of Z
  int cached_b = -1;   // the step factor depends on b only: looked up once per thread
  V cached_st;
  template <int R> HD void store(int b, int ql, int qs, V (&x)[R]) {
    if (b >= bmax) return;
    const unsigned r2 = (unsigned)(r20 + b);
    const unsigned u = (unsigned)(p + ql * M);
    const unsigned du = (unsigned)(qs * M);
    V t = nroot_t<T>(nt, r2 * u);
    if (b != cached_b) {
      cached_st = nroot_t<T>(nt, r2 * du);
      if (SIGN < 0) cached_st.y = -cached_st.y;
      cached_b = b;
    }
    const V st = cached_st;
    if (SIGN < 0) t.y = -t.y;
    V *dst = Z + (size_t)u * K2 + r2;
#pragma unroll
    for (int c = 0; c < R; ++c) {
      dst[(size_t)c * du * K2] = cmul(x[c], t);
      t = cmul(t, st);
    }
  }
};

// ---- Body: single-kernel pruned inverse transform (K' <= 1024) -------------------
template <typename T> struct SingleArgs {
  const ScaleDesc *descs;  // device
  const cx<T> *Bbuf;       // band products
  cx<T> *W;                // [rows][n0]
  const cx<T> *tw;         // pass twiddle tables (fft_tile.cuh: tw_offset)
  NTab nt;
  long long n0;
  unsigned N;
  int first;               // descs[first + blockIdx.y]
  int epi;                 // EPI_STORE / EPI_MULCONJ
};

template <typename T, int K> struct SingleBody {
  static constexpr int NTB = TileCfg<T>::NT;   // threads per CTA of this kernel
  static constexpr int NT = NTB;
  using V = cx<T>;
  using Args = SingleArgs<T>;
  using LY = Lay<T, K>;
  static constexpr int NP = Plan<K>::NP;
  static_assert(NP >= 2, "single-kernel path needs a multi-pass plan");
  static constexpr int NPHASE = NP;
  static constexpr size_t SMEM = LY::BYTES;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *smraw) {
    V *sm = (V *)smraw;
    const ScaleDesc d = a.descs[a.first + by];
    const int M = (int)(a.N / K);
    const int p0 = bx * LY::P;
    if constexpr (PH == 0) {
      GenLoader<T, K, Plan<K>::R1> ld;
      ld.B = a.Bbuf + d.boff;
      ld.nt = a.nt;
      ld.rsplit = d.rsplit;
      ld.p0 = (unsigned)p0;
      tile_first<T, K, +1>(sm, a.tw, ld, tid);
    } else if constexpr (PH == 1 && NP == 3) {
      tile_second<T, K, +1>(sm, a.tw, tid);
    } else {
      OutStorer<T> st;
      st.row = a.W + (size_t)d.row * a.n0;
      st.nout = a.n0;
      st.u0 = p0;
      st.U = M;
      st.epi.mode = a.epi;
      pass_last<T, K, +1>(sm, st, tid);
    }
  }
};


// ---- Body: K' = K1*1024 with small K1 (2, 4, 8) in ONE kernel -------------------------------
// The K1-point transform over r1 is evaluated as a direct sum while the tile is filled, so the
// Z round trip of the two-kernel path disappears:
//   in[u][r2] = e^{2 pi i r2 u / N} * sum_{r1 < K1} B[r1*1024 + r2] * w_u^{k1},  w_u = e^{2 pi i u / U},
//   W[u + q2*U] = sum_{r2} in[u][r2] e^{2 pi i r2 q2 / 1024}
// (k1 = r1 - K1 [r >= rsplit] is the signed row of residue r; no alignment of the window needed).
template <typename T, int K1> struct DirectBody {
  static constexpr int NTB = TileCfg<T>::NT;   // threads per CTA of this kernel
  static constexpr int NT = NTB;
  using V = cx<T>;
  using Args = SingleArgs<T>;
  static constexpr int K = K2C;
  using LY = Lay<T, K>;
  static constexpr int NP = Plan<K>::NP;
  static constexpr int P = LY::P;
  static constexpr int NPHASE = 2 + NP;
  static constexpr int NW = 2 * K1 * P;   // w_u^{k1} for k1 = r1 and r1 - K1, per b
  static constexpr size_t SMEM = LY::TILE_BYTES + NW * sizeof(V);
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *smraw) {
    V *sm = (V *)smraw;
    V *wt = (V *)((char *)smraw + LY::TILE_BYTES);   // [b][2][K1]
    const ScaleDesc d = a.descs[a.first + by];
    const int U = (int)(a.N / K);
    const int u0 = bx * P;
    if constexpr (PH == 0) {
      for (int i = tid; i < NW; i += NT) {
        const int b = i / (2 * K1), s = (i / K1) & 1, r1 = i % K1;
        const int k1 = r1 - (s ? K1 : 0);
        wt[i] = nroot_t<T>(a.nt, (unsigned)k1 * (unsigned)(u0 + b) * (unsigned)K);
      }
    } else if constexpr (PH == 1) {
      const V *B = a.Bbuf + d.boff;
      // Positions r2 = tid + NT*it are handled IB at a time: the K1*IB band values stay in
      // registers while the K1 weights of each batch index b are read from shared memory once
      // (they depend on (b, r1) only, except on the single row r1s that the signed-bin split
      // cuts, where the sign is chosen per position).
      constexpr int NIT = K / NT;
      constexpr int IB = (8 / K1) < 1 ? 1 : ((8 / K1) < NIT ? (8 / K1) : NIT);
      const int r1s = d.rsplit / K, r2s = d.rsplit % K;   // residues >= rsplit are "negative"
      V e = nroot_t<T>(a.nt, (unsigned)tid * (unsigned)u0);    // e^{2 pi i r2 u0 / N}
      const V se = nroot_t<T>(a.nt, (unsigned)NT * (unsigned)u0);
      V dr = nroot_t<T>(a.nt, (unsigned)tid);                  // e^{2 pi i r2 / N}
      const V sdr = nroot_t<T>(a.nt, (unsigned)NT);
      if constexpr (K1 >= 8) {
        // many terms per position: one position at a time, weights straight from shared memory
        for (int it = 0; it < NIT; ++it) {
          const int r2 = tid + NT * it;
          V bv[K1];
          bool neg[K1];
#pragma unroll
          for (int r1 = 0; r1 < K1; ++r1) {
            bv[r1] = ldg(&B[r1 * K + r2]);
            neg[r1] = (r1 * K + r2) >= d.rsplit;
          }
          V t = e;
#pragma unroll
          for (int b = 0; b < P; ++b) {
            V acc = mk<T>(0, 0);
#pragma unroll
            for (int r1 = 0; r1 < K1; ++r1)
              acc = cadd(acc, cmul(bv[r1], wt[(b * 2 + (neg[r1] ? 1 : 0)) * K1 + r1]));
            sm[LY::phys(b, r2)] = cmul(acc, t);
            t = cmul(t, dr);
          }
          e = cmul(e, se);
          dr = cmul(dr, sdr);
        }
      } else
      for (int it0 = 0; it0 < NIT; it0 += IB) {
        V bv[IB][K1], t[IB], dd[IB];
#pragma unroll
        for (int q = 0; q < IB; ++q) {
          const int r2 = tid + NT * (it0 + q);
#pragma unroll
          for (int r1 = 0; r1 < K1; ++r1) bv[q][r1] = ldg(&B[r1 * K + r2]);
          t[q] = e;
          dd[q] = dr;
          e = cmul(e, se);
          dr = cmul(dr, sdr);
        }
#pragma unroll
        for (int b = 0; b < P; ++b) {
          V acc[IB];
#pragma unroll
          for (int q = 0; q < IB; ++q) acc[q] = mk<T>(0, 0);
#pragma unroll
          for (int r1 = 0; r1 < K1; ++r1) {
            if (r1 != r1s) {   // warp-uniform: one weight for the whole row
              const V w = wt[(b * 2 + (r1 > r1s ? 1 : 0)) * K1 + r1];
#pragma unroll
              for (int q = 0; q < IB; ++q) acc[q] = cadd(acc[q], cmul(bv[q][r1], w));
            } else {
              const V wp = wt[(b * 2 + 0) * K1 + r1], wn = wt[(b * 2 + 1) * K1 + r1];
#pragma unroll
              for (int q = 0; q < IB; ++q) {
                const bool neg = (tid + NT * (it0 + q)) >= r2s;
                acc[q] = cadd(acc[q], cmul(bv[q][r1], neg ? wn : wp));
              }
            }
          }
#pragma unroll
          for (int q = 0; q < IB; ++q) {
            sm[LY::phys(b, tid + NT * (it0 + q))] = cmul(acc[q], t[q]);
            t[q] = cmul(t[q], dd[q]);
          }
        }
      }
    } else if constexpr (PH == 2) {
      SmemLoader<T, K> ld;
      ld.sm = sm;
      tile_first<T, K, +1>(sm, a.tw, ld, tid);
    } else if constexpr (PH == 3 && NP == 3) {
      tile_second<T, K, +1>(sm, a.tw, tid);
    } else {
      OutStorer<T> st;
      st.row = a.W + (size_t)d.row * a.n0;
      st.nout = a.n0;
      st.u0 = u0;
      st.U = U;
      st.epi.mode = a.epi;
      pass_last<T, K, +1>(sm, st, tid);
    }
  }
};

// ---- Body: second kernel of the two-kernel path: K2 = 1024 or 512 over r2, rows of Z -------
template <typename T> struct PassBArgs {
  const cx<T> *Z;          // [ny][U][K2]
  cx<T> *out;              // [rows][pitch]
  const cx<T> *tw;
  const ScaleDesc *descs;  // may be null: output row = blockIdx.y + row0
  const double *grow;      // EPI_GAUSS: per-row coefficient g
  long long pitch, nout;
  double post;
  unsigned N;
  int first, row0;
  int epi;
  int zmod;                // Z slot of row `by` is by % zmod
  int pf_dist;             // L2 prefetch distance in tiles (0 = off)
  int ny;                  // gridDim.y of this launch (rows)
  int by0;                 // global index of this launch's first Z row (interleave bookkeeping)
  int ileave;              // > 1: Z row `by` is sub-transform by % ileave of output row by / ileave
                           // (final index n*ileave + by % ileave): three-level path, Np > 2^20
  int rev;                 // rows are processed last-to-first: the first kernel wrote the last rows
                           // of Z most recently, they are the ones still resident in L2
};

// K2 = 1024 leaves P = TILE/K2 = Q/2 transforms per tile (64-byte output runs, 2-way bank
// conflict on the last pass of the unskewed row layout); K2 = 512 has P = Q: 128-byte output
// runs, conflict-free.  The pruned (band) scales use 512, the dense ones need 1024 (K1 <= 1024).
template <typename T, int SIGN, int K2 = K2C> struct PassBBody {
  static constexpr int NTB = TileCfg<T>::NT;   // threads per CTA of this kernel
  static constexpr int NT = NTB;
  using V = cx<T>;
  using Args = PassBArgs<T>;
  static constexpr int K = K2;
  using LY = Lay<T, K, true>;   // rows are filled by bulk-async copies: no skew
  static constexpr int NP = Plan<K>::NP;
  // phase 0: one thread issues the bulk-async (TMA) copies of the tile's rows -- the rows
  // Z[u0 .. u0+P) are contiguous in global memory -- then the FFT passes run from shared memory
  static constexpr int NPHASE = NP + 1;
  static constexpr size_t SMEM = LY::TILE_BYTES + 16;
  // bulk-async copies need 16-byte aligned shared-memory destinations: every row start
  static constexpr bool ROWS_ALIGNED = (LY::PITCH * sizeof(V)) % 16 == 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *smraw) {
    static_assert(ROWS_ALIGNED, "PassB: tile rows must start on 16-byte boundaries");
    const int ey = by;                   // position in execution order
    if (a.rev) by = a.ny - 1 - ey;
    V *sm = (V *)smraw;
    const int U = (int)(a.N / K);
    const int u0 = bx * LY::P;
    TileBarrier tb;
    tb.bar = (unsigned long long *)((char *)smraw + LY::TILE_BYTES);
    if constexpr (PH == 0) {
      const int nvalid = (U - u0) < LY::P ? (U - u0) : LY::P;
      const V *src = a.Z + (size_t)(by % a.zmod) * a.N + (size_t)u0 * K;
      if constexpr (LY::CHUNKED) {
        // skewed rows (compile-time option CWTB_ROWS_SKEW): 16-element pieces issued by the
        // lanes of warp 0 after lane 0 has armed the barrier
        if (tid < 32) {
          if (tid == 0) tb.init_and_expect((unsigned)(nvalid * K * sizeof(V)));
          warp_sync();
          constexpr int NCH = K / 16;
          for (int i = tid; i < nvalid * NCH; i += 32) {
            const int b = i / NCH, ch = i % NCH;
            tb.copy(sm + LY::phys(b, 16 * ch), src + (size_t)b * K + 16 * ch, (unsigned)(16 * sizeof(V)));
          }
        }
      } else if (tid == 0) {
        // one thread arms the barrier and issues one bulk copy per row
        tb.init_and_expect((unsigned)(nvalid * K * sizeof(V)));
        for (int b = 0; b < nvalid; ++b)
          tb.copy(sm + LY::phys(b, 0), src + (size_t)b * K, (unsigned)(K * sizeof(V)));
      }
      // warm L2 with the tile a CTA `pf_dist` blocks ahead will load (same row of the grid,
      // or the next row when this one is exhausted): its TMA copies then hit L2
      if (tid == 0 && a.pf_dist > 0) {
        long long t = (long long)bx + a.pf_dist;
        int pe = ey;
        const int tiles = (U + LY::P - 1) / LY::P;
        while (t >= tiles && pe + 1 < a.ny) { t -= tiles; ++pe; }
        const int py = a.rev ? a.ny - 1 - pe : pe;
        if (t < tiles && t * LY::P + LY::P <= U)
          TileBarrier::prefetch_l2(a.Z + (size_t)(py % a.zmod) * a.N + (size_t)t * LY::P * K,
                                   (unsigned)(LY::P * K * sizeof(V)));
      }
      for (int b = nvalid; b < LY::P; ++b)
        for (int i = tid; i < K; i += NT) sm[LY::phys(b, i)] = mk<T>(0, 0);
    } else if constexpr (PH == 1) {
      tb.wait(0);
      SmemLoader<T, K, true> ld;
      ld.sm = sm;
      tile_first<T, K, SIGN, SmemLoader<T, K, true>, true>(sm, a.tw, ld, tid);
    } else if constexpr (PH == 2 && NP == 3) {
      tile_second<T, K, SIGN, true>(sm, a.tw, tid);
    } else {
      const int il = a.ileave > 1 ? a.ileave : 1;
      const int outer = (a.by0 + by) / il;
      const int row = a.descs ? a.descs[a.first + outer].row : a.row0 + outer;
      OutStorer<T> st;
      st.row = a.out + (size_t)row * a.pitch;
      st.nout = a.nout;
      st.u0 = u0;
      st.U = U;
      st.ostride = il;
      st.ooff = (a.by0 + by) % il;
      st.epi.mode = a.epi;
      if (a.epi == EPI_GAUSS) {
        st.epi.g = a.grow[row];
        st.epi.invn = 1.0 / ((double)a.N * il);
        st.epi.post = a.post;
        st.epi.nfreq = (long long)a.N * il;
      }
      pass_last<T, K, SIGN, OutStorer<T>, true>(sm, st, tid);
      if (tid == 0) tb.inval();   // every thread passed wait() two barriers ago
    }
  }
};

// ---- Body: first kernel of the two-kernel path: K1-point transforms over r1 --------
// (Measured and dropped, profiles/r2/sweep_k.txt: band scales that evaluate x^ * conj(psi^) * norm while the
// tile is filled instead of reading the band buffer -- the first kernel of Np/K' = 2 scales got 55 % slower,
// more than the band-product launch it saves: config 5 7.83 -> 7.92 ms, config 3 Paul 0.283 -> 0.321 ms.)
enum { MODE_DENSE = 0, MODE_BAND = 1, MODE_REAL = 2, MODE_CPLX = 3 };

template <typename T> struct PassAArgs {
  const ScaleDesc *descs;
  const cx<T> *spec;   // x^ (MODE_DENSE)
  const cx<T> *Bbuf;   // band products (MODE_BAND)
  const void *in;      // T* (MODE_REAL) or cx<T>* (MODE_CPLX), rows of `in_pitch`
  cx<T> *Z;            // [ny][U][K2]
  const cx<T> *tw;
  Fam fam;
  NTab nt;
  long long in_pitch, n_in;
  unsigned N;
  int first, row0;
  int zmod;            // Z slot of row `by` is by % zmod (ring of Z buffers in the fused kernel)
  int pf_dist;         // L2 prefetch distance in tiles for the band-product rows (0 = off)
  int gauss_rec;       // dense Morlet: evaluate the Gaussian by recurrence along each thread's bins
  unsigned K2;         // row length of Z: 1024 (second kernel = PassB) or 2^20 (pre-pass of the
                       // three-level path for Np > 2^20, where the rows are transformed again)
};

template <typename T, int K1, int MODE, int SIGN> struct PassABody {
  static constexpr int NTB = TileCfg<T>::NT;   // threads per CTA of this kernel
  static constexpr int NT = NTB;
  using V = cx<T>;
  using Args = PassAArgs<T>;
  using LY = Lay<T, K1>;
  static constexpr int NP = Plan<K1>::NP;
  static constexpr int P = LY::P;
  static constexpr int T2 = P < K2C ? P : K2C;  // r2 values per tile (a.K2 is a multiple of it)
  static constexpr int NPHASE = NP == 1 ? 1 : NP + 1;
  static constexpr size_t SMEM = LY::BYTES;

  struct Src {
    const Args &a;
    ScaleDesc d;
    int by, p;
    V twist0;
    HD Src(const Args &a_, int by_, int p_) : a(a_), by(by_), p(p_) {
      if (MODE == MODE_DENSE || MODE == MODE_BAND) d = a.descs[a.first + by];
    }
    // element r = pos*K2 + r2 of the K'-point input
    HD V get(int pos, int r2) const {
      const unsigned r = (unsigned)pos * a.K2 + (unsigned)r2;
      if (MODE == MODE_DENSE) {
        const int k = (int)r - (r >= a.N / 2 ? (int)a.N : 0);
        // outside the scale's band the response is below the pruning threshold: same rule as
        // the pruned classes (their band product is exactly zero there); skips the exp
        if (a.fam.family != 3 && (k < d.k_lo || k > d.k_hi)) return mk<T>(0, 0);
        return band_value<T>(a.fam, d, a.spec, r, k, a.N);
      } else if (MODE == MODE_BAND) {
        V v = ldg(&a.Bbuf[d.boff + r]);
        if (p == 0 || NP > 1) return v;   // multi-pass plans apply the twist in pass 1
        const int k1 = pos - ((int)r >= d.rsplit ? K1 : 0);
        // e^{2 pi i k1 p / (K1 M)} = e^{2 pi i (k1 p K2) / N}
        V w = nroot_t<T>(a.nt, (unsigned)k1 * (unsigned)p * a.K2);
        return cmul(v, w);
      } else if (MODE == MODE_REAL) {
        const T *row = (const T *)a.in + (size_t)(a.row0 + by) * a.in_pitch;
        return mk<T>((long long)r < a.n_in ? ldg(&row[r]) : (T)0, (T)0);
      } else {
        const V *row = (const V *)a.in + (size_t)(a.row0 + by) * a.in_pitch;
        return (long long)r < a.n_in ? ldg(&row[r]) : mk<T>(0, 0);
      }
    }
  };

  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *smraw) {
    V *sm = (V *)smraw;
    const int NTILE2 = (int)(a.K2 / T2);
    const int p = bx / NTILE2;
    const int r20 = (bx % NTILE2) * T2;
    const int M = (int)(a.N / ((unsigned)K1 * a.K2));
    ZStorer<T, SIGN> st;
    st.Z = a.Z + (size_t)(by % a.zmod) * a.N;
    st.nt = a.nt;
    st.p = p;
    st.M = M;
    st.r20 = r20;
    st.bmax = T2;
    st.K2 = a.K2;
    if constexpr (NP == 1) {
      Src src(a, by, p);
      for (int b = tid; b < T2; b += NT) {
        V x[K1];
#pragma unroll
        for (int i = 0; i < K1; ++i) x[i] = src.get(i, r20 + b);
        dftR<K1, SIGN, T>(x);
        st.store(b, 0, 1, x);
      }
    } else if constexpr (PH == 0) {
      Src src(a, by, p);
      // warm L2 with the band-product rows of the tile `pf_dist` blocks ahead (same scale)
      if (MODE == MODE_BAND && a.pf_dist > 0 && T2 * sizeof(V) >= 256) {
        const int tiles = M * NTILE2;
        const int t = bx + a.pf_dist;
        if (t < tiles) {
          const int r20n = (t % NTILE2) * T2;
          const V *base = a.Bbuf + src.d.boff + r20n;
          for (int pos = tid; pos < K1; pos += NT)
            TileBarrier::prefetch_l2(base + (size_t)pos * a.K2, (unsigned)(T2 * sizeof(V)));
        }
      }
      // the same for the rows of a batched row transform (coherence smoothing, coarse transforms): the
      // tile `pf_dist` blocks ahead of this one in the same row
      if (MODE == MODE_CPLX && a.pf_dist > 0 && T2 * sizeof(V) >= 256) {
        const int t = bx + a.pf_dist;
        if (t < M * NTILE2) {
          const V *row = (const V *)a.in + (size_t)(a.row0 + by) * a.in_pitch + (t % NTILE2) * T2;
          for (int pos = tid; pos < K1; pos += NT)
            if ((long long)pos * a.K2 + (t % NTILE2) * T2 + T2 <= a.n_in)
              TileBarrier::prefetch_l2(row + (size_t)pos * a.K2, (unsigned)(T2 * sizeof(V)));
        }
      }
      if (MODE == MODE_DENSE && a.fam.family == 0 && a.gauss_rec && T2 <= NT) {
        // Morlet, dense scale: a thread's bins are k0, k0 + D, k0 + 2D, ... (D = (NT/T2)*K2), so
        //   g(k + D) = g(k) * rho(k),  rho(k + D) = rho(k) * exp(-a^2),  a = s * w_D,
        // replaces the exp per bin by two multiplies.  Re-seeded with exact exp() when the
        // band is entered, at the signed-bin wrap and every 16 steps (error <= ~1e-14 relative).
        constexpr int DPOS = NT / T2;
        const ScaleDesc &d = src.d;
        const int b = tid % T2;
        const long long D = (long long)DPOS * a.K2;
        const double wd = 6.283185307179586 * ((double)D * a.fam.dw);
        const double aa = d.s * wd;
        const double q = exp(-aa * aa);
        double g = 0, rho = 0;
        long long kprev = 0;
        int since = 1 << 30;
        // Batches of UB bins: the spectrum loads of a batch are issued together (independent of the
        // recurrence), then the Gaussian values follow one another.  One load per iteration, as the
        // plain loop compiles, leaves every thread waiting a full L2 round trip 32 times per tile.
        constexpr int UB = CWTB_PASSA_BATCH;
        const V *sp = a.spec + (size_t)d.chan * a.N + (unsigned)(r20 + b);
        for (int pos0 = tid / T2; pos0 < K1; pos0 += DPOS * UB) {
          V raw[UB];
          int kk[UB];
#pragma unroll
          for (int u = 0; u < UB; ++u) {
            const int pos = pos0 + u * DPOS;
            const unsigned r = (unsigned)pos * a.K2 + (unsigned)(r20 + b);
            const int k = (int)r - (r >= a.N / 2 ? (int)a.N : 0);
            const bool in = pos < K1 && k >= d.k_lo && k <= d.k_hi;
            kk[u] = in ? k : (int)0x7fffffff;
            raw[u] = in ? ldg(&sp[(size_t)pos * a.K2]) : mk<T>(0, 0);
          }
#pragma unroll
          for (int u = 0; u < UB; ++u) {
            const int pos = pos0 + u * DPOS;
            if (pos >= K1) break;
            V v = mk<T>(0, 0);
            if (kk[u] != (int)0x7fffffff) {
              const int k = kk[u];
              // (a value in the subnormal range has lost its relative precision: with band_eps = 0 the
              // band reaches bins where exp() is below 1e-308, and the recurrence would carry that
              // error up to the peak -- re-seed until the value is a normal number again)
              if (since >= 16 || (long long)k != kprev + D || g < 1e-290) {
                const double f = d.s * (6.283185307179586 * ((double)k * a.fam.dw));
                const double dd = f - a.fam.f0;
                g = exp(-0.5 * dd * dd);
                rho = exp(-aa * dd - 0.5 * aa * aa);
                since = 0;
              } else {
                g *= rho;
                rho *= q;
                ++since;
              }
              kprev = k;
              v = cscale(raw[u], (T)(g * d.amp));
            } else {
              since = 1 << 30;
            }
            sm[LY::phys(b, pos)] = v;
          }
        }
      } else if (CWTB_PASSA_ASYNC && MODE == MODE_BAND) {
        // band products are copied as they are (multi-pass plans apply the twist in pass 1):
        // asynchronous copies, the thread's 32 elements in flight together
        const V *base = a.Bbuf + src.d.boff + r20;
        for (int idx = tid; idx < K1 * T2; idx += NT) {
          const int b = idx % T2, pos = idx / T2;
          cp_async(&sm[LY::phys(b, pos)], base + (size_t)pos * a.K2 + b);
        }
        cp_async_wait();
      } else if (CWTB_PASSA_ASYNC && MODE == MODE_CPLX) {
        const V *row = (const V *)a.in + (size_t)(a.row0 + by) * a.in_pitch;
        for (int idx = tid; idx < K1 * T2; idx += NT) {
          const int b = idx % T2, pos = idx / T2;
          const unsigned r = (unsigned)pos * a.K2 + (unsigned)(r20 + b);
          if ((long long)r < a.n_in) cp_async(&sm[LY::phys(b, pos)], row + r);
          else sm[LY::phys(b, pos)] = mk<T>(0, 0);
        }
        cp_async_wait();
      } else {
        // (the compiler batches four loads per round trip on its own; eight in flight measured ...)
        CWTB_PRAGMA_UNROLL_A
        for (int idx = tid; idx < K1 * T2; idx += NT) {
          const int b = idx % T2, pos = idx / T2;
          sm[LY::phys(b, pos)] = src.get(pos, r20 + b);
        }
      }
    } else if constexpr (PH == 1) {
      if (MODE == MODE_BAND && p != 0) {
        SmemTwistLoader<T, K1, Plan<K1>::R1> ld;
        ld.sm = sm;
        ld.nt = a.nt;
        ld.rsplit_row = a.descs[a.first + by].rsplit / (int)a.K2;
        ld.pk2 = (unsigned)p * a.K2;
        tile_first<T, K1, SIGN>(sm, a.tw, ld, tid);
      } else {
        SmemLoader<T, K1> ld;
        ld.sm = sm;
        tile_first<T, K1, SIGN>(sm, a.tw, ld, tid);
      }
    } else if constexpr (PH == 2 && NP == 3) {
      tile_second<T, K1, SIGN>(sm, a.tw, tid);
    } else {
      pass_last<T, K1, SIGN>(sm, st, tid);
    }
  }
};

// ==================================================================================================
// Band-limited expansion path.  A scale whose response is confined to the bins [k_lo, k_hi]
// (Kb of the Np bins) is a trigonometric polynomial of Kb terms: it is fully determined by
// Nc >= 2 Kb samples.  Instead of running Np/K' pruned transforms of K' points each, the engine
//   (1) forms the band product shifted to the centre bin kc and divided by the transform of the
//       interpolation kernel (ExpandBandBody),
//   (2) inverse-transforms it on the coarse grid of Nc points (the ordinary batched FFT), and
//   (3) expands the Nc samples to the Np output points with a polyphase Kaiser-Bessel kernel of
//       `taps` real weights per output and re-modulates by e^{2 pi i kc n / Np} (ExpandBody):
//         W[R m + rho] = e^{2 pi i kc n/Np} * sum_t c[m + t - (taps/2 - 1)] * h[t][rho],  R = Np / Nc.
// With phi the kernel and phi^ its transform, sum_m e^{2 pi i k m/Nc} phi(x - m) =
// sum_l phi^(k/Nc + l) e^{2 pi i (k/Nc + l) x}: the l = 0 term is the exact value after the division
// by phi^(k/Nc), the others are the aliasing error, bounded on the host by
// max_{|xi| <= xi_max} sum_{l != 0} |phi^(xi + l)| / |phi^(xi)| (engine.cu: kb_alias_bound).  The host
// picks (Nc, taps) so that the bound stays below the context's expansion tolerance (default
// 5e-13: measured error 1e-13, three orders inside the 1e-10 parity gate; 0 = path off).
// Cost per output point: 2*taps + 8 fp64 FMAs, one 16-byte shared-memory read, one 16-byte store --
// a streaming kernel bounded by the W store, with no intermediate in global memory.
// ==================================================================================================
template <typename T> struct ExpandBandArgs {
  const ScaleDesc *descs;
  const cx<T> *spec;
  cx<T> *Cin;       // coarse spectra, rows at descs[].ip_coff
  Fam fam;
  unsigned N;
  int first;
};
template <typename T> struct ExpandBandBody {
  using V = cx<T>;
  using Args = ExpandBandArgs<T>;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  static constexpr int PER = 4;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const ScaleDesc d = a.descs[a.first + by];
    const int Nc = 1 << d.ip_log2Nc;
    const double pw = 3.14159265358979323846 * (double)d.ip_w;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int r = (bx * PER + i) * NT + tid;
      if (r >= Nc) return;
      const int kp = r < Nc / 2 ? r : r - Nc;       // signed offset from the centre bin
      const int k = d.ip_kc + kp;
      V v = mk<T>(0, 0);
      if (k >= d.k_lo && k <= d.k_hi) {
        const V b = band_value<T>(a.fam, d, a.spec, (unsigned)k & (a.N - 1), k, a.N);
        // 1 / phi^(kp / Nc),  phi^(xi) = taps / I0(beta) * sinh(z) / z,  z = sqrt(beta^2 - (pi taps xi)^2)
        const double x = pw * ((double)kp / (double)Nc);
        const double z = sqrt(d.ip_beta * d.ip_beta - x * x);      // > 0: |xi| <= 1/4 < 1 - xi_max
        const double f = d.ip_dc * (z / sinh(z));
        v = mk<T>((T)((double)b.x * f), (T)((double)b.y * f));
      }
      a.Cin[d.ip_coff + r] = v;
    }
  }
};

template <typename T> struct ExpandArgs {
  const ScaleDesc *descs;
  const cx<T> *C;      // coarse samples (inverse transforms of the coarse spectra)
  const double *wt;    // weight tables [taps][R] (fp64 for both engines)
  cx<T> *W;            // [rows][n0]
  NTab nt;
  long long n0;
  unsigned N;
  int first;
  int epi;             // EPI_STORE / EPI_MULCONJ
  int log2N;           // R = N / Nc = 1 << (log2N - ip_log2Nc) per row: one launch serves every
                       // coarse length (each row has N / (NT * 32) tiles whatever its R)
};

// CTA tile: RB = min(R, NT) consecutive phases rho  x  NRUN = NT / RB runs of L = 32 consecutive
// coarse positions m.  A thread keeps its `TAPS` weights (fixed rho) and a sliding window of TAPS
// coarse samples in registers and walks its run (fully unrolled: window slots are compile-time
// registers): one new sample (shared-memory read, the same address for the lanes of a run) and one
// 16-byte store per output; lanes run over rho, so a warp stores min(R, 32) consecutive points
// per run.  Measured on B200 (profiles/r2): the kernel is bound by the fp64 pipe (2 taps + ~12
// other fp64 instructions per point at 64 lanes per SM and clock); 8 accumulator chains and 4 CTAs
// per SM keep that pipe 63 % busy, longer runs or fewer chains were slower.
template <typename T, int TAPS, int EPI = EPI_STORE> struct ExpandBody {
  static constexpr int NTB = TileCfg<T>::NT;
  static constexpr int NT = NTB;
  static constexpr int MINB = sizeof(T) == 8 ? 4 : 2;   // CTAs per SM the register budget is capped for
  using V = cx<T>;
  using Args = ExpandArgs<T>;
  static constexpr int L = 32;                       // coarse positions per run
  static constexpr int MINR = 4;                     // smallest expansion factor R = Np / Nc
  static constexpr int MAXRUN = NT / MINR;
  static constexpr int STAGE = MAXRUN * L + TAPS;    // staged coarse samples (incl. halo)
  HD static int skew(int i) { return i + (i >> 5); } // runs start 33 elements apart: no bank conflict
  static constexpr int NPHASE = 2;
  static constexpr size_t SMEM = (size_t)(STAGE + STAGE / 32 + 2) * sizeof(V);
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *smraw) {
    V *sm = (V *)smraw;
    const ScaleDesc &d = a.descs[a.first + by];
    const int log2R = a.log2N - d.ip_log2Nc;
    const int R = 1 << log2R;
    const int Nc = 1 << d.ip_log2Nc;
    const int RB = R < NT ? R : NT;
    const int NRUN = NT / RB;
    const int MT = NRUN * L;                         // coarse positions per CTA
    const int mtiles = (Nc + MT - 1) / MT;
    const int mt = bx % mtiles, rb = bx / mtiles;
    if (rb * RB >= R) return;                        // short coarse grid: fewer tiles than the launch has
    const int m0 = mt * MT;
    if constexpr (PH == 0) {
      const V *c = a.C + d.ip_coff;
      for (int i = tid; i < MT + TAPS; i += NT) {
        const int m = (m0 - (TAPS / 2 - 1) + i) & (Nc - 1);     // periodic on the coarse grid
        sm[skew(i)] = ldg(&c[m]);
      }
    } else {
      const int rl = tid & (RB - 1), j = tid / RB;
      const int rho = rb * RB + rl;
      const int ms = m0 + j * L;                     // first coarse position of this thread's run
      // outputs n = R m + rho for m = ms .. ms + L - 1; kept while m < Nc and n < n0
      const long long nfirst = ((long long)ms << log2R) + rho;
      long long keep = (a.n0 - nfirst + R - 1) >> log2R;      // steps with n < n0
      if (keep > Nc - ms) keep = Nc - ms;
      const int smax = keep < 0 ? 0 : (keep > L ? L : (int)keep);
      if (smax == 0) return;
      T hw[TAPS];
      const double *wt = a.wt + d.ip_woff + rho;
#pragma unroll
      for (int t = 0; t < TAPS; ++t) hw[t] = (T)ldg(&wt[(size_t)t * R]);
      const V *run = sm + 33 * j;                    // skew(j*L + i) = 33 j + i + (i >> 5), i < L + TAPS
      V win[TAPS];
#pragma unroll
      for (int t = 0; t < TAPS - 1; ++t) win[t] = run[t + (t >> 5)];
      // re-modulation e^{2 pi i kc n / Np}: table value (fp64 roots) every RESEED steps, recurrence
      // (step e^{2 pi i kc R / Np}) in between, in the engine's arithmetic: fp64 drifts 1e-16 per
      // step (16 steps), fp32 6e-8 per step (8 steps: 5e-7 of the 1e-5 budget)
      constexpr int RESEED = sizeof(T) == 8 ? 16 : 8;
      const unsigned kc = (unsigned)d.ip_kc;
      const unsigned nlo = (unsigned)nfirst;
      const V stepw = nroot_t<T>(a.nt, kc << log2R);
      V tw = mk<T>(1, 0);
      V *p = a.W + (size_t)d.row * a.n0 + nfirst;
#pragma unroll
      for (int s = 0; s < L; ++s) {
        win[(s + TAPS - 1) % TAPS] = run[(s + TAPS - 1) + ((s + TAPS - 1) >> 5)];
        if (s % RESEED == 0) tw = nroot_t<T>(a.nt, kc * (nlo + ((unsigned)s << log2R)));
        // 8 independent chains (4 per component): the fp64 pipe needs that much parallelism per warp;
        // the fp32 kernel is bound by instruction issue (ncu: 70 % issue slots busy, 49 instructions per
        // point for 24 useful ones) and runs two chains per component
        constexpr int NCH = sizeof(T) == 8 ? 4 : 2;
        T ar[4] = {0, 0, 0, 0}, ai[4] = {0, 0, 0, 0};
#pragma unroll
        for (int t = 0; t < TAPS; ++t) {
          const V cv = win[(s + t) % TAPS];
          ar[t & (NCH - 1)] += cv.x * hw[t];
          ai[t & (NCH - 1)] += cv.y * hw[t];
        }
        const V acc = NCH == 4 ? mk<T>((ar[0] + ar[1]) + (ar[2] + ar[3]), (ai[0] + ai[1]) + (ai[2] + ai[3]))
                               : mk<T>(ar[0] + ar[1], ai[0] + ai[1]);
        const V x = cmul(acc, tw);
        tw = cmul(tw, stepw);
        if (s < smax) {
          if (EPI == EPI_MULCONJ) *p = cmul(*p, cconj(x));
          else st_stream(p, x);
        }
        p += R;
      }
    }
  }
};

#ifndef CWTB_HOST_EMU
// ---- the fp64 expansion with the tap sums on the tensor cores ---------------------------------------
// The tap sum  acc[m][rho] = sum_t c[m + t - (taps/2 - 1)] * h[t][rho]  is a Toeplitz product: for 8
// consecutive coarse positions m and 8 consecutive phases rho it is an (8 x taps) x (taps x 8) real
// matrix product per component, i.e. taps/4 `mma.sync.m8n8k4.f64` (SASS DMMA.8x8x4) for the real and
// as many for the imaginary part.  DMMA shares the fp64 pipe with DFMA on B200 (profiles/r2/
// dmma_vs_dfma.txt: times add) but moves 20 % more FMAs through it, and the accumulation happens
// inside the instruction: the scalar kernel's 2 x taps DFMA + 6 DADD per point (of ~38 fp64
// instructions, the pipe that bounds it) become taps/2 DMMA per 64 points.
//   A fragment (8 x 4, row m, column t):  lane holds c[m0 + lane/4 + 4 ks + lane%4]   (shared memory)
//   B fragment (4 x 8, row t, column rho): lane holds h[4 ks + lane%4][rho0 + lane/4] (registers)
//   C fragment (8 x 8): lane holds acc[m0 + lane/4][rho0 + 2 (lane%4) + {0, 1}]: two adjacent outputs,
//                       stored as one 32-byte access when the row is 32-byte aligned.
// A warp owns 8 phases and a run of L coarse positions; a CTA (4 warps) covers min(R, 32) phases
// x 4 L / (min(R, 32) / 8) coarse positions = 32 L outputs.  Tap counts 10 and 14 are padded to 12 / 16
// with zero weights.  Not part of the host-emulation build (warp-collective instruction): the
// emulated tests run the scalar ExpandBody, which stays the fp32 engine's kernel and the fallback.
// (An fp32 counterpart on 3xTF32 -- x = x_hi + x_lo, three mma.sync.m16n8k8.tf32 per component and eight
// taps -- gives the same 5e-7 parity but runs SLOWER than the scalar fp32 kernel, 3.54 vs 2.74 ms on
// config 5: the legacy HMMA path of sm_100a issues ~15 cycles per MMA and SM here, no faster than FFMA.
// Measured and dropped: profiles/r2/sweep_x_tf32x3_expansion_dropped.txt.)
__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
template <int TAPS, int EPI = EPI_STORE> struct ExpandMmaBody {
  static constexpr int NTB = 128;
  static constexpr int NT = NTB;
  static constexpr int MINB = 4;
  using V = double2;
  using Args = ExpandArgs<double>;
#ifndef CWTB_MMA_L
#define CWTB_MMA_L 128
#endif
  static constexpr int L = CWTB_MMA_L;              // coarse positions per warp run (8 L outputs per warp)
  static constexpr int KS = (TAPS + 3) / 4;         // k-steps of four taps
  static constexpr int KS4 = (TAPS + 4) / 4;        // R = 4: one more tap column (see body<.., true>)
  static constexpr int OUT_PER_CTA = 32 * L;
  static constexpr int STAGE = 8 * L + 4 * KS4;     // staged coarse samples incl. halo (R = 4: 4 runs of 2 L)
  static constexpr int NPHASE = 2;
  static constexpr size_t SMEM = (size_t)STAGE * sizeof(V);
  template <int PH> __device__ static void phase(const Args &a, int bx, int by, int tid, void *smraw) {
    const ScaleDesc &d = a.descs[a.first + by];
    if (a.log2N - d.ip_log2Nc == 2) body<PH, true>(a, d, bx, tid, (V *)smraw);
    else body<PH, false>(a, d, bx, tid, (V *)smraw);
  }
  // R4 = false (R >= 8): MMA rows = 8 consecutive coarse positions, columns = 8 consecutive phases.
  // R4 = true  (R == 4): the 8 columns are 2 coarse positions x 4 phases, the rows step by two coarse
  //   positions: acc[m0 + 2 i + dm][rho] = sum_t' c[m0 + 2 i + t' - (taps/2 - 1)] * h[t' - dm][rho],
  //   t' < taps + 1 (B holds the weights shifted by dm, zero outside).  A warp then covers 16 coarse
  //   positions per MMA block and runs over 2 L of them: the same 8 L outputs per warp.
  template <int PH, bool R4>
  __device__ static void body(const Args &a, const ScaleDesc &d, int bx, int tid, V *sm) {
    constexpr int KSr = R4 ? KS4 : KS;
    constexpr int Lr = R4 ? 2 * L : L;              // coarse positions per warp run
    constexpr int MB = R4 ? 16 : 8;                 // coarse positions per MMA block
    const int log2R = a.log2N - d.ip_log2Nc;
    const int R = 1 << log2R;
    const int Nc = 1 << d.ip_log2Nc;
    const int wpb = R4 ? 1 : ((R < 32 ? R : 32) >> 3);   // warps side by side in rho: 1, 2 or 4
    const int nrun = 4 / wpb;                       // runs per CTA
    const int MT = nrun * Lr;
    const int mtiles = (Nc + MT - 1) / MT;
    const int mt = bx % mtiles, rb = bx / mtiles;
    if (rb * 32 >= R && rb > 0) return;             // short rows use the first tiles of the launch only
    const int m0 = mt * MT;
    if constexpr (PH == 0) {
      const V *c = a.C + d.ip_coff;
      for (int i = tid; i < MT + 4 * KSr; i += NT) sm[i] = ldg(&c[(m0 - (TAPS / 2 - 1) + i) & (Nc - 1)]);
    } else {
      const int wid = tid >> 5, lane = tid & 31;
      const int g = lane >> 2, q = lane & 3;
      const int pb = wid % wpb, j = wid / wpb;
      const int rho0 = R4 ? 0 : rb * 32 + pb * 8;
      const int ms = m0 + j * Lr;
      double bf[KSr];
#pragma unroll
      for (int ks = 0; ks < KSr; ++ks) {
        const int t = 4 * ks + q - (R4 ? (g >> 2) : 0);
        const int rho = R4 ? (g & 3) : rho0 + g;
        bf[ks] = (t >= 0 && t < TAPS) ? ldg(&a.wt[d.ip_woff + (size_t)t * R + rho]) : 0.0;
      }
      // re-modulation e^{2 pi i kc n / Np} of this lane's two outputs: table values for the first
      // block, then steps of e^{2 pi i kc 64 / Np ... } = one MMA block of coarse positions further
      const unsigned kc = (unsigned)d.ip_kc;
      const int mlane = R4 ? 2 * g + (q >> 1) : g;              // coarse position of this lane inside a block
      const int rlane = R4 ? 2 * (q & 1) : rho0 + 2 * q;        // first of its two adjacent phases
      const unsigned n00 = ((unsigned)(ms + mlane) << log2R) + (unsigned)rlane;
      V tw0 = nroot(a.nt, kc * n00);
      V tw1 = cmul(tw0, nroot(a.nt, kc));
      const V stepb = nroot(a.nt, (kc * (unsigned)MB) << log2R);
      const V *run = sm + j * Lr + (R4 ? 2 * g : g) + q;
      V *rowp = a.W + (size_t)d.row * a.n0;
      const bool wide = (((size_t)d.row * (size_t)a.n0) & 1) == 0;   // 32-byte aligned pairs
#pragma unroll 4
      for (int mb = 0; mb < Lr / MB; ++mb) {
        if (ms + MB * mb >= Nc) break;                // warp-uniform: short coarse grids end inside the run
        double cr0 = 0, cr1 = 0, ci0 = 0, ci1 = 0;
#pragma unroll
        for (int ks = 0; ks < KSr; ++ks) {
          const V s = run[MB * mb + 4 * ks];
          dmma884(cr0, cr1, s.x, bf[ks]);
          dmma884(ci0, ci1, s.y, bf[ks]);
        }
        const int m = ms + MB * mb + mlane;
        const long long n = ((long long)m << log2R) + rlane;
        V x0 = cmul(make_double2(cr0, ci0), tw0);
        V x1 = cmul(make_double2(cr1, ci1), tw1);
        tw0 = cmul(tw0, stepb);
        tw1 = cmul(tw1, stepb);
        if (m < Nc && n < a.n0) {
          V *p = rowp + n;
          const bool two = n + 1 < a.n0;
          if (EPI == EPI_MULCONJ) {
            x0 = cmul(p[0], cconj(x0));
            if (two) x1 = cmul(p[1], cconj(x1));
            p[0] = x0;
            if (two) p[1] = x1;
          } else if (wide && two) {
            asm volatile("st.global.cs.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(x0.x), "d"(x0.y), "d"(x1.x), "d"(x1.y)
                         : "memory");
          } else {
            st_stream(p, x0);
            if (two) st_stream(p + 1, x1);
          }
        }
      }
    }
  }
};
#endif

// ---- Body: band product B[r] = x^[k] * conj(psi_ft) * norm / Np for pruned scales ------
template <typename T> struct BandArgs {
  const ScaleDesc *descs;
  const cx<T> *spec;
  cx<T> *Bbuf;
  Fam fam;
  unsigned N;
  int first;
};
template <typename T> struct BandBody {
  using V = cx<T>;
  using Args = BandArgs<T>;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  static constexpr int PER = 4;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const ScaleDesc d = a.descs[a.first + by];
    const int K = 1 << d.log2K;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int r = (bx * PER + i) * NT + tid;
      if (r >= K) return;
      const int k = r - (r >= d.rsplit ? K : 0);
      V v = mk<T>(0, 0);
      if (k >= d.k_lo && k <= d.k_hi) v = band_value<T>(a.fam, d, a.spec, (unsigned)k & (a.N - 1), k, a.N);
      a.Bbuf[d.boff + r] = v;
    }
  }
};

// ---- Body: batched K-point FFT over matrix rows (N <= 1024): forward FFT of short
// signals, the c2c test hook, the Gaussian smoothing transforms ----------------------
template <typename T> struct RowsArgs {
  const void *in;      // T* if real_in else cx<T>*
  cx<T> *out;
  const cx<T> *tw;
  const double *grow;  // EPI_GAUSS: per-row coefficient (null: plain store)
  long long in_pitch, out_pitch, n_in, nout;
  double post;
  int nrows, real_in, n;
};

template <typename T, int K> struct RowsLoader {
  using V = cx<T>;
  const RowsArgs<T> *a;
  int row0;
  int base, stride;
  HD void begin(int base_, int stride_, int, int) { base = base_; stride = stride_; }
  HD V get(int b, int pos) const {
    const int row = row0 + b;
    if (row >= a->nrows || pos >= a->n_in) return mk<T>(0, 0);
    if (a->real_in) return mk<T>(ldg((const T *)a->in + (size_t)row * a->in_pitch + pos), (T)0);
    return ldg((const V *)a->in + (size_t)row * a->in_pitch + pos);
  }
  template <int R> HD void load(int b, V (&x)[R]) const {
#pragma unroll
    for (int i = 0; i < R; ++i) x[i] = get(b, base + i * stride);
  }
};
template <typename T> struct RowsStorer {
  using V = cx<T>;
  const RowsArgs<T> *a;
  int row0;
  template <int R> HD void store(int b, int ql, int qs, V (&x)[R]) const {
    const int row = row0 + b;
    if (row >= a->nrows) return;
#pragma unroll
    for (int c = 0; c < R; ++c) {
      const int q = ql + c * qs;
      if (q >= a->nout) continue;
      V v = x[c];
      if (a->grow) {
        Epilogue<T> e;
        e.mode = EPI_GAUSS; e.g = a->grow[row]; e.invn = 1.0 / (double)a->n; e.post = a->post; e.nfreq = a->n;
        v = e.apply(v, v, q);
      }
      a->out[(size_t)row * a->out_pitch + q] = v;
    }
  }
};
template <typename T, int K, int SIGN> struct RowsBody {
  static constexpr int NTB = TileCfg<T>::NT;   // threads per CTA of this kernel
  static constexpr int NT = NTB;
  using V = cx<T>;
  using Args = RowsArgs<T>;
  using LY = Lay<T, K>;
  static constexpr int NP = Plan<K>::NP;
  static constexpr int NPHASE = NP;
  static constexpr size_t SMEM = LY::BYTES;
  template <int PH> HD static void phase(const Args &a, int bx, int, int tid, void *smraw) {
    V *sm = (V *)smraw;
    const int row0 = bx * LY::P;
    RowsStorer<T> st;
    st.a = &a;
    st.row0 = row0;
    RowsLoader<T, K> ld;
    ld.a = &a;
    ld.row0 = row0;
    if constexpr (NP == 1) {
      for (int b = tid; b < LY::P; b += NT) {
        V x[K];
#pragma unroll
        for (int i = 0; i < K; ++i) x[i] = ld.get(b, i);
        dftR<K, SIGN, T>(x);
        st.store(b, 0, 1, x);
      }
    } else if constexpr (PH == 0) {
      tile_first<T, K, SIGN>(sm, a.tw, ld, tid);
    } else if constexpr (PH == 1 && NP == 3) {
      tile_second<T, K, SIGN>(sm, a.tw, tid);
    } else {
      pass_last<T, K, SIGN>(sm, st, tid);
    }
  }
};

// ---- Body: direct O(N^2) transform for tiny padded lengths (Np < 32) ---------------
template <typename T> struct TinyArgs {
  const ScaleDesc *descs;
  const cx<T> *spec;
  cx<T> *W;
  Fam fam;
  long long n0;
  unsigned N;
  int first;
  int epi;
};
template <typename T> struct TinyBody {
  using V = cx<T>;
  using Args = TinyArgs<T>;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const ScaleDesc d = a.descs[a.first + by];
    const int n = bx * NT + tid;
    if (n >= a.n0) return;
    double sr = 0, si = 0;
    for (unsigned r = 0; r < a.N; ++r) {
      const int k = (int)r - (r >= a.N / 2 && a.N > 1 ? (int)a.N : 0);
      V v = band_value<T>(a.fam, d, a.spec, r, k, a.N);
      double sn, cs;
      sincospi_hd(2.0 * (double)((r * (unsigned)n) % a.N) / (double)a.N, &sn, &cs);
      sr += (double)v.x * cs - (double)v.y * sn;
      si += (double)v.x * sn + (double)v.y * cs;
    }
    V *dst = &a.W[(size_t)d.row * a.n0 + n];
    V val = mk<T>((T)sr, (T)si);
    *dst = a.epi == EPI_MULCONJ ? cmul(*dst, cconj(val)) : val;
  }
};
// forward DFT of a tiny real signal
template <typename T> struct TinyFwdArgs {
  const T *sig;
  cx<T> *spec;
  long long n0;
  unsigned N;
};
template <typename T> struct TinyFwdBody {
  using Args = TinyFwdArgs<T>;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int, int, int tid, void *) {
    if ((unsigned)tid >= a.N) return;
    double sr = 0, si = 0;
    for (unsigned n = 0; n < a.N && (long long)n < a.n0; ++n) {
      double sn, cs;
      sincospi_hd(2.0 * (double)(((unsigned)tid * n) % a.N) / (double)a.N, &sn, &cs);
      sr += (double)a.sig[n] * cs;
      si -= (double)a.sig[n] * sn;
    }
    a.spec[tid] = mk<T>((T)sr, (T)si);
  }
};


// ---- Body: icwt reduction  out[n] (+)= sum_j Re(W[j,n]) / sqrt(s_j)   (wavelet.py:169-170) ----
template <typename T> struct IcwtArgs {
  const cx<T> *W;
  const double *inv_sqrt_s;   // per row: 1 / sqrt(s_j)
  double *out;
  long long n, pitch;
  int rows, accumulate;
  int rows_per_block;         // gridDim.y blocks of rows; > 1 block: partial sums meet in `out` by atomics
};
// One column per thread, rows in blocks of `rows_per_block` (blockIdx.y), 8 independent loads in
// flight per thread: a streaming read of W at HBM rate (4.29 GB at config 2).
template <typename T> struct IcwtBody {
  using Args = IcwtArgs<T>;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const long long n = (long long)bx * NT + tid;
    if (n >= a.n) return;
    const int j0 = by * a.rows_per_block;
    const int j1 = j0 + a.rows_per_block < a.rows ? j0 + a.rows_per_block : a.rows;
    const cx<T> *p = a.W + (size_t)j0 * a.pitch + n;
    double acc0 = 0, acc1 = 0;
    int j = j0;
    for (; j + 8 <= j1; j += 8) {
      double v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = (double)ldg(&p[(size_t)u * a.pitch]).x;
#pragma unroll
      for (int u = 0; u < 8; u += 2) {
        acc0 += v[u] * a.inv_sqrt_s[j + u];
        acc1 += v[u + 1] * a.inv_sqrt_s[j + u + 1];
      }
      p += (size_t)8 * a.pitch;
    }
    for (; j < j1; ++j, p += a.pitch) acc0 += (double)ldg(p).x * a.inv_sqrt_s[j];
    const double acc = acc0 + acc1;
    if (a.rows_per_block >= a.rows) {
      a.out[n] = a.accumulate ? a.out[n] + acc : acc;
    } else {
#if defined(__CUDA_ARCH__) && !defined(CWTB_HOST_EMU)
      atomicAdd(&a.out[n], acc);
#else
      a.out[n] += acc;
#endif
    }
  }
};

// ---- Body: coherence inputs (wavelet.py:506-514) ---------------------------------------
//   C   = (|W1|^2 + i |W2|^2) / s   (two real fields packed into one complex field: the
//         smoothing filter is real, so one complex transform smooths both)
//   A12 = W1 conj(W2) / s,   aWCT = angle(W1 conj(W2))
struct WctPrepArgs {
  const double2 *W1, *W2;
  const double *scale;   // per row
  double2 *C, *A12;
  double *aWCT;          // may be null
  long long n;
};
struct WctPrepBody {
  using Args = WctPrepArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const long long n = (long long)bx * NT + tid;
    if (n >= a.n) return;
    const size_t i = (size_t)by * a.n + n;
    const double2 w1 = a.W1[i], w2 = a.W2[i];
    const double s = a.scale[by];
    const double2 w12 = cmul(w1, cconj(w2));
    a.C[i] = make_double2((w1.x * w1.x + w1.y * w1.y) / s, (w2.x * w2.x + w2.y * w2.y) / s);
    a.A12[i] = make_double2(w12.x / s, w12.y / s);
    if (a.aWCT) a.aWCT[i] = atan2(w12.y, w12.x);
  }
};

// ---- Body: white-noise surrogates on the device (seeded mode of the Monte-Carlo significance) ----
// Counter-based Philox4x32-10 (Salmon et al. 2011): sample pair (2j, 2j+1) of series `ser` of
// surrogate pair `pair` is a pure function of (seed, pair, ser, j) -- independent of the launch
// geometry, of the rank that draws it and of how the pairs are batched.  Two 53-bit uniforms ->
// two standard normals (Box-Muller).  The reference's surrogates are white noise as well
// (helpers.py:146-173 filters a length-1 axis, SURVEY 8a row 10); this mode reproduces their
// distribution, not numpy's bit stream (the host-RNG mode does that).
struct NoiseArgs {
  double *out;              // [n_pairs][2][n]
  unsigned long long seed;
  long long pair0;          // global index of the first pair
  long long n;
  int n_pairs;
};
HD void philox4x32_10(unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned k0, unsigned k1, unsigned (&o)[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0;
    const unsigned long long p1 = (unsigned long long)0xCD9E8D57u * c2;
    const unsigned n0 = (unsigned)(p1 >> 32) ^ c1 ^ k0, n1 = (unsigned)p1;
    const unsigned n2 = (unsigned)(p0 >> 32) ^ c3 ^ k1, n3 = (unsigned)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  o[0] = c0; o[1] = c1; o[2] = c2; o[3] = c3;
}
struct NoiseBody {
  using Args = NoiseArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const long long j = (long long)bx * NT + tid;        // sample pair index
    if (2 * j >= a.n) return;
    const long long pair = a.pair0 + by / 2;
    const int ser = by & 1;
    unsigned o[4];
    philox4x32_10((unsigned)j, (unsigned)((unsigned long long)j >> 32), (unsigned)pair,
                  ((unsigned)((unsigned long long)pair >> 32) << 1) | (unsigned)ser,
                  (unsigned)a.seed, (unsigned)(a.seed >> 32), o);
    // uniforms in (0, 1): 53 bits from two words, offset by half an ulp so that log() is finite
    const double u1 = ((double)(o[0] >> 5) * 67108864.0 + (double)(o[1] >> 6) + 0.5) * (1.0 / 9007199254740992.0);
    const double u2 = ((double)(o[2] >> 5) * 67108864.0 + (double)(o[3] >> 6) + 0.5) * (1.0 / 9007199254740992.0);
    const double r = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi_hd(2.0 * u2, &sn, &cs);
    double *dst = a.out + (size_t)by * a.n + 2 * j;
    dst[0] = r * cs;
    if (2 * j + 1 < a.n) dst[1] = r * sn;
  }
};

// ---- Body: scale-axis boxcar (mothers.py:100-102; scipy convolve2d 'same', zero fill) ------
//   out[i] = sum_t win[t] * in[i - (t - off)],  off = (K-1)//2, rows outside [0, m) are zero
struct BoxcarArgs {
  const double2 *in;
  double2 *out;
  const double *win;
  long long n;
  int rows, K;
};
HD double2 boxcar_at(const double2 *in, const double *win, int K, int rows, long long n, int i, long long col) {
  const int off = (K - 1) / 2;
  double re = 0, im = 0;
  for (int t = 0; t < K; ++t) {
    const int q = i - (t - off);
    if (q < 0 || q >= rows) continue;
    const double2 v = in[(size_t)q * n + col];
    re += win[t] * v.x;
    im += win[t] * v.y;
  }
  return make_double2(re, im);
}
struct BoxcarBody {
  using Args = BoxcarArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const long long n = (long long)bx * NT + tid;
    if (n >= a.n) return;
    a.out[(size_t)by * a.n + n] = boxcar_at(a.in, a.win, a.K, a.rows, a.n, by, n);
  }
};

// ---- Body: coherence  WCT = |S12|^2 / (S1 S2)  after the scale boxcar; optional histogram
// of floor(WCT * nbins) over masked points (wavelet.py:513, 624-630) ---------------------
struct WctFinalArgs {
  const double2 *C, *A12;   // time-smoothed fields
  const double *win;
  double *WCT;              // may be null (Monte-Carlo mode)
  const unsigned char *mask;   // [rows][n], may be null
  unsigned long long *hist;    // [rows][nbins], may be null
  long long n;
  int rows, K, maxscale, nbins;
};
// Tile: RS = 32 output rows x CW = 32 columns.  Phase 0 stages the RS + K - 1 input rows of both
// time-smoothed fields for these columns in shared memory (each input element is read from global
// memory (RS + K - 1) / RS times instead of K times); in phase 1 a thread produces 4 consecutive
// rows of one column, so every staged value feeds up to four accumulators.
template <int KMAX_> struct WctFinalBody {
  using Args = WctFinalArgs;
  static constexpr int NPHASE = 2;
  static constexpr int RS = 32, CW = 32, KMAX = KMAX_, RG = 4;   // KMAX sizes the shared memory
  static constexpr size_t SMEM = (size_t)2 * (RS + KMAX - 1) * CW * sizeof(double2) + KMAX * sizeof(double);
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *smraw) {
    const int K = a.K, off = (K - 1) / 2;
    const int nrow = RS + K - 1;
    double2 *sc = (double2 *)smraw;                   // [nrow][CW] of C
    double2 *sx = sc + (size_t)(RS + KMAX - 1) * CW;  // [nrow][CW] of A12
    double *sw = (double *)(sx + (size_t)(RS + KMAX - 1) * CW);
    const int i0 = by * RS;
    const long long n0 = (long long)bx * CW;
    const int rows_out = a.WCT ? a.rows : a.maxscale;  // Monte-Carlo mode: rows below maxscale only
    if (i0 >= rows_out) return;
    const int qlo = i0 + off - K + 1;
    if constexpr (PH == 0) {
      for (int idx = tid; idx < nrow * CW; idx += NT) {
        const int r = idx / CW, col = idx % CW;
        const int q = qlo + r;
        const long long n = n0 + col;
        double2 c = make_double2(0.0, 0.0), x = c;
        if (q >= 0 && q < a.rows && n < a.n) {
          c = a.C[(size_t)q * a.n + n];
          x = a.A12[(size_t)q * a.n + n];
        }
        sc[idx] = c;
        sx[idx] = x;
      }
      for (int t = tid; t < K; t += NT) sw[t] = a.win[t];
    } else {
      for (int task = tid; task < (RS / RG) * CW; task += NT) {
        const int col = task % CW, g = task / CW;
        const long long n = n0 + col;
        if (n >= a.n) continue;
        double cr[RG] = {0, 0, 0, 0}, ci[RG] = {0, 0, 0, 0}, xr[RG] = {0, 0, 0, 0}, xi[RG] = {0, 0, 0, 0};
        // staged row u feeds output row i0 + RG g + e with tap t = e + K - 1 - (u - RG g)
        for (int du = 0; du < K + RG - 1; ++du) {
          const int u = RG * g + du;
          const double2 c = sc[u * CW + col], x = sx[u * CW + col];
#pragma unroll
          for (int e = 0; e < RG; ++e) {
            const int t = e + K - 1 - du;
            if (t >= 0 && t < K) {
              const double w = sw[t];
              cr[e] += w * c.x; ci[e] += w * c.y;
              xr[e] += w * x.x; xi[e] += w * x.y;
            }
          }
        }
#pragma unroll
        for (int e = 0; e < RG; ++e) {
          const int i = i0 + RG * g + e;
          if (i >= rows_out) break;
          const double r2 = (xr[e] * xr[e] + xi[e] * xi[e]) / (cr[e] * ci[e]);
          const size_t o = (size_t)i * a.n + n;
          if (a.WCT) a.WCT[o] = r2;
          if (a.hist && i < a.maxscale && a.mask[o] && r2 == r2) {
            int bin = (int)floor(r2 * a.nbins);
            bin = bin < 0 ? 0 : (bin >= a.nbins ? a.nbins - 1 : bin);
#if defined(__CUDA_ARCH__) && !defined(CWTB_HOST_EMU)
            atomicAdd(&a.hist[(size_t)i * a.nbins + bin], 1ull);
#else
            a.hist[(size_t)i * a.nbins + bin] += 1ull;
#endif
          }
        }
      }
    }
  }
};

// ---- Body: |W|^2 and its row means (SURVEY 8f: device-side derived products) ---------------
template <typename T> struct PowerArgs {
  const cx<T> *W;
  double *power;     // [rows][n] or null
  double *rowsum;    // [rows] accumulated with atomics, or null
  long long n;
  const double *rowmul;        // per-row factor of the stored power (rectification 1/s_j), or null
  const long long *lo, *hi;    // per-row column range [lo, hi) of the row sum, or null (all)
};
template <typename T> struct PowerBody {
  using Args = PowerArgs<T>;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  static constexpr int PER = 64;   // columns per thread, in four rounds of 16 independent 16-byte loads
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    // one atomic per warp for the row sum; four rounds per CTA: the atomics of a row all hit one
    // address and serialise in L2 (2048 of them per 2^20-point row with one round per CTA cost as
    // much as the 4.29 GB read)
    double acc = 0;
    const double mul = a.rowmul ? a.rowmul[by] : 1.0;
    const long long lo = a.lo ? a.lo[by] : 0, hi = a.hi ? a.hi[by] : a.n;
    const cx<T> *row = a.W + (size_t)by * a.n;
    for (int rd = 0; rd < 4; ++rd) {
      const long long n0 = ((long long)bx * 4 + rd) * 16 * NT + tid;
      if (n0 - tid >= a.n) break;
      cx<T> w[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const long long n = n0 + (long long)i * NT;
        w[i] = n < a.n ? ldg(&row[n]) : mk<T>(0, 0);
      }
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const long long n = n0 + (long long)i * NT;
        const double p = ((double)w[i].x * w[i].x + (double)w[i].y * w[i].y) * mul;
        if (a.power && n < a.n) st_stream(&a.power[(size_t)by * a.n + n], p);
        if (n >= lo && n < hi) acc += p;
      }
    }
    if (a.rowsum) {
#if defined(__CUDA_ARCH__) && !defined(CWTB_HOST_EMU)
      // one atomic per warp (every lane reaches this point: no early return above)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
      if ((tid & 31) == 0) atomicAdd(&a.rowsum[by], acc);
#else
      a.rowsum[by] += acc;
#endif
    }
  }
};

// ---- Body: scale-averaged power  out[n] = sum_j w_j |W[j,n]|^2  (TC98 eq. 24; the sample
// scripts' `scale_avg`, simple_sample.py:88-91).  Rows with w_j = 0 are not read. ------------
template <typename T> struct ScaleAvgArgs {
  const cx<T> *W;
  const double *w;   // per row
  double *out;
  long long n;
  int rows;
  const int *sel;    // rows with a non-zero weight, ascending (device)
  int nsel;
  int sel_per_block; // gridDim.y blocks of selected rows; > 1 block: atomics into `out`
};
template <typename T> struct ScaleAvgBody {
  using Args = ScaleAvgArgs<T>;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const long long n = (long long)bx * NT + tid;
    if (n >= a.n) return;
    const int i0 = by * a.sel_per_block;
    const int i1 = i0 + a.sel_per_block < a.nsel ? i0 + a.sel_per_block : a.nsel;
    double acc0 = 0, acc1 = 0;
    int i = i0;
    for (; i + 4 <= i1; i += 4) {
      cx<T> v[4];
      double wj[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = a.sel[i + u];
        wj[u] = a.w[j];
        v[u] = ldg(&a.W[(size_t)j * a.n + n]);
      }
      acc0 += wj[0] * ((double)v[0].x * v[0].x + (double)v[0].y * v[0].y);
      acc1 += wj[1] * ((double)v[1].x * v[1].x + (double)v[1].y * v[1].y);
      acc0 += wj[2] * ((double)v[2].x * v[2].x + (double)v[2].y * v[2].y);
      acc1 += wj[3] * ((double)v[3].x * v[3].x + (double)v[3].y * v[3].y);
    }
    for (; i < i1; ++i) {
      const int j = a.sel[i];
      const cx<T> v = ldg(&a.W[(size_t)j * a.n + n]);
      acc0 += a.w[j] * ((double)v.x * v.x + (double)v.y * v.y);
    }
    const double acc = acc0 + acc1;
    if (a.sel_per_block >= a.nsel) {
      a.out[n] = acc;
    } else {
#if defined(__CUDA_ARCH__) && !defined(CWTB_HOST_EMU)
      atomicAdd(&a.out[n], acc);
#else
      a.out[n] += acc;
#endif
    }
  }
};

// ---- Body: per-channel products of a resident batch chunk W[nc][S][n] in one read ----------
// For every channel c (blockIdx.y) and rows j0 <= j < j1 (simple_sample.py lines in brackets):
//   rowsum[c][j]     += sum_n |W|^2                      (global spectrum before / n, :79)
//   rowsum_coi[c][j] += sum_{lo_j <= n < hi_j} |W|^2     (the same inside the COI)
//   band[c][b][n]    (+)= chan_scale[c] * sum_j wt[b][j] |W[c,j,n]|^2   (scale_avg, :88-91)
//   isum[c][n]       (+)= fac * sum_j Re(W[c,j,n]) / sqrt(s_j)          (iwave, :60; complex fac:
//                         isum[c][n][2] = (re, im))
// One CTA owns a tile of TILE columns of one channel across all rows of the launch, so the
// column outputs are written once by one thread, without atomics (bit-identical run to run).
// The row sums are reduced in the warp, then in shared memory, and leave the CTA as one atomic
// per row (PowerBody's note: per-warp atomics on one row address cost as much as the read).
// NB: band accumulators per column (the bands in use, nb <= NB, are a launch argument).
template <typename T> struct BatchProductsArgs {
  const cx<T> *W;              // [nc][S][n]
  const double *wt;            // [NB][S] band weights (rows b >= nb are not read)
  const double *inv_sqrt_s;    // [S]
  const long long *lo, *hi;    // [S] COI column ranges, or null
  const double *chan_scale;    // [nc] (chunk's first channel), or null (1)
  double *rowsum, *rowsum_coi; // [nc][S] (chunk's first channel); rowsum_coi null without ranges
  double *band;                // [nc][nb][n], or null
  double *isum;                // [nc][n] (icplx 0) or [nc][n][2] (icplx 1), or null
  double fre, fim;             // icwt factor dj sqrt(dt) / (Cdelta psi(0))
  long long n;
  int S, nb, icplx;
  int j0, j1, accumulate;      // rows of this launch (<= RMAX); accumulate: add to the column outputs
};
template <typename T, int NB> struct BatchProductsBody {
  using Args = BatchProductsArgs<T>;
  static constexpr int NPHASE = 3;
  static constexpr int NTB = 256, CPT = 8, TILE = NTB * CPT;   // 2048 columns per CTA
  static constexpr int U = sizeof(T) == 4 && NB <= 2 ? 2 : 1;  // rows per step: 16 loads of 8 B or 8 of 16 B in flight
  static constexpr int MINB = NB <= 2 ? 2 : 1;                 // 8 bands: 72 accumulators per thread
  static constexpr int RMAX = 1024;                            // rows per launch (shared row sums)
  static constexpr size_t SMEM = 2 * RMAX * sizeof(double);
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *smraw) {
    double *srow = (double *)smraw, *scoi = srow + RMAX;
    const int nr = a.j1 - a.j0;
    if constexpr (PH == 0) {
      for (int r = tid; r < nr; r += NTB) { srow[r] = 0; scoi[r] = 0; }
    } else if constexpr (PH == 1) {
      const int nbase = bx * TILE + tid, ncol = (int)a.n;   // (32-bit columns: n < 2^28)
      const cx<T> *Wc = a.W + (size_t)by * a.S * a.n;
      double bacc[NB][CPT], iacc[CPT];
#pragma unroll
      for (int i = 0; i < CPT; ++i) {
        iacc[i] = 0;
#pragma unroll
        for (int b = 0; b < NB; ++b) bacc[b][i] = 0;
      }
      for (int j = a.j0; j < a.j1; j += U) {
        cx<T> w[U][CPT];
        const cx<T> *row = Wc + (size_t)j * a.n + nbase;
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
          for (int i = 0; i < CPT; ++i)
            w[u][i] = (j + u < a.j1 && nbase + i * NTB < ncol) ? ldg(&row[(size_t)u * a.n + i * NTB]) : mk<T>(0, 0);
        double part[2 * U];   // row sum, COI row sum of each row of the step (this thread's columns)
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int jr = j + u < a.j1 ? j + u : a.j1 - 1;   // rows past the end hold zeros
          const double is = ldg(&a.inv_sqrt_s[jr]);
          double wb[NB];
#pragma unroll
          for (int b = 0; b < NB; ++b) wb[b] = b < a.nb ? ldg(&a.wt[(size_t)b * a.S + jr]) : 0.0;
          const int lo = a.lo ? (int)ldg(&a.lo[jr]) : 0, hi = a.lo ? (int)ldg(&a.hi[jr]) : 0;
          double rs = 0, rc = 0;
#pragma unroll
          for (int i = 0; i < CPT; ++i) {
            const int n = nbase + i * NTB;
            const double x = (double)w[u][i].x, y = (double)w[u][i].y;
            const double p = x * x + y * y;
            rs += p;
            rc += (n >= lo && n < hi) ? p : 0.0;
#pragma unroll
            for (int b = 0; b < NB; ++b) bacc[b][i] += wb[b] * p;
            iacc[i] += x * is;
          }
          part[2 * u] = rs;
          part[2 * u + 1] = rc;
        }
#if defined(__CUDA_ARCH__) && !defined(CWTB_HOST_EMU)
        // 2U sums over the warp in (2U - 1) + (5 - log2 2U) shuffles: each halving step trades half
        // of the values with the partner lane, so lane l ends with the total of value l % 2U
        const int lane = tid & 31;
#pragma unroll
        for (int h = U; h >= 1; h >>= 1) {
          const bool up = (lane & h) != 0;
#pragma unroll
          for (int v = 0; v < h; ++v) {
            const double send = up ? part[v] : part[v + h];
            const double keep = up ? part[v + h] : part[v];
            part[v] = keep + __shfl_xor_sync(0xffffffffu, send, h);
          }
        }
#pragma unroll
        for (int o = 2 * U; o < 32; o <<= 1) part[0] += __shfl_xor_sync(0xffffffffu, part[0], o);
        if (lane < 2 * U && j + lane / 2 < a.j1) atomicAdd(&((lane & 1) ? scoi : srow)[j + lane / 2 - a.j0], part[0]);
#else
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (j + u < a.j1) { srow[j + u - a.j0] += part[2 * u]; scoi[j + u - a.j0] += part[2 * u + 1]; }
#endif
      }
      const double cs = a.chan_scale ? a.chan_scale[by] : 1.0;
#pragma unroll
      for (int i = 0; i < CPT; ++i) {
        const int n = nbase + i * NTB;
        if (n >= ncol) continue;
        if (a.band)
#pragma unroll
          for (int b = 0; b < NB; ++b) {
            if (b >= a.nb) break;
            double *o = &a.band[((size_t)by * a.nb + b) * a.n + n];
            *o = a.accumulate ? *o + cs * bacc[b][i] : cs * bacc[b][i];
          }
        if (a.isum) {
          if (a.icplx) {
            double *o = &a.isum[((size_t)by * a.n + n) * 2];
            o[0] = a.accumulate ? o[0] + a.fre * iacc[i] : a.fre * iacc[i];
            o[1] = a.accumulate ? o[1] + a.fim * iacc[i] : a.fim * iacc[i];
          } else {
            double *o = &a.isum[(size_t)by * a.n + n];
            *o = a.accumulate ? *o + a.fre * iacc[i] : a.fre * iacc[i];
          }
        }
      }
    } else {
      for (int r = tid; r < nr; r += NTB) {
        const size_t o = (size_t)by * a.S + a.j0 + r;
#if defined(__CUDA_ARCH__) && !defined(CWTB_HOST_EMU)
        atomicAdd(&a.rowsum[o], srow[r]);
        if (a.rowsum_coi) atomicAdd(&a.rowsum_coi[o], scoi[r]);
#else
        a.rowsum[o] += srow[r];
        if (a.rowsum_coi) a.rowsum_coi[o] += scoi[r];
#endif
      }
    }
  }
};

// ---- Body: real -> complex widening / complex -> real part ---------------------------------
struct R2CArgs { const double *in; double2 *out; long long count; };
struct R2CBody {
  using Args = R2CArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int, int tid, void *) {
    const long long i = (long long)bx * NT + tid;
    if (i < a.count) a.out[i] = make_double2(a.in[i], 0.0);
  }
};

// ---- Body: out[i] = in[i] * f ------------------------------------------------------------
struct ScaleCopyArgs { const double *in; double *out; long long count; double f; };
struct ScaleCopyBody {
  using Args = ScaleCopyArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int, int tid, void *) {
    const long long i = (long long)bx * NT + tid;
    if (i < a.count) a.out[i] = a.in[i] * a.f;
  }
};

// ---- Body: complex64 -> complex128 (fp32 transforms returned through the reference API) ----
struct WidenArgs { const float2 *in; double2 *out; long long count; };
struct WidenBody {
  using Args = WidenArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int, int tid, void *) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long long i = ((long long)bx * 4 + u) * NT + tid;
      if (i < a.count) {
        const float2 v = a.in[i];
        a.out[i] = make_double2((double)v.x, (double)v.y);
      }
    }
  }
};

// ---- Bluestein (chirp-z) pieces: DFT of ARBITRARY length n through power-of-two transforms ----
// (un-padded mode, pycwt/helpers.py:15-19: with pyfftw installed the reference transforms at the
// signal's own length).  With w_s[k] = e^{s i pi k^2 / n}  (s = -1 forward, +1 inverse):
//   X[k] = sum_j x[j] e^{s 2 pi i jk/n} = w_s[k] * sum_j (x[j] w_s[j]) conj(w_s[k-j]),
// a linear convolution of length 2n-1 evaluated with transforms of length L = 2^m >= 2n-1:
//   a = x * w_s (zero-padded to L),  b[m] = conj(w_s[|m|]) for |m| < n (wrapped mod L),
//   X[k] = w_s[k] / L * IFFT_L( FFT_L(a) * FFT_L(b) )[k].
// One table wm[k] = e^{-i pi k^2/n} serves both signs (w_+ = conj(wm)); k^2 is reduced mod 2n in
// integers so the phase is exact.
struct BlueChirpArgs { double2 *wm; unsigned n; };
struct BlueChirpBody {
  using Args = BlueChirpArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int, int tid, void *) {
    const unsigned long long k = (unsigned long long)bx * NT + tid;
    if (k >= a.n) return;
    const unsigned long long m = (k * k) % (2ull * a.n);
    double sn, cs;
    sincospi_hd((double)m / (double)a.n, &sn, &cs);
    a.wm[k] = make_double2(cs, -sn);
  }
};

HD double2 blue_w(const double2 *wm, unsigned k, int sign) {   // w_s[k]
  const double2 v = wm[k];
  return sign < 0 ? v : make_double2(v.x, -v.y);
}

struct BlueFilterArgs { const double2 *wm; double2 *b; unsigned n, L; int sign; };
struct BlueFilterBody {
  using Args = BlueFilterArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int, int tid, void *) {
    const unsigned m = (unsigned)bx * NT + tid;
    if (m >= a.L) return;
    double2 v = make_double2(0.0, 0.0);
    if (m < a.n) v = blue_w(a.wm, m, -a.sign);             // conj(w_s[m])
    else if (m > a.L - a.n) v = blue_w(a.wm, a.L - m, -a.sign);
    a.b[m] = v;
  }
};

// a[r][k] = in[r][k] * w_s[k]   (rows of a generic transform)
struct BluePreArgs {
  const void *in; double2 *out; const double2 *wm;
  long long in_pitch, out_pitch; unsigned n; int real_in, sign;
};
struct BluePreBody {
  using Args = BluePreArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const unsigned k = (unsigned)bx * NT + tid;
    if (k >= a.n) return;
    double2 x;
    if (a.real_in) x = make_double2(((const double *)a.in)[(size_t)by * a.in_pitch + k], 0.0);
    else x = ((const double2 *)a.in)[(size_t)by * a.in_pitch + k];
    a.out[(size_t)by * a.out_pitch + k] = cmul(x, blue_w(a.wm, k, a.sign));
  }
};

// a[r][k] = x^[k] * norm_j conj(psi^(s_j w_k)) / n * w_+[k]: product of wavelet.py:102-104 and the
// chirp pre-multiplication of the inverse transform in one pass
struct BlueProdArgs {
  const ScaleDesc *descs; const double2 *spec; double2 *out; const double2 *wm;
  Fam fam; long long out_pitch; unsigned n; int first;
};
struct BlueProdBody {
  using Args = BlueProdArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const unsigned k = (unsigned)bx * NT + tid;
    if (k >= a.n) return;
    const ScaleDesc d = a.descs[a.first + by];
    // numpy fftfreq ordering for any n: bins 0 .. (n-1)/2 are non-negative
    const int ks = k < (a.n + 1) / 2 ? (int)k : (int)k - (int)a.n;
    double2 v = make_double2(0.0, 0.0);
    if (a.fam.family == 3 || (ks >= d.k_lo && ks <= d.k_hi)) v = band_value<double>(a.fam, d, a.spec, k, ks, a.n);
    a.out[(size_t)by * a.out_pitch + k] = cmul(v, blue_w(a.wm, k, +1));
  }
};

struct BlueMulArgs { double2 *x; const double2 *bf; unsigned L; };
struct BlueMulBody {
  using Args = BlueMulArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const unsigned m = (unsigned)bx * NT + tid;
    if (m >= a.L) return;
    double2 *p = a.x + (size_t)by * a.L + m;
    *p = cmul(*p, a.bf[m]);
  }
};

// F[r][k] *= filt[r][k] * post: a caller-supplied real frequency response per row (time smoothing
// with a filter other than Morlet's Gaussian: cwtb_set_smooth_filter)
struct FilterMulArgs { double2 *f; const double *filt; long long pitch; unsigned n; double post; };
struct FilterMulBody {
  using Args = FilterMulArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const unsigned k = (unsigned)bx * NT + tid;
    if (k >= a.n) return;
    const double m = a.filt[(size_t)by * a.n + k] * a.post;
    double2 *p = a.f + (size_t)by * a.pitch + k;
    p->x *= m; p->y *= m;
  }
};

// out[row][k] = epilogue(y[r][k] * w_s[k] * scale)
struct BluePostArgs {
  const double2 *y; double2 *out; const double2 *wm; const ScaleDesc *descs;   // descs may be null
  long long out_pitch, nout; double scale; unsigned L; int first, row0, sign, epi;
};
struct BluePostBody {
  using Args = BluePostArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const long long k = (long long)bx * NT + tid;
    if (k >= a.nout) return;
    const int row = a.descs ? a.descs[a.first + by].row : a.row0 + by;
    double2 v = cmul(a.y[(size_t)by * a.L + k], blue_w(a.wm, (unsigned)k, a.sign));
    v.x *= a.scale; v.y *= a.scale;
    double2 *o = a.out + (size_t)row * a.out_pitch + k;
    if (a.epi == EPI_MULCONJ) v = cmul(*o, cconj(v));
    *o = v;
  }
};

// F[r][k] *= exp(g_r * w_k^2) * post,  w_k = 2 pi fftfreq(n)[k]: the Gaussian time filter of
// Morlet.smooth (mothers.py:83-91) for a transform length that is not a power of two
struct BlueGaussArgs { double2 *f; const double *g; long long pitch; unsigned n; double post; };
struct BlueGaussBody {
  using Args = BlueGaussArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int by, int tid, void *) {
    const unsigned k = (unsigned)bx * NT + tid;
    if (k >= a.n) return;
    const long long ks = k < (a.n + 1) / 2 ? (long long)k : (long long)k - (long long)a.n;
    const double w = 6.283185307179586 * ((double)ks * (1.0 / (double)a.n));
    const double m = exp(a.g[by] * (w * w)) * a.post;
    double2 *p = a.f + (size_t)by * a.pitch + k;
    p->x *= m; p->y *= m;
  }
};

// ---- Body: pass twiddle tables in [c][j] layout (see fft_tile.cuh: tw_offset) -------------
struct PassTwArgs {
  double2 *out64;
  float2 *out32;
};
struct PassTwBody {
  using Args = PassTwArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int, int tid, void *) {
    const int idx = bx * NT + tid;
    if (idx >= TW_TOTAL) return;
    int L = 32;
    while (L < 1024 && idx >= tw_offset(2 * L)) L *= 2;
    const int R = tw_radix(L), Ln = L / R;
    const int rel = idx - tw_offset(L);
    const int c = rel / Ln + 1, j = rel % Ln;
    double sn, cs;
    sincospi_hd(2.0 * (double)(j * c) / (double)L, &sn, &cs);
    (void)R;
    a.out64[idx] = make_double2(cs, sn);
    a.out32[idx] = make_float2((float)cs, (float)sn);
  }
};

// ---- Body: twiddle tables ---------------------------------------------------------
struct TabArgs {
  double2 *out64;
  float2 *out32;
  unsigned count;
  double step;  // entry i = e^{2 pi i * i * step}
};
struct TabBody {
  using Args = TabArgs;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int, int tid, void *) {
    const unsigned i = (unsigned)bx * NT + tid;
    if (i >= a.count) return;
    double sn, cs;
    sincospi_hd(2.0 * ((double)i * a.step), &sn, &cs);
    if (a.out64) a.out64[i] = make_double2(cs, sn);
    if (a.out32) a.out32[i] = make_float2((float)cs, (float)sn);
  }
};

}  // namespace cwtb
