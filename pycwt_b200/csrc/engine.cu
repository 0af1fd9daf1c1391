// B200-native CWT engine: host planning, kernel launches and the C ABI of
// include/cwt_b200.h.  Device code is in kernels.cuh / fft_tile.cuh / cplx.cuh.
//
// Build (sm_100a):   nvcc -std=c++17 -O3 -lineinfo -gencode arch=compute_100a,code=sm_100a
//                         -Xcompiler -fPIC -shared engine.cu -o libcwtb200.so
// Build (CPU emulation of the kernels, TESTS ONLY, never shipped/loaded by the package):
//                    nvcc -std=c++17 -O2 -DCWTB_HOST_EMU ... -o libcwtb200_emu.so
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <set>
#include <string>
#include <type_traits>
#include <vector>

#include <cuda_runtime.h>
#ifndef CWTB_HOST_EMU
#include <dlfcn.h>
#endif

#include "../../include/cwt_b200.h"
#include "kernels.cuh"

using namespace cwtb;

// threads per CTA of a kernel body: Body::NTB if it declares one (tile kernels: per precision),
// else the global NT
template <class B, class = void> struct BodyNT { static constexpr int value = NT; };
template <class B> struct BodyNT<B, std::void_t<decltype(B::NTB)>> { static constexpr int value = B::NTB; };


// ======================================================================================
// runtime abstraction
// ======================================================================================
#ifdef CWTB_HOST_EMU
typedef int rt_stream;
static inline int rt_malloc(void **p, size_t n) { *p = malloc(n ? n : 1); return *p ? 0 : 1; }
static inline int rt_free(void *p) { free(p); return 0; }
static inline int rt_host_alloc(void **p, size_t n) { *p = malloc(n ? n : 1); return *p ? 0 : 1; }
static inline int rt_host_free(void *p) { free(p); return 0; }
static inline int rt_h2d(void *d, const void *s, size_t n, rt_stream) { memcpy(d, s, n); return 0; }
static inline int rt_d2h(void *d, const void *s, size_t n, rt_stream) { memcpy(d, s, n); return 0; }
static inline int rt_memset(void *d, int v, size_t n, rt_stream) { memset(d, v, n); return 0; }
static inline int rt_sync(rt_stream) { return 0; }
static inline const char *rt_errstr(int) { return "emulation error"; }
#else
typedef cudaStream_t rt_stream;
static inline int rt_malloc(void **p, size_t n) { return (int)cudaMalloc(p, n ? n : 1); }
static inline int rt_free(void *p) { return (int)cudaFree(p); }
static inline int rt_host_alloc(void **p, size_t n) { return (int)cudaHostAlloc(p, n ? n : 1, cudaHostAllocDefault); }
static inline int rt_host_free(void *p) { return (int)cudaFreeHost(p); }
static inline int rt_h2d(void *d, const void *s, size_t n, rt_stream st) {
  return (int)cudaMemcpyAsync(d, s, n, cudaMemcpyHostToDevice, st);
}
static inline int rt_d2h(void *d, const void *s, size_t n, rt_stream st) {
  return (int)cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, st);
}
static inline int rt_memset(void *d, int v, size_t n, rt_stream st) { return (int)cudaMemsetAsync(d, v, n, st); }
static inline int rt_sync(rt_stream st) { return (int)cudaStreamSynchronize(st); }
static inline const char *rt_errstr(int e) { return cudaGetErrorString((cudaError_t)e); }

template <class B, class = void> struct BodyMinB { static constexpr int value = CWTB_MINB; };
template <class B> struct BodyMinB<B, std::void_t<decltype(B::MINB)>> { static constexpr int value = B::MINB; };

template <class Body, int PH>
__device__ __forceinline__ void run_phases(const typename Body::Args &a, void *sm) {
  Body::template phase<PH>(a, (int)blockIdx.x, (int)blockIdx.y, (int)threadIdx.x, sm);
  if constexpr (PH + 1 < Body::NPHASE) {
    __syncthreads();
    run_phases<Body, PH + 1>(a, sm);
  }
}
template <class Body, int PH>
__device__ __forceinline__ void run_phases_at(const typename Body::Args &a, int bx, int by, void *sm) {
  Body::template phase<PH>(a, bx, by, (int)threadIdx.x, sm);
  if constexpr (PH + 1 < Body::NPHASE) {
    __syncthreads();
    run_phases_at<Body, PH + 1>(a, bx, by, sm);
  }
}
template <class Body>
__global__ void __launch_bounds__(BodyNT<Body>::value, BodyMinB<Body>::value) k_run(const __grid_constant__ typename Body::Args a) {
  extern __shared__ __align__(16) unsigned char smraw[];
  run_phases<Body, 0>(a, smraw);
}
#endif

// ======================================================================================
// context
// ======================================================================================
struct Buf {
  void *p = nullptr;
  size_t bytes = 0;
};

struct ClassRun {   // scales sharing one execution plan
  int log2K;        // exact path: pruned length K' = 1 << log2K
  int first, count; // range in the sorted descriptor array
  int expand = 0;   // 1: band-limited expansion path (coarse transform + interpolation)
  int log2Nc = 0;   // expansion: coarse grid length
  int taps = 0;     // expansion: interpolation taps
  long long woff = 0;   // expansion: offset of the class's weight table
};

struct Job {
  bool valid = false;
  int precision = 0;       // CWTB_F64 / CWTB_F32
  long long n0 = 0;
  unsigned N = 0;
  int log2N = 0;
  int S = 0;          // scales per channel
  int nbatch = 1;     // channels transformed together (rows = nbatch * S)
  double dt = 0;
  Fam fam{};
  std::vector<ScaleDesc> descs;   // sorted by class
  std::vector<ClassRun> classes;
  std::vector<int> plan_log2K;    // per input scale
  std::vector<double> scales;     // per input scale (= output row)
  size_t b_single = 0;            // elements of the band buffer used by single-kernel scales
  size_t coarse_elems = 0;        // elements of the coarse buffers used by the expansion rows
  int sig_is_f32 = 0;
  bool exact = false;             // un-padded mode: N = n0 (not a power of two), Bluestein transforms
};

struct BluePlan {   // chirp tables of one transform length (device memory, owned by the context)
  unsigned n = 0, L = 0;
  double2 *wm = nullptr;                 // e^{-i pi k^2 / n}, k < n
  double2 *bf[2] = {nullptr, nullptr};   // FFT_L of the chirp filter for sign -1 / +1
};

struct NTabDev {
  double2 *hi = nullptr, *lo = nullptr;
  int h = 0;
};

struct cwtb_ctx {
  int device = 0;
  rt_stream stream{};
  rt_stream aux_stream{};        // single-kernel classes run here, concurrently with the two-kernel chains
  rt_stream prio_stream{};       // highest-priority stream: the chain of small launches in front of the
                                 // expansion kernels (band products + coarse transforms) -- its CTAs are
                                 // dispatched before the pending CTAs of the big launches on the other streams
  rt_stream prio_aux[7]{};       // the coarse transforms of different lengths are independent: they fan out
                                 // over the priority stream and these (own intermediates Zxs[]), so that the
                                 // chain in front of the expansion kernels is as long as its longest member,
                                 // not their sum (CWTB_PRIO_FAN=1..8 streams)
  int prio_fan = 4;
  int prio_mode = 1;             // CWTB_PRIO: 0 = no priority stream, 1 = coarse chain, 2 = coarse chain and
                                 // the expansion kernels
  rt_stream chain_streams[3]{};  // two-kernel classes rotate over the engine's stream and these (own Z
                                 // and band-chunk region per chain)
  int n_chains = 2;              // chains in use, 1..4 (CWTB_CHAINS)
  rt_stream cur{};               // stream the launcher uses right now
  int pad_pow2 = 1;              // 1: transform length = next power of two (reference default,
                                 // helpers.py:27-30); 0: the signal's own length (pyfftw policy,
                                 // helpers.py:15-19) -- cwtb_set_padding
  std::map<unsigned, BluePlan> blue;
  long long serial = 0;          // counts transforms: identifies what is resident (cwtb_job_serial)
  int two_streams = 1;           // CWTB_STREAMS=1 disables the overlap
  int three_streams = 1;         // CWTB_STREAMS=2: single-kernel classes only
  rt_stream copy_streams[4]{};   // large D2H copies are split over several streams / copy engines
  int d2h_split = 1;             // CWTB_D2H_SPLIT
  std::string err;
  double band_eps = 1e-16;
  double band_eps32 = 1e-9;      // fp32 engine: pruning threshold matched to the arithmetic (fp32
                                 // rounding is 6e-8; the dropped terms stay two orders below it)
  double expand_eps = 5e-13;     // fp64 engine: bound on the aliasing error of the expansion path
                                 // (0: path off, every scale through the exact pruned transforms)
  double expand_eps32 = 2e-7;    // fp32 engine
  int expand_mma = 1;            // fp64 expansion kernels with DMMA tap sums (CWTB_EXPAND_MMA=0: scalar kernel)
  int dense_margin = 2;          // pruned lengths within this many octaves of Np run as dense scales
                                 // (CWTB_DENSE_MARGIN; config 2: 1.710 -> 1.686 ms, profiles/r2/sweep_e.txt)
  int expand_min_log2R = 3;      // expansion needs Np / Nc >= 8 (CWTB_EXPAND_MIN_R: log2)
  Buf *ztmp = nullptr;           // intermediate of two_kernel_rows (set per stream; default Z)
  void *comm = nullptr;          // ncclComm_t of cwtb_comm_init (one rank per context)
  int comm_world = 1, comm_rank = 0;
  Buf comm_send, comm_recv;      // device staging of the host-buffer collectives
  int group = 0;   // rows per two-kernel chunk; 0 = as many as fit in group_bytes of Z (CWTB_GROUP)
  size_t group_bytes = (size_t)512 << 20;
  size_t rows_chunk_bytes = (size_t)256 << 20;  // CWTB_ROWS_CHUNK_MB: launches of >= 8 waves beat keeping the
                                                // intermediate in L2 (measured: wct 5.7 ms at 64 MiB, 4.8 ms at 256 MiB)
  int l2_persist = 0;
  int direct_max_log2 = 13;
  int fused = 0;     // experimental: two-kernel scales through one persistent kernel (CWTB_FUSED=1)
  int ring = 3;      // Z ring slots of the fused kernel
  int pipe_ahead = 2;   // CWTB_FUSED=2: scales the first kernel runs in front of the second (CWTB_AHEAD)
  int num_sms = 148;
  int pf_dist = 148;   // PassB: L2 prefetch distance in tiles (CWTB_PF_DIST)
  int gauss_rec = 1;   // dense Morlet scales: Gaussian by recurrence (CWTB_GAUSS_REC=0: exp per bin)
  int pf_rows_a = 32, pf_rows_b = 32;   // the same for the batched row transforms (CWTB_PF_ROWS_A / _B; wct 4.35 -> 4.25 ms)
  int pf_dist_a = 148;  // PassA (band): L2 prefetch distance in tiles (CWTB_PF_DIST_A)
  int k2_512_max_log2 = 16;  // largest K' that uses the 512-point second pass (CWTB_K2_512_MAX)
  int passb_rev = 1;    // second kernel walks the rows of a launch last-to-first (CWTB_PASSB_REV)
  int k2_band_log2 = 9; // second-pass length of the pruned two-kernel scales: 2^9 or 2^10 (CWTB_K2_BAND)
  size_t batch_bytes = (size_t)4 << 30;   // coefficients per chunk of cwtb_cwt_batch  // K' <= 2^13 handled by one kernel (K' > 1024: DirectBody)
  double2 *tw64 = nullptr;
  float2 *tw32 = nullptr;
  std::map<unsigned, NTabDev> ntabs;
  Buf filt;                      // caller-supplied time-smoothing responses [S][N] (cwtb_set_smooth_filter)
  int filt_rows = 0;
  long long filt_n = 0;
  Buf Zxs[7];                    // intermediates of the coarse transforms on prio_aux[]
  Buf Zx, Cin, Cout, wtab;       // expansion path: its own transform intermediate, coarse spectra /
                                 // samples, interpolation weight tables
  std::map<std::array<long long, 3>, long long> wtab_index;   // (log2R, taps, round(beta*1e6)) -> offset
  std::vector<double> wtab_host; // host mirror of wtab (tables are appended, never moved)
  size_t wtab_uploaded = 0;      // elements already on the device
  Buf ctr, sig, sig2, spec, Z, Zc[3], Y, B, W, W2, descs, table, scratch, C, A12, F, aux, rowd, win, mask, hist, noise, wide, blueA, blueX, blueY;
  Job job;
  // what the resident plan (job + uploaded descriptors) was built from: a call with the same
  // geometry and settings reuses it (planning + descriptor upload: ~0.3 ms for 256 scales, several ms
  // for the 8192 rows of a batch chunk)
  struct PlanKey {
    long long n0 = -1;
    double dt = 0, param = 0, band_eps = 0, band_eps32 = 0, expand_eps = 0, expand_eps32 = 0;
    int S = 0, family = 0, precision = 0, nbatch = 0, pad = 0;
    std::vector<double> scales;
    bool operator==(const PlanKey &o) const {
      return n0 == o.n0 && dt == o.dt && param == o.param && band_eps == o.band_eps && band_eps32 == o.band_eps32 &&
             expand_eps == o.expand_eps && expand_eps32 == o.expand_eps32 && S == o.S && family == o.family &&
             precision == o.precision && nbatch == o.nbatch && pad == o.pad && scales == o.scales;
    }
  } plan_key;
  int plan_reuse = 1;            // CWTB_PLAN_REUSE=0: plan every call
  // cwtb_cwt_batch pipeline: two page-locked staging buffers and two device input buffers so that the
  // host copy and the H2D of chunk k+1 overlap the kernels of chunk k; per-row power of every chunk is
  // accumulated on the device and read back once
  void *stage_host[2] = {nullptr, nullptr};
  size_t stage_bytes = 0;
  Buf stage_dev[2], batch_power;
  int batch_pipeline = 1;        // CWTB_BATCH_PIPELINE=0: one synchronous chunk after the other
  double *angle_host = nullptr;  // cwtb_wct: host destination of the phase angle, copied on a copy stream
                                 // as soon as it exists (before the smoothing transforms), not after them
  const void *job_dsig = nullptr;  // device signal of the last cwt_dev call (not owned)
  double last_ms = 0;
  int launches = 0;
  std::set<const void *> configured;
  // per-launch event profiling (cwtb_profile_last)
  bool profiling = false;
  int prof_saved_streams = 1;
  const char *prof_tag = "";     // prefix of the kernel names recorded while profiling: "fwd:" (forward
                                 // transform of the signal), "coarse:" (coarse-grid transforms of the
                                 // expansion path); W-writing launches carry no tag
  struct ProfRec { std::string name; unsigned gx, gy; int ev; };
  std::vector<ProfRec> prof;
#ifndef CWTB_HOST_EMU
  std::vector<cudaEvent_t> prof_events;
#endif
  std::set<void *> pinned, devallocs;
#ifndef CWTB_HOST_EMU
  cudaEvent_t e0{}, e1{};
  cudaEvent_t ev_fork{}, ev_join{}, ev_joinc[3]{}, ev_coarse{};
  cudaEvent_t ev_h2d[2]{}, ev_used[2]{};
  cudaEvent_t ev_xband{}, ev_pj[7]{}, ev_angle{};
#endif
};

static int fail(cwtb_ctx *c, int code, const std::string &msg);
static void apply_l2_policy(cwtb_ctx *c);
static int fail(cwtb_ctx *c, int code, const std::string &msg) {
  if (c) c->err = msg;
  return code;
}
#define RT(call)                                                                             \
  do {                                                                                       \
    int e_ = (call);                                                                         \
    if (e_ != 0) return fail(c, CWTB_ERR_CUDA, std::string(#call) + ": " + rt_errstr(e_));   \
  } while (0)

// Keep the Z buffer (intermediate of the two-kernel scales) resident in L2: persisting access
// policy window on the engine's stream; everything else keeps the default policy and W is
// written with streaming stores.  Re-applied whenever Z is (re)allocated.
static void apply_l2_policy(cwtb_ctx *c) {
#ifndef CWTB_HOST_EMU
  if (!c->l2_persist || !c->Z.p) return;
  int max_persist = 0, max_window = 0;
  cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, c->device);
  cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, c->device);
  if (max_persist <= 0 || max_window <= 0) return;
  const size_t want = std::min<size_t>(c->Z.bytes, (size_t)max_persist);
  cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want);
  cudaStreamAttrValue v{};
  v.accessPolicyWindow.base_ptr = c->Z.p;
  v.accessPolicyWindow.num_bytes = std::min<size_t>(c->Z.bytes, (size_t)max_window);
  v.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)want / (double)v.accessPolicyWindow.num_bytes);
  v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
  v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  cudaStreamSetAttribute(c->stream, cudaStreamAttributeAccessPolicyWindow, &v);
  cudaGetLastError();
#else
  (void)c;
#endif
}

static int ensure(cwtb_ctx *c, Buf &b, size_t bytes) {
  if (b.bytes >= bytes && b.p) return 0;
  if (b.p) rt_free(b.p);
  b.p = nullptr;
  b.bytes = 0;
  if (rt_malloc(&b.p, bytes) != 0) return fail(c, CWTB_ERR_NOMEM, "device allocation failed");
  b.bytes = bytes;
  if (&b == &c->Z) apply_l2_policy(c);
  return 0;
}

// ======================================================================================
// launcher
// ======================================================================================
#ifdef CWTB_HOST_EMU
template <class Body, int PH>
static void emu_phases(const typename Body::Args &a, int bx, int by, void *sm) {
  for (int tid = 0; tid < BodyNT<Body>::value; ++tid) Body::template phase<PH>(a, bx, by, tid, sm);
  if constexpr (PH + 1 < Body::NPHASE) emu_phases<Body, PH + 1>(a, bx, by, sm);
}
#endif

// "... [with Body = cwtb::PassBBody<double, 1>]"  ->  "PassBBody<double, 1>"
static std::string body_name(const char *pretty) {
  std::string s(pretty);
  size_t i = s.find("Body = ");
  if (i == std::string::npos) return s;
  s = s.substr(i + 7);
  size_t j = s.find_first_of(";]");
  if (j != std::string::npos) s = s.substr(0, j);
  if (s.rfind("cwtb::", 0) == 0) s = s.substr(6);
  return s;
}

template <class Body>
static int launch(cwtb_ctx *c, unsigned gx, unsigned gy, const typename Body::Args &a) {
  if (gx == 0 || gy == 0) return 0;
#ifdef CWTB_HOST_EMU
  std::vector<unsigned char> smv(Body::SMEM + 64);
  unsigned char *sm = smv.data();
  sm += (16 - ((unsigned long long)sm & 15)) & 15;   // 16-byte aligned base, like the device's
  for (unsigned by = 0; by < gy; ++by)
    for (unsigned bx = 0; bx < gx; ++bx) emu_phases<Body, 0>(a, (int)bx, (int)by, sm);
  c->launches++;
  if (emu_bulk_copy_faults() != 0) {
    emu_bulk_copy_faults() = 0;
    return fail(c, CWTB_ERR_CUDA, "emulation: bulk-async copy with a misaligned address or size");
  }
  return 0;
#else
  const void *fn = (const void *)k_run<Body>;
  if (Body::SMEM > 48 * 1024 && !c->configured.count(fn)) {
    RT(cudaFuncSetAttribute(k_run<Body>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Body::SMEM));
    c->configured.insert(fn);
  }
  // gridDim.y is limited to 65535
  if (gy > 65535) return fail(c, CWTB_ERR_ARG, "too many rows in one launch");
  int ev = -1;
  if (c->profiling) {
    ev = (int)c->prof.size() * 2;
    while ((int)c->prof_events.size() < ev + 2) {
      cudaEvent_t e;
      RT(cudaEventCreate(&e));
      c->prof_events.push_back(e);
    }
    c->prof.push_back({std::string(c->prof_tag) + body_name(__PRETTY_FUNCTION__), gx, gy, ev});
    RT(cudaEventRecord(c->prof_events[ev], c->cur));
  }
  k_run<Body><<<dim3(gx, gy), BodyNT<Body>::value, Body::SMEM, c->cur>>>(a);
  RT(cudaGetLastError());
  if (ev >= 0) RT(cudaEventRecord(c->prof_events[ev + 1], c->cur));
  c->launches++;
  return 0;
#endif
}

// ======================================================================================
// tables
// ======================================================================================
static int make_table(cwtb_ctx *c, double2 *o64, float2 *o32, unsigned count, double step) {
  TabArgs a{o64, o32, count, step};
  return launch<TabBody>(c, (count + NT - 1) / NT, 1, a);
}

static int init_tables(cwtb_ctx *c) {
  RT(rt_malloc((void **)&c->tw64, sizeof(double2) * TW_TOTAL));
  RT(rt_malloc((void **)&c->tw32, sizeof(float2) * TW_TOTAL));
  PassTwArgs a{c->tw64, c->tw32};
  return launch<PassTwBody>(c, (TW_TOTAL + NT - 1) / NT, 1, a);
}

static int get_ntab(cwtb_ctx *c, unsigned N, int log2N, NTab *out) {
  auto it = c->ntabs.find(N);
  if (it == c->ntabs.end()) {
    NTabDev t;
    t.h = (log2N + 1) / 2;
    unsigned nlo = 1u << t.h, nhi = N >> t.h;
    if (nhi == 0) nhi = 1;
    RT(rt_malloc((void **)&t.lo, sizeof(double2) * nlo));
    RT(rt_malloc((void **)&t.hi, sizeof(double2) * nhi));
    int e = make_table(c, t.lo, nullptr, nlo, 1.0 / (double)N);
    if (e) return e;
    e = make_table(c, t.hi, nullptr, nhi, (double)nlo / (double)N);
    if (e) return e;
    it = c->ntabs.emplace(N, t).first;
  }
  out->hi = it->second.hi;
  out->lo = it->second.lo;
  out->h = it->second.h;
  out->lomask = (1u << it->second.h) - 1;
  out->nmask = N - 1;
  return 0;
}

// ======================================================================================
// planning (host): band of each scale -> pruned length K'
// ======================================================================================
static int ilog2(unsigned long long v) {
  int l = 0;
  while ((1ull << l) < v) ++l;
  return l;
}

// largest f (beyond the maximum of g) with  m*ln f - a(f) = target
static double solve_upper(double m, bool gaussian, double target, double fstart) {
  auto g = [&](double f) { return m * std::log(f) - (gaussian ? 0.5 * f * f : f); };
  double lo = fstart, hi = fstart + 1;
  while (g(hi) > target && hi < 1e7) hi *= 2;
  for (int it = 0; it < 200; ++it) {
    double mid = 0.5 * (lo + hi);
    if (g(mid) > target) lo = mid; else hi = mid;
  }
  return hi;
}

// frequency-domain support [flo, fhi] (in f = s*w) where |psi_ft| >= eps * max|psi_ft|
static void family_band(int family, double param, double eps, double *flo, double *fhi, bool *pos_only) {
  const double LN_MIN = -745.2;  // exp() underflows to exactly 0 below this
  const double lneps = eps > 0 ? std::log(eps) : 0;
  *pos_only = false;
  if (family == CWTB_MORLET) {
    double xc = std::sqrt(-2.0 * (eps > 0 ? lneps : LN_MIN));
    *flo = param - xc;
    *fhi = param + xc;
  } else if (family == CWTB_PAUL) {
    double m = param;
    double target = eps > 0 ? lneps + (m * std::log(m) - m) : LN_MIN;
    *flo = 0;
    *fhi = solve_upper(m, false, target, m);
    *pos_only = true;
  } else {  // DOG
    double m = param;
    double mx = m > 0 ? 0.5 * m * std::log(m) - 0.5 * m : 0.0;
    double target = eps > 0 ? lneps + mx : LN_MIN;
    double fc = solve_upper(m, true, target, std::sqrt(m > 0 ? m : 1.0));
    *flo = -fc;
    *fhi = fc;
  }
}

// ---- band-limited expansion path: Kaiser-Bessel kernel, alias bound, weight tables ------------
// phi(x) = I0(beta sqrt(1 - (2x/w)^2)) / I0(beta) on |x| <= w/2; its transform is
// phi^(xi) = w / I0(beta) * sinh(z)/z, z = sqrt(beta^2 - (pi w xi)^2)  (sin(z)/z beyond the cut-off).
static double kb_hat_shape(double xi, int w, double beta) {   // phi^(xi) * I0(beta) / w
  const double x = M_PI * w * xi;
  const double z2 = beta * beta - x * x;
  const double z = std::sqrt(std::fabs(z2));
  if (z < 1e-8) return 1.0;
  return z2 > 0 ? std::sinh(z) / z : std::sin(z) / z;
}
// max over |xi| <= xi_b of sum_{l != 0} |phi^(xi + l)| / |phi^(xi)|, beta = pi w (1 - xi_b): the
// relative aliasing error of the expansion for a band of half-width xi_b * Nc bins
static double kb_alias_bound(double xi_b, int w) {
  const double beta = M_PI * w * (1.0 - xi_b);
  double worst = 0;
  for (int i = 0; i <= 64; ++i) {
    const double xi = xi_b * i / 64.0;
    double num = 0;
    for (int l = 1; l <= 4; ++l) num += std::fabs(kb_hat_shape(xi + l, w, beta)) + std::fabs(kb_hat_shape(xi - l, w, beta));
    worst = std::max(worst, num / std::fabs(kb_hat_shape(xi, w, beta)));
  }
  return worst;
}
// Buckets of the relative band half-width xi = (band half-width) / Nc and the tap counts tried for
// them.  Beyond xi = 1/4 (coarse grid less than 2x oversampled) the kernel needs 16..20 taps for
// the fp64 tolerance: affordable only where the tap sums run on the tensor cores (ExpandMmaBody),
// `max_taps` says how far the caller may go (16 for the scalar kernels).  The buckets stop at 11/32:
// the coarse spectrum is the band product divided by phi^(xi), and phi^(0) / phi^(xi_b) -- the factor by
// which the rounding noise of the coarse transform can exceed the signal when the energy of the band
// sits at its edge -- is 9 at xi_b = 1/4 (16 taps), 450 at 11/32 (20 taps), 1e4 at 3/8 (24 taps) and
// 1e9 at 7/16 (32 taps; measured on the emulation: 4e-9 error for a Paul scale whose peak is
// off-centre).  450 x 1e-16 stays below the alias tolerance for every signal.
static const double kExpandXi[] = {1.0 / 16, 3.0 / 32, 1.0 / 8, 5.0 / 32, 3.0 / 16, 7.0 / 32, 1.0 / 4,
                                   9.0 / 32, 5.0 / 16, 11.0 / 32};
static const int kExpandBuckets = 10;
static const int kExpandTaps64[] = {10, 12, 14, 16, 20};
static const int kExpandTaps32[] = {6, 8, 10};

// smallest tap count whose alias bound at the bucket of `xi` is <= eps; 0 if none.  *xi_b: bucket.
static int expand_taps(double xi, double eps, bool f32, int max_taps, double *xi_b) {
  // (bucket, taps) -> bound; shared by every context of the process (one per GPU, possibly driven from
  // different host threads)
  static std::map<std::pair<int, int>, double> cache;
  static std::mutex cache_mutex;
  std::lock_guard<std::mutex> cache_lock(cache_mutex);
  int b = -1;
  for (int i = 0; i < kExpandBuckets; ++i)
    if (xi <= kExpandXi[i] * (1 + 1e-12)) { b = i; break; }
  if (b < 0) return 0;
  *xi_b = kExpandXi[b];
  const int *taps = f32 ? kExpandTaps32 : kExpandTaps64;
  const int ntaps = f32 ? 3 : 5;
  for (int i = 0; i < ntaps && taps[i] <= max_taps; ++i) {
    auto key = std::make_pair(b, taps[i]);
    auto it = cache.find(key);
    if (it == cache.end()) it = cache.emplace(key, kb_alias_bound(kExpandXi[b], taps[i])).first;
    if (it->second <= eps) return taps[i];
  }
  return 0;
}

// Dynamic-range check of a candidate (coarse length, taps) beyond xi_b = 1/4: the coarse spectrum is
// the band product divided by phi^(xi); the rounding noise of the coarse transform, relative to the
// largest coarse component, comes back multiplied by up to phi^(0).  Returns
// max_k |psi^(k)| / max|psi^| * phi^(0) / phi^(xi_k) over the band: ~1 when the response peaks at the
// band centre (Morlet, DOG), large when it peaks near an edge (Paul: one-sided band, peak at f = m).
static double expand_gain(const Fam &fam, double s, long long klo, long long khi, long long kc, int log2Nc,
                          int w, double beta) {
  const double Nc = (double)(1ll << log2Nc);
  double peak_amp = 0, worst = 0;
  const double at_centre = beta / std::sinh(beta);
  for (int pass = 0; pass < 2; ++pass)
    for (int i = 0; i <= 256; ++i) {
      const long long k = klo + (long long)std::llround((double)(khi - klo) * i / 256.0);
      const double amp = std::fabs(amp_eval(fam, s, (int)k));
      const double x = M_PI * w * ((double)(k - kc) / Nc);
      const double z = std::sqrt(std::max(beta * beta - x * x, 1e-30));
      const double inv_phi = z / std::sinh(z);          // 1 / phi^ up to a constant
      if (pass == 0) {
        if (amp > peak_amp) peak_amp = amp;
      } else if (peak_amp > 0) {
        worst = std::max(worst, (amp / peak_amp) * (inv_phi / at_centre));
      }
    }
  return worst;
}

// weight table of one class: h[t][rho] = phi(rho / R - (t - (w/2 - 1))), t < w, rho < R (doubles,
// appended to the context's host mirror; uploaded by upload_descs when it grew)
static long long expand_weights(cwtb_ctx *c, std::vector<double> &host, int log2R, int w, double beta) {
  const std::array<long long, 3> key{log2R, w, (long long)std::llround(beta * 1e6)};
  auto it = c->wtab_index.find(key);
  if (it != c->wtab_index.end()) return it->second;
  const long long off = (long long)host.size();
  const int R = 1 << log2R;
  host.resize(host.size() + (size_t)w * R);
  const double i0b = std::cyl_bessel_i(0.0, beta);
  for (int t = 0; t < w; ++t)
    for (int rho = 0; rho < R; ++rho) {
      const double x = (double)rho / R - (double)(t - (w / 2 - 1));
      const double a = 1.0 - (2.0 * x / w) * (2.0 * x / w);
      host[off + (size_t)t * R + rho] = a >= 0 ? std::cyl_bessel_i(0.0, beta * std::sqrt(a)) / i0b : 0.0;
    }
  c->wtab_index.emplace(key, off);
  return off;
}

static int build_job(cwtb_ctx *c, Job &job, long long n0, double dt, const double *scales, int S,
                     int family, double param, int precision, bool have_table, int nbatch = 1) {
  if (n0 < 1 || S < 1 || !(dt > 0)) return fail(c, CWTB_ERR_ARG, "bad n0 / n_scales / dt");
  if (family < 0 || family > 3) return fail(c, CWTB_ERR_ARG, "unknown wavelet family");
  if (family == CWTB_TABLE && !have_table) return fail(c, CWTB_ERR_ARG, "CWTB_TABLE needs a table");
  if ((family == CWTB_PAUL || family == CWTB_DOG) && (param != std::floor(param) || param < 1 || param > 64))
    return fail(c, CWTB_ERR_ARG, "Paul/DOG order must be an integer in [1, 64]");
  if (n0 > (1ll << 28)) return fail(c, CWTB_ERR_UNSUPPORTED, "signal longer than 2^28");
  job = Job();
  // expansion weight tables are cached across calls; start over if many transform geometries
  // have piled up more than 256 MiB of them (offsets are per job, assigned below)
  if (c->wtab_host.size() > ((size_t)32 << 20)) {
    c->wtab_host.clear();
    c->wtab_index.clear();
    c->wtab_uploaded = 0;
  }
  job.precision = precision;
  job.n0 = n0;
  job.log2N = ilog2((unsigned long long)n0);   // pycwt/helpers.py:27-30
  job.N = 1u << job.log2N;
  if (!c->pad_pow2 && (n0 & (n0 - 1)) != 0) {
    // un-padded mode (helpers.py:15-19): transform length = n0; a power-of-two n0 is the
    // padded case anyway
    if (precision != CWTB_F64) return fail(c, CWTB_ERR_UNSUPPORTED, "un-padded transforms run in fp64");
    if (nbatch != 1) return fail(c, CWTB_ERR_UNSUPPORTED, "batched transforms need the padded mode");
    if (n0 > (1ll << 24)) return fail(c, CWTB_ERR_UNSUPPORTED, "un-padded transform longer than 2^24");
    job.exact = true;
    job.N = (unsigned)n0;
  }
  job.S = S;
  job.nbatch = nbatch;
  job.dt = dt;
  const unsigned N = job.N;
  Fam &fam = job.fam;
  fam.family = family;
  fam.m = (int)param;
  fam.f0 = param;
  fam.unit = 0;
  fam.dw = 1.0 / ((double)N * dt);
  fam.table = nullptr;
  fam.tpitch = N;
  double fconst = 1.0;
  if (family == CWTB_MORLET) fconst = std::pow(M_PI, -0.25);
  else if (family == CWTB_PAUL) {
    int m = (int)param;
    double fact = 1;
    for (int i = 2; i < 2 * m; ++i) fact *= i;  // prod(range(2, 2m)) = (2m-1)!
    fconst = std::pow(2.0, m) / std::sqrt(m * fact);
  } else if (family == CWTB_DOG) {
    int m = (int)param;
    fconst = 1.0 / std::sqrt(std::tgamma(m + 0.5));
    // conj(-(1j**m)):  m%4: 0 -> -1, 1 -> +i, 2 -> +1, 3 -> -i
    static const int unit_of[4] = {2, 1, 0, 3};
    fam.unit = unit_of[m & 3];
  }
  // ftfreqs[1]; for Np == 2 numpy's fftfreq(2)[1] is -0.5/dt, so the reference's
  // normalisation sqrt(s*w1*Np) is NaN there -- reproduced.
  const double w1 = 6.283185307179586 * ((N == 2 ? -1.0 : 1.0) * fam.dw);
  double flo = 0, fhi = 0;
  bool pos_only = false;
  // eps = 0 (exact mode) applies to both engines
  const double beps = (precision == CWTB_F32 && c->band_eps > 0) ? std::max(c->band_eps, c->band_eps32) : c->band_eps;
  if (family != CWTB_TABLE) family_band(family, param, beps, &flo, &fhi, &pos_only);

  std::vector<ScaleDesc> ds(S);
  job.plan_log2K.assign(S, 0);
  job.scales.assign(scales, scales + S);
  const long long half = (long long)N / 2;
  for (int j = 0; j < S; ++j) {
    ScaleDesc &d = ds[j];
    const double s = scales[j];
    d.s = s;
    d.row = j;
    d.trow = j;
    d.chan = 0;
    d.pad_ = 0;
    d.boff = 0;
    const double norm = std::sqrt(s * w1 * (double)N);  // wavelet.py:103
    d.amp = (family == CWTB_TABLE ? 1.0 : norm * fconst) / (double)N;
    long long klo = -half, khi = ((long long)N - 1) / 2;   // numpy fftfreq's signed bins, any N
    if (family != CWTB_TABLE && s > 0 && std::isfinite(s)) {
      const double cc = (double)N * dt / (6.283185307179586 * s);
      double a = std::ceil(flo * cc) - 1, b = std::floor(fhi * cc) + 1;
      if (a > (double)klo) klo = (long long)a;
      if (b < (double)khi) khi = (long long)b;
      if (pos_only && klo < 1) klo = 1;
    }
    if (N == 1) { klo = 0; khi = 0; }
    if (khi < klo) { klo = 1; khi = 0; }  // empty band: every B is zero
    d.k_lo = (int)klo;
    d.k_hi = (int)khi;
    // window [lo, lo + K') must contain k = 0 (see DESIGN.md "pruned transform")
    long long lo = std::min<long long>(klo, 0), hi = std::max<long long>(khi, 0);
    if (khi < klo) { lo = 0; hi = 0; }
    int lk = std::max(5, ilog2((unsigned long long)(hi - lo + 1)));
    if (lk > c->direct_max_log2) {  // two-kernel path: negative part must be a multiple of K2
      lo = -((-lo + K2C - 1) / K2C) * K2C;
      lk = std::max(c->direct_max_log2 + 1, ilog2((unsigned long long)(hi - lo + 1)));
    }
    if (lk > 20) lk = job.log2N;   // pruned lengths above 2^20 are not built: treat as dense
    const bool band_limited = lk < job.log2N;   // (before the promotion below: such a scale may still expand)
    // a pruned length of 2^18 or more within `dense_margin` octaves of the full one saves nothing
    // over the dense kernel pair (first kernels of 256 / 512 points cost what the 1024-point dense
    // one does once the band-product launch is counted): treat as dense (CWTB_DENSE_MARGIN)
    if (lk >= 18 && lk < job.log2N && job.log2N - lk <= c->dense_margin && job.log2N <= 20) lk = job.log2N;
    if (lk >= job.log2N) {  // dense
      lk = job.log2N;
      d.rsplit = (int)half;
      if (N == 1) d.rsplit = 1;
    } else {
      d.rsplit = (int)((1ll << lk) + lo);  // lo <= 0
    }
    d.log2K = lk;
    job.plan_log2K[j] = job.exact ? -1 : ((N < 32) ? 0 : lk);
    // ---- band-limited expansion instead of the pruned transforms (kernels.cuh: ExpandBody) ----
    d.ip_log2Nc = 0; d.ip_kc = 0; d.ip_w = 0; d.ip_pad_ = 0; d.ip_coff = 0; d.ip_woff = 0;
    d.ip_beta = 0; d.ip_dc = 0;
    const double xeps = precision == CWTB_F64 ? c->expand_eps : c->expand_eps32;
    if (xeps > 0 && !job.exact && family != CWTB_TABLE && khi >= klo && job.log2N >= 9 && band_limited) {
      const long long kc = (klo + khi) / 2 - (((klo + khi) % 2 != 0 && (klo + khi) < 0) ? 1 : 0);   // floor
      const long long hw = std::max(khi - kc, kc - klo);
      // the tensor-core kernel (fp64, Np >= 4096, every row expanding by 8 or more) makes 20 taps
      // affordable: coarse grids down to 32/11 of the band half-width instead of 4x
#ifdef CWTB_HOST_EMU
      const bool mma = false;
      const int max_taps = precision == CWTB_F64 ? 20 : 10;   // the emulated scalar kernel has every tap count
#else
      const bool mma = precision == CWTB_F64 && c->expand_mma && job.log2N >= 12;
      const int max_taps = mma ? 20 : (precision == CWTB_F64 ? 16 : 10);
#endif
      const long long need = max_taps > 16 ? (32 * hw + 10) / 11 : 4 * hw;
      int lmin = std::max(6, ilog2((unsigned long long)std::max<long long>(need, 1)));
      lmin = std::max(lmin, job.log2N - 14);          // weight tables of at most 2^14 phases
      double best = 1e300;
      // smallest expansion factor: 8.  Both kernels also run R = 4 (CWTB_EXPAND_MIN_R=2), but the coarse
      // transform of Np/4 points is a two-kernel one itself: measured no gain (config 2 1.480 -> 1.496 ms,
      // xwt 1.00 -> 1.18 ms; with the coarse transforms fanned out over streams 1.477 -> 1.466 ms, xwt
      // unchanged, wct +0.7 %: profiles/r2/sweep_t_r4.txt)
      const int min_log2R = c->expand_min_log2R;
      for (int l = lmin; l <= lmin + 2 && job.log2N - l >= min_log2R; ++l) {
        double xi_b = 0;
        int w = expand_taps((double)hw / (double)(1ll << l), xeps, precision != CWTB_F64, max_taps, &xi_b);
        if (!w) continue;
        if (mma) w = (w + 3) / 4 * 4;   // the tensor-core kernel pads to DMMA steps of four taps anyway: 10 -> 12 and
                                        // 14 -> 16 cost nothing, lower the alias error and merge two launches
        if (xi_b > 0.25 && expand_gain(fam, s, klo, khi, kc, l, w, M_PI * w * (1.0 - xi_b)) > 64.0) continue;
        // cost model (us at Np = 2^20): the expansion kernel + the coarse transform.  Scalar kernel: its
        // fp64 work; tensor-core kernel: the W store until the DMMA steps of four taps exceed it
        // (measured, profiles/r2/sweep_r.txt: 2.72 us with three DMMA steps of four taps, 3.33 with four, 4.1 with five)
        const int ksteps = job.log2N - l == 2 ? (w + 4) / 4 : (w + 3) / 4;   // R = 4 needs one more tap column
        const double xcost = mma ? std::max(2.72, 0.83 * ksteps) : 0.06 * (2 * w + 8);
        const double cost = xcost + (mma ? 18.0 : 12.0) * (double)(1ll << l) / (double)N;
        if (cost < best) {
          best = cost;
          d.ip_log2Nc = l; d.ip_kc = (int)kc; d.ip_w = w;
          d.ip_beta = M_PI * w * (1.0 - xi_b);
          d.ip_dc = std::cyl_bessel_i(0.0, d.ip_beta) / w;
        }
      }
      if (d.ip_log2Nc) {
        d.ip_woff = expand_weights(c, c->wtab_host, job.log2N - d.ip_log2Nc, d.ip_w, d.ip_beta);
        job.plan_log2K[j] = -d.ip_log2Nc;
      }
    }
  }
  // one descriptor per (channel, scale) row; rows of channel ch are ch*S .. ch*S+S-1
  if (nbatch > 1) {
    ds.resize((size_t)S * nbatch);
    for (int ch = 1; ch < nbatch; ++ch)
      for (int j = 0; j < S; ++j) {
        ScaleDesc d = ds[j];
        d.chan = ch;
        d.row = ch * S + j;
        ds[(size_t)ch * S + j] = d;
      }
  }
  const int R = S * nbatch;
  // sort by class (descending K': small scales first), stable
  std::vector<int> order(R);
  for (int j = 0; j < R; ++j) order[j] = j;
  // exact classes first (two-kernel, then single-kernel: descending K'), expansion classes last
  // (descending coarse length, then taps / weight table)
  auto sort_key = [&](const ScaleDesc &d) -> long long {
    if (!d.ip_log2Nc) return (1ll << 40) + d.log2K;
    return ((long long)(64 - d.ip_w) << 32) + ((long long)d.ip_log2Nc << 24) - (d.ip_woff & 0xffffff);
  };
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return sort_key(ds[a]) > sort_key(ds[b]); });
  job.descs.resize(R);
  size_t boff = 0, coff = 0;
  for (int i = 0; i < R; ++i) {
    job.descs[i] = ds[order[i]];
    ScaleDesc &d = job.descs[i];
    bool same = !job.classes.empty();
    if (same) {
      const ClassRun &b = job.classes.back();
      same = d.ip_log2Nc ? (b.expand && b.log2Nc == d.ip_log2Nc && b.taps == d.ip_w && b.woff == d.ip_woff)
                         : (!b.expand && b.log2K == d.log2K);
    }
    if (!same) {
      ClassRun cl{d.log2K, i, 0};
      if (d.ip_log2Nc) { cl.expand = 1; cl.log2Nc = d.ip_log2Nc; cl.taps = d.ip_w; cl.woff = d.ip_woff; }
      job.classes.push_back(cl);
    }
    job.classes.back().count++;
    if (d.ip_log2Nc) {
      d.ip_coff = (long long)coff;
      coff += (size_t)1 << d.ip_log2Nc;
    } else if (d.log2K <= 10 || (d.log2K <= c->direct_max_log2 && d.log2K < job.log2N)) {  // single-kernel scale
      d.boff = (long long)boff;
      boff += (size_t)1 << d.log2K;
    }
  }
  job.b_single = boff;
  job.coarse_elems = coff;
  job.valid = true;
  return 0;
}

// ======================================================================================
// execution
// ======================================================================================
template <typename T> struct Tw;
template <> struct Tw<double> { static const double2 *get(cwtb_ctx *c) { return c->tw64; } };
template <> struct Tw<float> { static const float2 *get(cwtb_ctx *c) { return c->tw32; } };

// batched FFT over matrix rows, any power-of-two n >= 2; in/out on device.
// real_in: input rows are T (zero-padded from n_in to n); else cx<T>.
template <typename T, int SIGN>
static int fft_rows(cwtb_ctx *c, const void *in, int real_in, long long in_pitch, long long n_in,
                    cx<T> *out, long long out_pitch, unsigned n, int nrows, long long nout = -1,
                    const double *grow = nullptr, double post = 1.0);

template <typename T, int SIGN, int K>
static int fft_rows_small(cwtb_ctx *c, const RowsArgs<T> &a) {
  constexpr int P = Lay<T, K>::P;
  return launch<RowsBody<T, K, SIGN>>(c, (a.nrows + P - 1) / P, 1, a);
}

template <typename T, int SIGN, int K1, int MODE>
static int launch_passA(cwtb_ctx *c, const PassAArgs<T> &a, int ny) {
  using B = PassABody<T, K1, MODE, SIGN>;
  // a tile covers T2 consecutive r2 of one output row: a shorter row would launch no block at all
  if (a.K2 % B::T2 != 0) return fail(c, CWTB_ERR_STATE, "first kernel: row length not a multiple of its tile");
  const unsigned M = a.N / ((unsigned)K1 * a.K2);
  return launch<B>(c, M * (a.K2 / B::T2), ny, a);
}

template <typename T, int SIGN, int MODE>
static int dispatch_passA(cwtb_ctx *c, int log2K1, const PassAArgs<T> &a, int ny) {
  switch (log2K1) {
    case 1: return launch_passA<T, SIGN, 2, MODE>(c, a, ny);
    case 2: return launch_passA<T, SIGN, 4, MODE>(c, a, ny);
    case 3: return launch_passA<T, SIGN, 8, MODE>(c, a, ny);
    case 4: return launch_passA<T, SIGN, 16, MODE>(c, a, ny);
    case 5: return launch_passA<T, SIGN, 32, MODE>(c, a, ny);
    case 6: return launch_passA<T, SIGN, 64, MODE>(c, a, ny);
    case 7: return launch_passA<T, SIGN, 128, MODE>(c, a, ny);
    case 8: return launch_passA<T, SIGN, 256, MODE>(c, a, ny);
    case 9: return launch_passA<T, SIGN, 512, MODE>(c, a, ny);
    case 10: return launch_passA<T, SIGN, 1024, MODE>(c, a, ny);
  }
  return fail(c, CWTB_ERR_UNSUPPORTED, "transform longer than 2^20 per row is not supported yet");
}

// Rows of length n (1024 < n <= 2^20) through PassA<REAL|CPLX> + PassB, in chunks that fit the
// Z buffer.  Input row g becomes sub-transform g % ileave of output row out_row0 + g / ileave
// (ileave = 1: plain rows).  Output rows are renamed through descs[first + outer].row if given.
template <typename T, int SIGN>
static int two_kernel_rows(cwtb_ctx *c, const void *in, int real_in, long long in_pitch, long long n_in,
                           cx<T> *out, long long out_pitch, unsigned n, int nrows, long long nout,
                           const double *grow, double post, int ileave, const ScaleDesc *descs, int first,
                           int out_row0, int epi) {
  const int l2 = ilog2(n);
  NTab nt;
  int e = get_ntab(c, n, l2, &nt);
  if (e) return e;
  // rows per chunk: the intermediate of a chunk (rows_chunk_bytes, default 64 MiB) stays in L2
  // between the two kernels
  const int chunk = std::max(1, std::min(nrows, (int)std::max<size_t>(1, c->rows_chunk_bytes / ((size_t)n * sizeof(cx<T>)))));
  Buf &Zt = c->ztmp ? *c->ztmp : c->Z;
  if ((e = ensure(c, Zt, (size_t)chunk * n * sizeof(cx<T>)))) return e;
  for (int r0 = 0; r0 < nrows; r0 += chunk) {
    const int nr = std::min(chunk, nrows - r0);
    PassAArgs<T> a{};
    a.in = in; a.Z = (cx<T> *)Zt.p; a.tw = Tw<T>::get(c); a.nt = nt;
    a.in_pitch = in_pitch; a.n_in = n_in; a.N = n; a.first = 0; a.zmod = 1 << 30; a.K2 = K2C;
    a.row0 = (ileave > 1 ? 0 : out_row0) + r0;   // interleaved input rows are numbered from 0
    a.pf_dist = c->pf_rows_a;
    e = real_in ? dispatch_passA<T, SIGN, MODE_REAL>(c, l2 - 10, a, nr)
                : dispatch_passA<T, SIGN, MODE_CPLX>(c, l2 - 10, a, nr);
    if (e) return e;
    PassBArgs<T> b{};
    b.Z = (const cx<T> *)Zt.p; b.out = out; b.tw = Tw<T>::get(c); b.descs = descs;
    b.pitch = out_pitch; b.nout = nout; b.N = n; b.first = first;
    b.epi = grow ? EPI_GAUSS : epi; b.grow = grow; b.post = post; b.zmod = 1 << 30;
    b.pf_dist = c->pf_rows_b; b.ny = nr; b.ileave = ileave; b.rev = c->passb_rev;
    if (ileave > 1) { b.row0 = out_row0; b.by0 = r0; } else { b.row0 = out_row0 + r0; b.by0 = 0; }
    e = launch<PassBBody<T, SIGN>>(c, (n / K2C + Lay<T, K2C>::P - 1) / Lay<T, K2C>::P, nr, b);
    if (e) return e;
  }
  return 0;
}

template <typename T, int SIGN>
static int fft_rows(cwtb_ctx *c, const void *in, int real_in, long long in_pitch, long long n_in,
                    cx<T> *out, long long out_pitch, unsigned n, int nrows, long long nout,
                    const double *grow, double post) {
  const int l2 = ilog2(n);
  if (nout < 0) nout = n;
  if (n <= 1024) {
    RowsArgs<T> a;
    a.in = in; a.out = out; a.tw = Tw<T>::get(c); a.grow = grow;
    a.in_pitch = in_pitch; a.out_pitch = out_pitch; a.n_in = n_in; a.nout = nout;
    a.post = post; a.nrows = nrows; a.real_in = real_in; a.n = (int)n;
    switch (l2) {
      case 1: return fft_rows_small<T, SIGN, 2>(c, a);
      case 2: return fft_rows_small<T, SIGN, 4>(c, a);
      case 3: return fft_rows_small<T, SIGN, 8>(c, a);
      case 4: return fft_rows_small<T, SIGN, 16>(c, a);
      case 5: return fft_rows_small<T, SIGN, 32>(c, a);
      case 6: return fft_rows_small<T, SIGN, 64>(c, a);
      case 7: return fft_rows_small<T, SIGN, 128>(c, a);
      case 8: return fft_rows_small<T, SIGN, 256>(c, a);
      case 9: return fft_rows_small<T, SIGN, 512>(c, a);
      case 10: return fft_rows_small<T, SIGN, 1024>(c, a);
    }
    return fail(c, CWTB_ERR_ARG, "fft_rows: bad length");
  }
  if (n <= (1u << 20))
    return two_kernel_rows<T, SIGN>(c, in, real_in, in_pitch, n_in, out, out_pitch, n, nrows, nout, grow, post,
                                    1, nullptr, 0, 0, EPI_STORE);
  // ---- Np > 2^20: three levels.  A pre-pass (PassA with K1 = K0 = n / 2^20 and rows of 2^20)
  // turns each row into K0 twiddled sequences y_c[j]; output bin K0*q + c is bin q of the
  // 2^20-point transform of y_c, computed by the two-kernel path with interleaved stores.
  const int l0 = l2 - 20;
  const unsigned K0 = 1u << l0, Nsub = 1u << 20;
  NTab nt;
  int e = get_ntab(c, n, l2, &nt);
  if (e) return e;
  const int chunk = std::max(1, std::min(nrows, (int)std::max<size_t>(1, ((size_t)512 << 20) / ((size_t)n * sizeof(cx<T>)))));
  if ((e = ensure(c, c->Y, (size_t)chunk * n * sizeof(cx<T>)))) return e;
  for (int r0 = 0; r0 < nrows; r0 += chunk) {
    const int nr = std::min(chunk, nrows - r0);
    PassAArgs<T> a{};
    a.in = in; a.Z = (cx<T> *)c->Y.p; a.tw = Tw<T>::get(c); a.nt = nt;
    a.in_pitch = in_pitch; a.n_in = n_in; a.N = n; a.first = 0; a.row0 = r0; a.zmod = 1 << 30; a.K2 = Nsub;
    e = real_in ? dispatch_passA<T, SIGN, MODE_REAL>(c, l0, a, nr)
                : dispatch_passA<T, SIGN, MODE_CPLX>(c, l0, a, nr);
    if (e) return e;
    if ((e = two_kernel_rows<T, SIGN>(c, c->Y.p, 0, Nsub, Nsub, out, out_pitch, Nsub, nr * (int)K0, nout, grow, post,
                                      (int)K0, nullptr, 0, r0, EPI_STORE)))
      return e;
  }
  return 0;
}


// ======================================================================================
// un-padded mode (pycwt/helpers.py:15-19, the reference's pyfftw branch): transforms at the
// signal's own length n through Bluestein's chirp-z algorithm on the power-of-two kernels.
// A compatibility path: ~2 transforms of length >= 2n per scale and no band pruning.
// ======================================================================================
static int get_blue(cwtb_ctx *c, unsigned n, const BluePlan **out) {
  auto it = c->blue.find(n);
  if (it == c->blue.end()) {
    // keep at most a few lengths resident
    if (c->blue.size() >= 4) {
      for (auto &kv : c->blue) { rt_free(kv.second.wm); rt_free(kv.second.bf[0]); rt_free(kv.second.bf[1]); }
      c->blue.clear();
    }
    BluePlan pl;
    pl.n = n;
    pl.L = 1u << ilog2(2ull * n - 1);
    RT(rt_malloc((void **)&pl.wm, sizeof(double2) * n));
    BlueChirpArgs ca{pl.wm, n};
    int e = launch<BlueChirpBody>(c, (n + NT - 1) / NT, 1, ca);
    if (e) return e;
    if ((e = ensure(c, c->blueX, (size_t)pl.L * sizeof(double2)))) return e;
    for (int si = 0; si < 2; ++si) {
      RT(rt_malloc((void **)&pl.bf[si], sizeof(double2) * pl.L));
      BlueFilterArgs fa{pl.wm, (double2 *)c->blueX.p, n, pl.L, si ? +1 : -1};
      if ((e = launch<BlueFilterBody>(c, (pl.L + NT - 1) / NT, 1, fa))) return e;
      if ((e = fft_rows<double, -1>(c, c->blueX.p, 0, pl.L, pl.L, pl.bf[si], pl.L, pl.L, 1, -1, nullptr, 1.0))) return e;
    }
    it = c->blue.emplace(n, pl).first;
  }
  *out = &it->second;
  return 0;
}

// rows of the convolution buffers a chunk may use (two buffers of L complex per row)
static int blue_chunk_rows(unsigned L, int nrows) {
  const size_t per_row = (size_t)L * sizeof(double2);
  return (int)std::max<size_t>(1, std::min<size_t>((size_t)nrows, ((size_t)1 << 30) / per_row));
}

// convolution core: blueA rows (pitch n) already hold a = x * w_s; result rows y in blueY
static int blue_convolve(cwtb_ctx *c, const BluePlan &pl, int nr, int sign) {
  int e;
  if ((e = fft_rows<double, -1>(c, c->blueA.p, 0, pl.n, pl.n, (double2 *)c->blueX.p, pl.L, pl.L, nr, -1, nullptr, 1.0)))
    return e;
  BlueMulArgs ma{(double2 *)c->blueX.p, pl.bf[sign > 0 ? 1 : 0], pl.L};
  if ((e = launch<BlueMulBody>(c, (pl.L + NT - 1) / NT, nr, ma))) return e;
  return fft_rows<double, +1>(c, c->blueX.p, 0, pl.L, pl.L, (double2 *)c->blueY.p, pl.L, pl.L, nr, -1, nullptr, 1.0);
}

// out[r][k] = scale * sum_j in[r][j] e^{sign 2 pi i jk/n}, k < nout, for rows of any length n >= 2
static int blue_rows(cwtb_ctx *c, const void *in, int real_in, long long in_pitch, double2 *out,
                     long long out_pitch, unsigned n, int nrows, int sign, double scale, long long nout) {
  const BluePlan *pl;
  int e = get_blue(c, n, &pl);
  if (e) return e;
  const int chunk = blue_chunk_rows(pl->L, nrows);
  if ((e = ensure(c, c->blueA, (size_t)chunk * n * sizeof(double2)))) return e;
  if ((e = ensure(c, c->blueX, (size_t)chunk * pl->L * sizeof(double2)))) return e;
  if ((e = ensure(c, c->blueY, (size_t)chunk * pl->L * sizeof(double2)))) return e;
  const size_t isz = real_in ? sizeof(double) : sizeof(double2);
  for (int r0 = 0; r0 < nrows; r0 += chunk) {
    const int nr = std::min(chunk, nrows - r0);
    BluePreArgs pa{(const char *)in + (size_t)r0 * in_pitch * isz, (double2 *)c->blueA.p, pl->wm,
                   in_pitch, (long long)n, n, real_in, sign};
    if ((e = launch<BluePreBody>(c, (n + NT - 1) / NT, nr, pa))) return e;
    if ((e = blue_convolve(c, *pl, nr, sign))) return e;
    BluePostArgs po{(const double2 *)c->blueY.p, out, pl->wm, nullptr, out_pitch, nout,
                    scale / (double)pl->L, pl->L, 0, r0, sign, EPI_STORE};
    if ((e = launch<BluePostBody>(c, (unsigned)((nout + NT - 1) / NT), nr, po))) return e;
  }
  return 0;
}

// every kernel of one un-padded transform (fp64): spectrum at length n0, then for chunks of scales
// product + inverse transform at length n0
static int run_job_exact(cwtb_ctx *c, const Job &job, const double *dsig, double2 *Wout, int epi) {
  const unsigned n = job.N;
  const int S = job.S;
  int e;
  if (job.nbatch != 1) return fail(c, CWTB_ERR_UNSUPPORTED, "batched transforms need the padded mode");
  if ((e = ensure(c, c->spec, (size_t)n * sizeof(double2)))) return e;
  if (!Wout) {
    if ((e = ensure(c, c->W, (size_t)S * job.n0 * sizeof(double2)))) return e;
    Wout = (double2 *)c->W.p;
  }
  if ((e = blue_rows(c, dsig, 1, n, (double2 *)c->spec.p, n, n, 1, -1, 1.0, n))) return e;
  const BluePlan *pl;
  if ((e = get_blue(c, n, &pl))) return e;
  Fam fam = job.fam;
  if (fam.family == CWTB_TABLE) fam.table = (const double2 *)c->table.p;
  const int chunk = blue_chunk_rows(pl->L, S);
  if ((e = ensure(c, c->blueA, (size_t)chunk * n * sizeof(double2)))) return e;
  if ((e = ensure(c, c->blueX, (size_t)chunk * pl->L * sizeof(double2)))) return e;
  if ((e = ensure(c, c->blueY, (size_t)chunk * pl->L * sizeof(double2)))) return e;
  const ScaleDesc *ddesc = (const ScaleDesc *)c->descs.p;
  for (int r0 = 0; r0 < S; r0 += chunk) {
    const int nr = std::min(chunk, S - r0);
    BlueProdArgs pa{ddesc, (const double2 *)c->spec.p, (double2 *)c->blueA.p, pl->wm, fam, (long long)n, n, r0};
    if ((e = launch<BlueProdBody>(c, (n + NT - 1) / NT, nr, pa))) return e;
    if ((e = blue_convolve(c, *pl, nr, +1))) return e;
    // descriptor amplitudes already carry the 1/n of the inverse transform
    BluePostArgs po{(const double2 *)c->blueY.p, Wout, pl->wm, ddesc, job.n0, job.n0,
                    1.0 / (double)pl->L, pl->L, r0, 0, +1, epi};
    if ((e = launch<BluePostBody>(c, (unsigned)((job.n0 + NT - 1) / NT), nr, po))) return e;
  }
  return 0;
}

// ======================================================================================
// fused persistent two-pass kernel: PassA and PassB tiles of every scale of one class run in
// ONE launch.  A global tile queue is consumed in the order
//     A(0) A(1) B(0) A(2) B(1) ... A(n-1) B(n-2) B(n-1)
// (A(s)/B(s) = all tiles of scale s); B(s) waits for the A(s) tiles through a global counter,
// A(s) waits for B(s-ring) before reusing its Z slot.  Z is a ring of `ring` scale buffers
// (ring * 16 MiB at Np = 2^20) that lives in L2, so the intermediate never goes to HBM and
// there are no per-scale launch tails.
// ======================================================================================
template <typename T> struct FusedArgs {
  PassAArgs<T> a;
  PassBArgs<T> b;
  unsigned *ctr;    // [0] queue head, [1 .. n] doneA, [1+n .. 2n] doneB
  int nscales, ring;
  unsigned tilesA, tilesB;
};

// position t of the queue -> (isB, scale, tile)
HD void fused_decode(unsigned t, int n, unsigned TA, unsigned TB, int *isB, int *s, unsigned *tile) {
  if (t < TA) { *isB = 0; *s = 0; *tile = t; return; }
  t -= TA;
  const unsigned per = TA + TB;
  const unsigned blk = t / per, off = t % per;
  if ((int)blk < n - 1) {
    if (off < TA) { *isB = 0; *s = (int)blk + 1; *tile = off; }
    else { *isB = 1; *s = (int)blk; *tile = off - TA; }
  } else {  // tail: B(n-1)
    *isB = 1; *s = n - 1; *tile = t - (unsigned)(n - 1) * per;
  }
}

#ifndef CWTB_HOST_EMU
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
template <typename T, int K1, int MODE>
__global__ void __launch_bounds__(TileCfg<T>::NT, 3) k_fused(const __grid_constant__ FusedArgs<T> f) {
  extern __shared__ __align__(16) unsigned char smraw[];
  __shared__ unsigned s_t;
  using A = PassABody<T, K1, MODE, +1>;
  using B = PassBBody<T, +1>;
  const int n = f.nscales;
  const unsigned total = (unsigned)n * (f.tilesA + f.tilesB);
  unsigned *doneA = f.ctr + 1, *doneB = f.ctr + 1 + n;
  for (;;) {
    __syncthreads();  // previous tile's shared memory is free
    if (threadIdx.x == 0) s_t = atomicAdd(f.ctr, 1u);
    __syncthreads();
    const unsigned t = s_t;
    if (t >= total) break;
    int isB, s;
    unsigned tile;
    fused_decode(t, n, f.tilesA, f.tilesB, &isB, &s, &tile);
    if (threadIdx.x == 0) {
      if (isB) {
        while (ld_acquire_u32(&doneA[s]) < f.tilesA) __nanosleep(100);
      } else if (s >= f.ring) {
        while (ld_acquire_u32(&doneB[s - f.ring]) < f.tilesB) __nanosleep(100);
      }
      asm volatile("fence.proxy.async;" ::: "memory");
    }
    __syncthreads();
    if (isB) run_phases_at<B, 0>(f.b, (int)tile, s, smraw);
    else run_phases_at<A, 0>(f.a, (int)tile, s, smraw);
    __syncthreads();
    if (threadIdx.x == 0)   // release-add, no L1 invalidate (see k_pipe)
      asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(isB ? &doneB[s] : &doneA[s]), "r"(1u) : "memory");
  }
}
#endif

template <typename T, int K1, int MODE>
static int launch_fused(cwtb_ctx *c, const PassAArgs<T> &a, const PassBArgs<T> &b, int nscales) {
  using A = PassABody<T, K1, MODE, +1>;
  using B = PassBBody<T, +1>;
  FusedArgs<T> f;
  f.a = a; f.b = b;
  f.nscales = nscales;
  f.ring = c->ring;
  f.a.zmod = f.b.zmod = c->ring;
  const unsigned M = a.N / ((unsigned)K1 * K2C);
  f.tilesA = M * (K2C / A::T2);
  f.tilesB = (a.N / K2C + Lay<T, K2C>::P - 1) / Lay<T, K2C>::P;
  int e = ensure(c, c->ctr, (size_t)(1 + 2 * nscales) * sizeof(unsigned));
  if (e) return e;
  f.ctr = (unsigned *)c->ctr.p;
  RT(rt_memset(c->ctr.p, 0, (size_t)(1 + 2 * nscales) * sizeof(unsigned), c->stream));
#ifdef CWTB_HOST_EMU
  std::vector<unsigned char> sm(std::max(A::SMEM, B::SMEM) + 64);
  const unsigned total = (unsigned)nscales * (f.tilesA + f.tilesB);
  for (unsigned t = 0; t < total; ++t) {
    int isB, s;
    unsigned tile;
    fused_decode(t, nscales, f.tilesA, f.tilesB, &isB, &s, &tile);
    if (isB) emu_phases<B, 0>(f.b, (int)tile, s, sm.data());
    else emu_phases<A, 0>(f.a, (int)tile, s, sm.data());
  }
  c->launches++;
  return 0;
#else
  const size_t smem = std::max(A::SMEM, B::SMEM);
  auto kern = k_fused<T, K1, MODE>;
  const void *fn = (const void *)kern;
  if (!c->configured.count(fn)) {
    RT(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    c->configured.insert(fn);
  }
  int occ = 0;
  RT(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, TileCfg<T>::NT, smem));
  if (occ < 1) return fail(c, CWTB_ERR_CUDA, "fused kernel does not fit on an SM");
  const unsigned total = (unsigned)nscales * (f.tilesA + f.tilesB);
  const unsigned grid = std::min<unsigned>(total, (unsigned)(occ * c->num_sms));
  int ev = -1;
  if (c->profiling) {
    ev = (int)c->prof.size() * 2;
    while ((int)c->prof_events.size() < ev + 2) {
      cudaEvent_t e2;
      RT(cudaEventCreate(&e2));
      c->prof_events.push_back(e2);
    }
    c->prof.push_back({body_name(__PRETTY_FUNCTION__), grid, (unsigned)nscales, ev});
    RT(cudaEventRecord(c->prof_events[ev], c->stream));
  }
  kern<<<grid, TileCfg<T>::NT, smem, c->stream>>>(f);
  RT(cudaGetLastError());
  if (ev >= 0) RT(cudaEventRecord(c->prof_events[ev + 1], c->stream));
  c->launches++;
  return 0;
#endif
}

template <typename T, int MODE>
static int dispatch_fused(cwtb_ctx *c, int log2K1, const PassAArgs<T> &a, const PassBArgs<T> &b, int n) {
  switch (log2K1) {
    case 1: return launch_fused<T, 2, MODE>(c, a, b, n);
    case 2: return launch_fused<T, 4, MODE>(c, a, b, n);
    case 3: return launch_fused<T, 8, MODE>(c, a, b, n);
    case 4: return launch_fused<T, 16, MODE>(c, a, b, n);
    case 5: return launch_fused<T, 32, MODE>(c, a, b, n);
    case 6: return launch_fused<T, 64, MODE>(c, a, b, n);
    case 7: return launch_fused<T, 128, MODE>(c, a, b, n);
    case 8: return launch_fused<T, 256, MODE>(c, a, b, n);
    case 9: return launch_fused<T, 512, MODE>(c, a, b, n);
    case 10: return launch_fused<T, 1024, MODE>(c, a, b, n);
  }
  return fail(c, CWTB_ERR_UNSUPPORTED, "transform longer than 2^20 per row is not supported yet");
}

// ======================================================================================
// Pipelined persistent two-pass kernel (CWTB_FUSED=2): like k_fused, but built so that the
// bookkeeping stays off the critical path.
//   * static schedule: CTA b runs tiles b, b + grid, b + 2 grid, ... of the global order
//         A(0) .. A(ahead-1) | A(ahead) B(0) | A(ahead+1) B(1) | ... | B(n-ahead) .. B(n-1)
//     (no queue atomic); the first kernel runs `ahead` scales in front of the second one, so the
//     tiles a B(s) tile depends on were handed out >= ahead*tilesA positions earlier -- more than
//     the number of resident CTAs for ahead = 2 -- and the dependency wait almost never blocks;
//   * a CTA tests a dependency once per scale (not per tile): counters doneA[s] / doneB[s];
//   * completion is published by the LAST thread of the CTA (fence + relaxed add) while the
//     first warp already issues the next tile's bulk copies.
// Z is a ring of `ring` >= ahead + 2 scale buffers (16 MiB each at Np = 2^20) that stays in L2:
// the second kernel's tile loads hit L2 and the intermediate never reaches HBM.
// ======================================================================================
template <typename T> struct PipeArgs {
  PassAArgs<T> a;
  PassBArgs<T> b;
  unsigned *ctr;    // [0 .. n) doneA, [n .. 2n) doneB
  int nscales, ring, ahead;
  unsigned tilesA, tilesB;
};

HD void pipe_decode(unsigned t, int n, int ahead, unsigned TA, unsigned TB, int *isB, int *s, unsigned *tile) {
  const int na = ahead < n ? ahead : n;
  if (t < (unsigned)na * TA) { *isB = 0; *s = (int)(t / TA); *tile = t % TA; return; }
  t -= (unsigned)na * TA;
  const unsigned per = TA + TB;
  const int nmid = n - na;
  if (t < (unsigned)nmid * per) {
    const unsigned blk = t / per, off = t % per;
    if (off < TA) { *isB = 0; *s = na + (int)blk; *tile = off; }
    else { *isB = 1; *s = (int)blk; *tile = off - TA; }
    return;
  }
  t -= (unsigned)nmid * per;
  *isB = 1; *s = nmid + (int)(t / TB); *tile = t % TB;
}

#ifndef CWTB_HOST_EMU
template <typename T, int K1, int MODE>
__global__ void __launch_bounds__(TileCfg<T>::NT, 3) k_pipe(const __grid_constant__ PipeArgs<T> f) {
  extern __shared__ __align__(16) unsigned char smraw[];
  using A = PassABody<T, K1, MODE, +1>;
  using B = PassBBody<T, +1>;
  const int n = f.nscales;
  const unsigned total = (unsigned)n * (f.tilesA + f.tilesB);
  unsigned *doneA = f.ctr, *doneB = f.ctr + n;
  int okA = -1, okB = -1;    // dependencies already seen complete by this CTA
  for (unsigned t = blockIdx.x; t < total; t += gridDim.x) {
    int isB, s;
    unsigned tile;
    pipe_decode(t, n, f.ahead, f.tilesA, f.tilesB, &isB, &s, &tile);
    const int dep = isB ? s : s - f.ring;          // A(s) reuses the slot of B(s - ring)
    if (dep >= 0 && dep > (isB ? okA : okB)) {
      if (threadIdx.x == 0) {
        const unsigned *flag = isB ? &doneA[dep] : &doneB[dep];
        const unsigned want = isB ? f.tilesA : f.tilesB;
        while (ld_acquire_u32(flag) < want) __nanosleep(64);
        asm volatile("fence.proxy.async;" ::: "memory");
      }
      __syncthreads();
      if (isB) okA = dep; else okB = dep;
    }
    if (isB) run_phases_at<B, 0>(f.b, (int)tile, s, smraw);
    else run_phases_at<A, 0>(f.a, (int)tile, s, smraw);
    __syncthreads();   // shared memory is free again; every store of the tile has been issued
    if (threadIdx.x == blockDim.x - 1) {
      // release-add: orders the tile's stores (made visible to this thread by the barrier) before
      // the count.  NOT __threadfence(): a gpu-scope fence also invalidates the SM's L1
      // (SASS CCTL.IVALL) -- once per tile that evicts the twiddle / root tables of every
      // resident CTA; the release form compiles to MEMBAR.ALL.GPU + REDG only.
      asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(isB ? &doneB[s] : &doneA[s]), "r"(1u) : "memory");
    }
  }
}
#endif

template <typename T, int K1, int MODE>
static int launch_pipe(cwtb_ctx *c, const PassAArgs<T> &a, const PassBArgs<T> &b, int nscales) {
  using A = PassABody<T, K1, MODE, +1>;
  using B = PassBBody<T, +1>;
  PipeArgs<T> f;
  f.a = a; f.b = b;
  f.nscales = nscales;
  f.ring = c->ring;
  f.ahead = std::max(1, std::min(c->pipe_ahead, c->ring - 1));
  f.a.zmod = f.b.zmod = c->ring;
  f.b.rev = 0; f.b.pf_dist = 0; f.a.pf_dist = 0;
  const unsigned M = a.N / ((unsigned)K1 * K2C);
  f.tilesA = M * (K2C / A::T2);
  f.tilesB = (a.N / K2C + Lay<T, K2C>::P - 1) / Lay<T, K2C>::P;
  int e = ensure(c, c->ctr, (size_t)(2 * nscales) * sizeof(unsigned));
  if (e) return e;
  f.ctr = (unsigned *)c->ctr.p;
  RT(rt_memset(c->ctr.p, 0, (size_t)(2 * nscales) * sizeof(unsigned), c->cur));
#ifdef CWTB_HOST_EMU
  std::vector<unsigned char> sm(std::max(A::SMEM, B::SMEM) + 64);
  const unsigned total = (unsigned)nscales * (f.tilesA + f.tilesB);
  std::vector<int> seenA(nscales, 0), seenB(nscales, 0);
  for (unsigned t = 0; t < total; ++t) {
    int isB, s;
    unsigned tile;
    pipe_decode(t, nscales, f.ahead, f.tilesA, f.tilesB, &isB, &s, &tile);
    // the sequential emulation checks the schedule's invariants instead of waiting
    if (isB && seenA[s] != (int)f.tilesA) return fail(c, CWTB_ERR_STATE, "pipe schedule: B before its A tiles");
    if (!isB && s >= f.ring && seenB[s - f.ring] != (int)f.tilesB)
      return fail(c, CWTB_ERR_STATE, "pipe schedule: Z slot reused before its B tiles");
    if (isB) { emu_phases<B, 0>(f.b, (int)tile, s, sm.data()); seenB[s]++; }
    else { emu_phases<A, 0>(f.a, (int)tile, s, sm.data()); seenA[s]++; }
  }
  c->launches++;
  return 0;
#else
  const size_t smem = std::max(A::SMEM, B::SMEM);
  auto kern = k_pipe<T, K1, MODE>;
  const void *fn = (const void *)kern;
  if (!c->configured.count(fn)) {
    RT(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    c->configured.insert(fn);
  }
  int occ = 0;
  RT(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, TileCfg<T>::NT, smem));
  if (occ < 1) return fail(c, CWTB_ERR_CUDA, "pipelined kernel does not fit on an SM");
  const unsigned total = (unsigned)nscales * (f.tilesA + f.tilesB);
  // every CTA must be resident (they wait for one another): at most occ per SM
  const unsigned grid = std::min<unsigned>(total, (unsigned)(occ * c->num_sms));
  int ev = -1;
  if (c->profiling) {
    ev = (int)c->prof.size() * 2;
    while ((int)c->prof_events.size() < ev + 2) {
      cudaEvent_t e2;
      RT(cudaEventCreate(&e2));
      c->prof_events.push_back(e2);
    }
    char nm[64];
    snprintf(nm, sizeof nm, "PipeAB<%s, %d, %d>", sizeof(T) == 8 ? "double" : "float", K1, MODE);
    c->prof.push_back({nm, grid, (unsigned)nscales, ev});
    RT(cudaEventRecord(c->prof_events[ev], c->cur));
  }
  kern<<<grid, TileCfg<T>::NT, smem, c->cur>>>(f);
  RT(cudaGetLastError());
  if (ev >= 0) RT(cudaEventRecord(c->prof_events[ev + 1], c->cur));
  c->launches++;
  return 0;
#endif
}

template <typename T, int MODE>
static int dispatch_pipe(cwtb_ctx *c, int log2K1, const PassAArgs<T> &a, const PassBArgs<T> &b, int n) {
  switch (log2K1) {
    case 4: return launch_pipe<T, 16, MODE>(c, a, b, n);
    case 5: return launch_pipe<T, 32, MODE>(c, a, b, n);
    case 6: return launch_pipe<T, 64, MODE>(c, a, b, n);
    case 7: return launch_pipe<T, 128, MODE>(c, a, b, n);
    case 8: return launch_pipe<T, 256, MODE>(c, a, b, n);
    case 9: return launch_pipe<T, 512, MODE>(c, a, b, n);
    case 10: return launch_pipe<T, 1024, MODE>(c, a, b, n);
  }
  return fail(c, CWTB_ERR_UNSUPPORTED, "pipelined two-pass kernel: unsupported first-pass length");
}

template <typename T, int K>
static int launch_single(cwtb_ctx *c, const SingleArgs<T> &a, int count) {
  constexpr int P = Lay<T, K>::P;
  const unsigned M = a.N / K;
  return launch<SingleBody<T, K>>(c, (M + P - 1) / P, count, a);
}

// rows (scale x channel) per chunk of the two-kernel path: the Z intermediate of a chunk is
// rows * Np elements
static int chunk_rows(const cwtb_ctx *c, unsigned N, size_t elem_bytes) {
  if (c->group > 0) return c->group;
  size_t g = c->group_bytes / ((size_t)N * elem_bytes);
  return (int)std::max<size_t>(1, std::min<size_t>(g, 32768));
}

static bool class_single(const cwtb_ctx *c, const Job &job, const ClassRun &cl) {
  return !cl.expand && (cl.log2K <= 10 || (cl.log2K <= c->direct_max_log2 && cl.log2K < job.log2N));
}
static bool class_two_kernel(const cwtb_ctx *c, const Job &job, const ClassRun &cl) {
  return !cl.expand && !class_single(c, job, cl);
}
// two-kernel class that runs as ONE persistent launch over a ring of Z buffers
static bool class_persistent(const cwtb_ctx *c, const ClassRun &cl) {
  return c->fused == 1 || (c->fused == 2 && cl.log2K >= 14 && cl.log2K <= 20 && cl.count <= 256);
}

// Which band-chunk region / Z buffer / stream a two-kernel class uses: its position among the
// two-kernel classes modulo the number of chains (dense classes included, they only use Z).
static int job_chain_region(const cwtb_ctx *c, const Job &job, const ClassRun &cl) {
  int idx = 0;
  for (const ClassRun &o : job.classes) {
    if (&o == &cl) break;
    if (class_two_kernel(c, job, o)) ++idx;
  }
  return idx % std::max(1, c->n_chains);
}

// elements of one band-chunk region: the largest chunk of band products of any two-kernel class
static size_t band_chunk_elems(const cwtb_ctx *c, const Job &job, int G) {
  size_t bchunk = 0;
  for (const ClassRun &cl : job.classes)
    if (class_two_kernel(c, job, cl) && cl.log2K < job.log2N)
      bchunk = std::max(bchunk, (size_t)(class_persistent(c, cl) ? cl.count : std::min(G, cl.count)) << cl.log2K);
  return bchunk;
}

template <typename T, int TAPS>
static int launch_expand_t(cwtb_ctx *c, const ExpandArgs<T> &a, int rows, int min_log2Nc) {
  using B = ExpandBody<T, TAPS>;
  // tiles per row: (R / RB) * ceil(Nc / MT) with RB = min(R, NT), MT = (NT / RB) * L -- equal to
  // N / (NT * L) for every coarse length with Nc >= MT; rows with a shorter coarse grid use the
  // first tiles of the launch only
  const unsigned gx = std::max<unsigned>(1, a.N / (unsigned)(B::NT * B::L));
#ifndef CWTB_HOST_EMU
  // fp64: tap sums on the tensor cores (kernels.cuh: ExpandMmaBody) whenever every row expands by 8 or more
  if constexpr (std::is_same<T, double>::value) {
    static_assert(ExpandMmaBody<TAPS>::OUT_PER_CTA == 4096, "the planner assumes the tensor-core kernel from Np = 2^12");
    if (c->expand_mma && a.N >= (unsigned)ExpandMmaBody<TAPS>::OUT_PER_CTA) {
      // tiles per row: N / (32 L); a row whose coarse grid is shorter than one run (Nc < L, R > 32) needs
      // one tile per 32 phases instead
      const unsigned gm = a.N / (32u * std::min<unsigned>(ExpandMmaBody<TAPS>::L, 1u << min_log2Nc));
      if (a.epi == EPI_MULCONJ) return launch<ExpandMmaBody<TAPS, EPI_MULCONJ>>(c, gm, rows, a);
      return launch<ExpandMmaBody<TAPS>>(c, gm, rows, a);
    }
  }
#endif
#ifndef CWTB_HOST_EMU
  if constexpr (TAPS > 16) {
    return fail(c, CWTB_ERR_STATE, "expansion: tap counts above 16 exist on the tensor-core kernel only");
  } else
#endif
  {
    if (a.epi == EPI_MULCONJ) return launch<ExpandBody<T, TAPS, EPI_MULCONJ>>(c, gx, rows, a);
    return launch<B>(c, gx, rows, a);
  }
}
template <typename T>
static int launch_expand(cwtb_ctx *c, int taps, const ExpandArgs<T> &a, int rows, int min_log2Nc) {
  if constexpr (std::is_same<T, double>::value) {
    switch (taps) {
      case 10: return launch_expand_t<T, 10>(c, a, rows, min_log2Nc);
      case 12: return launch_expand_t<T, 12>(c, a, rows, min_log2Nc);
      case 14: return launch_expand_t<T, 14>(c, a, rows, min_log2Nc);
      case 16: return launch_expand_t<T, 16>(c, a, rows, min_log2Nc);
      case 20: return launch_expand_t<T, 20>(c, a, rows, min_log2Nc);
    }
  } else {
    switch (taps) {
      case 6: return launch_expand_t<T, 6>(c, a, rows, min_log2Nc);
      case 8: return launch_expand_t<T, 8>(c, a, rows, min_log2Nc);
      case 10: return launch_expand_t<T, 10>(c, a, rows, min_log2Nc);
    }
  }
  return fail(c, CWTB_ERR_STATE, "expansion: unsupported tap count");
}

// all kernels of one transform: forward FFT of the (device, type T) signal, then every scale
template <typename T>
static int run_job(cwtb_ctx *c, const Job &job, const T *dsig, cx<T> *Wout = nullptr, int epi = EPI_STORE) {
  using V = cx<T>;
  if (job.exact) {
    if constexpr (std::is_same<T, double>::value) return run_job_exact(c, job, dsig, Wout, epi);
    else return fail(c, CWTB_ERR_UNSUPPORTED, "un-padded transforms run in fp64");
  }
  const unsigned N = job.N;
  const int S = job.S * job.nbatch;   // rows: one per (channel, scale)
  int e;
  // whatever path leaves this function (also an error in the middle of the fork), the launcher
  // is back on the engine's stream afterwards
  struct CurGuard { cwtb_ctx *c; ~CurGuard() { c->cur = c->stream; c->prof_tag = ""; c->ztmp = nullptr; } } cur_guard{c};
  if ((e = ensure(c, c->spec, (size_t)job.nbatch * N * sizeof(V)))) return e;
  if (!Wout) {
    if ((e = ensure(c, c->W, (size_t)S * job.n0 * sizeof(V)))) return e;
    Wout = (V *)c->W.p;
  }
  V *spec = (V *)c->spec.p;
  V *W = Wout;
  const ScaleDesc *ddesc = (const ScaleDesc *)c->descs.p;
  Fam fam = job.fam;
  if (fam.family == CWTB_TABLE) fam.table = (const double2 *)c->table.p;

  // ---- forward transform of the zero-padded signal (wavelet.py:91) ----
  if (N < 32) {
    if (job.nbatch != 1) return fail(c, CWTB_ERR_UNSUPPORTED, "batched transform needs n0 > 16");
    TinyFwdArgs<T> fa{dsig, spec, job.n0, N};
    if ((e = launch<TinyFwdBody<T>>(c, 1, 1, fa))) return e;
    TinyArgs<T> ta{ddesc, spec, W, fam, job.n0, N, 0, epi};
    return launch<TinyBody<T>>(c, (unsigned)((job.n0 + NT - 1) / NT), S, ta);
  }
  c->prof_tag = "fwd:";
  e = fft_rows<T, -1>(c, dsig, 1, job.n0, job.n0, spec, N, N, job.nbatch);
  c->prof_tag = "";
  if (e) return e;

  NTab nt;
  if ((e = get_ntab(c, N, job.log2N, &nt))) return e;
  const int G = chunk_rows(c, N, sizeof(V));
  const size_t bchunk = band_chunk_elems(c, job, G);   // two regions: one per chain stream
  if ((e = ensure(c, c->B, (job.b_single + (size_t)std::max(1, c->n_chains) * bchunk) * sizeof(V)))) return e;
  V *Bbuf = (V *)c->B.p;

  // band products of every single-kernel scale in one launch (their descriptors are contiguous
  // in the class-sorted array; blocks beyond a scale's K' exit immediately)
  {
    int first = -1, maxlk = 0, nrows = 0;
    for (const ClassRun &cl : job.classes)
      if (class_single(c, job, cl)) {
        if (first < 0) first = cl.first;
        maxlk = std::max(maxlk, cl.log2K);
        nrows += cl.count;
      }
    if (first >= 0) {
      BandArgs<T> ba{ddesc, spec, Bbuf, fam, N, first};
      const unsigned Kmax = 1u << maxlk;
      if ((e = launch<BandBody<T>>(c, (Kmax + NT * BandBody<T>::PER - 1) / (NT * BandBody<T>::PER), nrows, ba)))
        return e;
    }
  }
  // The single-kernel classes (independent of the two-kernel chains: different W rows, read-only
  // band products) run on a second stream so that their CTAs fill the tails of the chains.
  const bool split = c->two_streams != 0;
#ifndef CWTB_HOST_EMU
  const bool split2 = split && c->three_streams && !c->fused;
  if (split) {
    RT(cudaEventRecord(c->ev_fork, c->stream));
    RT(cudaStreamWaitEvent(c->aux_stream, c->ev_fork, 0));
    if (split2)
      for (int k = 1; k < c->n_chains; ++k) RT(cudaStreamWaitEvent(c->chain_streams[k - 1], c->ev_fork, 0));
  }
#else
  const bool split2 = false;
#endif
  // ---- expansion classes (kernels.cuh: ExpandBody): coarse band spectra of every expansion row
  // in one launch, one batched coarse transform per coarse length, one expansion launch per class.
  // They run on the second stream like the single-kernel classes (own transform intermediate Zx).
  if (job.coarse_elems) {
#ifndef CWTB_HOST_EMU
    // the ~30 small launches in front of the expansion kernels go to the priority stream: queued
    // behind the big launches of the other streams they would only advance in those launches' tails
    const bool prio = split && c->prio_mode > 0;
    if (prio) RT(cudaStreamWaitEvent(c->prio_stream, c->ev_fork, 0));
    if (split) c->cur = prio ? c->prio_stream : c->aux_stream;
#endif
    if ((e = ensure(c, c->Cin, job.coarse_elems * sizeof(V)))) return e;
    if ((e = ensure(c, c->Cout, job.coarse_elems * sizeof(V)))) return e;
    int first = -1, maxl = 0, nrows = 0;
    for (const ClassRun &cl : job.classes)
      if (cl.expand) {
        if (first < 0) first = cl.first;
        maxl = std::max(maxl, cl.log2Nc);
        nrows += cl.count;
      }
    ExpandBandArgs<T> xa{ddesc, spec, (V *)c->Cin.p, fam, N, first};
    constexpr int XPER = ExpandBandBody<T>::PER;
    if ((e = launch<ExpandBandBody<T>>(c, ((1u << maxl) + NT * XPER - 1) / (NT * XPER), nrows, xa))) return e;
    c->ztmp = &c->Zx;
    c->prof_tag = "coarse:";
#ifndef CWTB_HOST_EMU
    const int fan = prio ? c->prio_fan : 1;   // groups of one coarse length rotate over this many streams
    int fan_used = 1, group = 0;
    if (fan > 1) RT(cudaEventRecord(c->ev_xband, c->prio_stream));
#endif
    for (size_t ci = 0; ci < job.classes.size() && !e; ++ci) {
      const ClassRun &cl = job.classes[ci];
      if (!cl.expand) continue;
      // coarse transforms: consecutive classes of one coarse length at once (rows are contiguous)
      if (ci == 0 || !job.classes[ci - 1].expand || job.classes[ci - 1].log2Nc != cl.log2Nc) {
        int rows = 0;
        for (size_t cj = ci; cj < job.classes.size() && job.classes[cj].expand && job.classes[cj].log2Nc == cl.log2Nc; ++cj)
          rows += job.classes[cj].count;
        const long long off = job.descs[cl.first].ip_coff;
        const unsigned Nc = 1u << cl.log2Nc;
#ifndef CWTB_HOST_EMU
        if (fan > 1) {
          const int slot = group++ % fan;
          if (slot > 0) {
            if (slot >= fan_used) {   // first use in this call: behind the band products
              RT(cudaStreamWaitEvent(c->prio_aux[slot - 1], c->ev_xband, 0));
              fan_used = slot + 1;
            }
            c->cur = c->prio_aux[slot - 1];
            c->ztmp = &c->Zxs[slot - 1];
          } else {
            c->cur = c->prio_stream;
            c->ztmp = &c->Zx;
          }
        }
#endif
        e = fft_rows<T, +1>(c, (const V *)c->Cin.p + off, 0, Nc, Nc, (V *)c->Cout.p + off, Nc, Nc, rows);
      }
    }
#ifndef CWTB_HOST_EMU
    if (fan > 1) {   // join the fan on the priority stream
      for (int k = 1; k < fan_used; ++k) {
        RT(cudaEventRecord(c->ev_pj[k - 1], c->prio_aux[k - 1]));
        RT(cudaStreamWaitEvent(c->prio_stream, c->ev_pj[k - 1], 0));
      }
      c->cur = c->prio_stream;
      c->ztmp = &c->Zx;
    }
#endif
    c->prof_tag = "";
#ifndef CWTB_HOST_EMU
    if (prio && c->prio_mode == 1) {   // expansion kernels: ordinary priority, after the coarse chain
      RT(cudaEventRecord(c->ev_coarse, c->prio_stream));
      RT(cudaStreamWaitEvent(c->aux_stream, c->ev_coarse, 0));
      c->cur = c->aux_stream;
    }
#endif
    // one expansion launch per tap count: classes are sorted by taps first
    for (size_t ci = 0; ci < job.classes.size() && !e; ++ci) {
      const ClassRun &cl = job.classes[ci];
      if (!cl.expand || (ci > 0 && job.classes[ci - 1].expand && job.classes[ci - 1].taps == cl.taps)) continue;
      int rows = 0, minl = 30;
      for (size_t cj = ci; cj < job.classes.size() && job.classes[cj].expand && job.classes[cj].taps == cl.taps; ++cj) {
        rows += job.classes[cj].count;
        minl = std::min(minl, job.classes[cj].log2Nc);
      }
      ExpandArgs<T> ea{ddesc, (const V *)c->Cout.p, (const double *)c->wtab.p, W, nt, job.n0, N, cl.first, epi,
                       job.log2N};
      e = launch_expand<T>(c, cl.taps, ea, rows, minl);
    }
    c->ztmp = nullptr;
#ifndef CWTB_HOST_EMU
    if (prio && c->prio_mode == 2 && !e) {   // later work of the second stream and the join follow the priority stream
      RT(cudaEventRecord(c->ev_coarse, c->prio_stream));
      RT(cudaStreamWaitEvent(c->aux_stream, c->ev_coarse, 0));
    }
#endif
    c->cur = c->stream;
    if (e) return e;
  }
  int chain_no = 0;
  for (int pass = 0; pass < 2; ++pass)
  for (const ClassRun &cl : job.classes) {
    if (cl.expand) continue;
    const unsigned K = 1u << cl.log2K;
    const bool single = class_single(c, job, cl);
    if (single != (pass == 0)) continue;   // pass 0: single-kernel classes, pass 1: two-kernel chains
    if (single) {
#ifndef CWTB_HOST_EMU
      if (split) c->cur = c->aux_stream;
#endif
      // ---- single kernel: pruned K'-point transforms from the band products ----
      SingleArgs<T> sa{ddesc, Bbuf, W, Tw<T>::get(c), nt, job.n0, N, cl.first, epi};
      switch (cl.log2K) {
        case 5: e = launch_single<T, 32>(c, sa, cl.count); break;
        case 6: e = launch_single<T, 64>(c, sa, cl.count); break;
        case 7: e = launch_single<T, 128>(c, sa, cl.count); break;
        case 8: e = launch_single<T, 256>(c, sa, cl.count); break;
        case 9: e = launch_single<T, 512>(c, sa, cl.count); break;
        case 10: e = launch_single<T, 1024>(c, sa, cl.count); break;
        case 11: e = launch<DirectBody<T, 2>>(c, (N / K2C + Lay<T, K2C>::P - 1) / Lay<T, K2C>::P, cl.count, sa); break;
        case 12: e = launch<DirectBody<T, 4>>(c, (N / K2C + Lay<T, K2C>::P - 1) / Lay<T, K2C>::P, cl.count, sa); break;
        case 13: e = launch<DirectBody<T, 8>>(c, (N / K2C + Lay<T, K2C>::P - 1) / Lay<T, K2C>::P, cl.count, sa); break;
        default: e = fail(c, CWTB_ERR_STATE, "bad single-kernel class");
      }
      c->cur = c->stream;
      if (e) return e;
      continue;
    }
    // ---- two kernels through Z ----
    const bool dense = (cl.log2K == job.log2N);
    if (dense && job.log2N > 20) {
      // ---- Np > 2^20: pre-pass (K0-point transforms over rows of 2^20, response generated
      // in-kernel) into Y, then the K0 interleaved 2^20-point transforms of every scale ----
      const int l0 = job.log2N - 20;
      const unsigned Nsub = 1u << 20;
      const int gy = std::max<int>(1, (int)std::min<size_t>((size_t)cl.count, ((size_t)512 << 20) / ((size_t)N * sizeof(V))));
      if ((e = ensure(c, c->Y, (size_t)gy * N * sizeof(V)))) return e;
      for (int g0 = 0; g0 < cl.count; g0 += gy) {
        const int ng = std::min(gy, cl.count - g0);
        PassAArgs<T> a{};
        a.descs = ddesc; a.spec = spec; a.Bbuf = Bbuf; a.Z = (V *)c->Y.p; a.tw = Tw<T>::get(c);
        a.fam = fam; a.nt = nt; a.N = N; a.first = cl.first + g0; a.row0 = 0; a.zmod = 1 << 30;
        a.pf_dist = 0; a.K2 = Nsub; a.gauss_rec = c->gauss_rec;
        if ((e = dispatch_passA<T, +1, MODE_DENSE>(c, l0, a, ng))) return e;
        if ((e = two_kernel_rows<T, +1>(c, c->Y.p, 0, Nsub, Nsub, W, job.n0, Nsub, ng << l0, job.n0, nullptr, 1.0,
                                         1 << l0, ddesc, cl.first + g0, 0, epi)))
          return e;
      }
      continue;
    }
    const bool persistent = class_persistent(c, cl);
    const int chunk = persistent ? cl.count : G;   // persistent: the whole class in one launch
    // successive two-kernel classes rotate over the chains, each with its own stream, Z buffer
    // and band-chunk region (descriptor offsets already point into the right region)
    const int chain = split2 ? job_chain_region(c, job, cl) : 0;
    Buf &Zb = chain > 0 ? c->Zc[chain - 1] : c->Z;
    if ((e = ensure(c, Zb, (size_t)(persistent ? c->ring : G) * N * sizeof(V)))) return e;
#ifndef CWTB_HOST_EMU
    c->cur = chain > 0 ? c->chain_streams[chain - 1] : c->stream;
#endif
    ++chain_no;
    for (int g0 = 0; g0 < cl.count; g0 += chunk) {
      const int ng = std::min(chunk, cl.count - g0);
      PassAArgs<T> a{};
      a.descs = ddesc; a.spec = spec; a.Bbuf = Bbuf; a.Z = (V *)Zb.p; a.tw = Tw<T>::get(c);
      a.fam = fam; a.nt = nt; a.N = N; a.first = cl.first + g0; a.row0 = 0; a.zmod = 1 << 30;
      // band scales: second pass of 512 points (full 128-byte output runs, conflict-free tile);
      // dense scales keep 1024 so that K1 = N/K2 <= 1024
      // (fp32: the 512-point tile has an odd row pitch, its rows would not be 16-byte aligned)
      constexpr bool k512_ok = (Lay<T, 512, true>::PITCH * sizeof(V)) % 16 == 0;
      // 512 pays up to K' = 2^16 (measured per class: first kernel + second kernel per row)
      // (a first kernel of K1 points covers TILE / K1 values of r2 per tile: at most 512 for rows
      // of 512, so K1 >= 8 in fp64; K' = 2^11 under CWTB_DIRECT_MAX=10 keeps 1024)
      const bool k1_fits_512 = (TileCfg<T>::TILE >> std::max(0, cl.log2K - 9)) <= 512;
      const int l2k = (dense || persistent || cl.log2K > c->k2_512_max_log2 || !k512_ok || !k1_fits_512)
                          ? 10 : c->k2_band_log2;
      a.pf_dist = c->pf_dist_a; a.K2 = 1u << l2k; a.gauss_rec = c->gauss_rec;
      PassBArgs<T> b{};
      b.Z = (const V *)Zb.p; b.out = W; b.tw = Tw<T>::get(c); b.descs = ddesc;
      b.pitch = job.n0; b.nout = job.n0; b.N = N; b.first = cl.first + g0; b.row0 = 0;
      b.epi = epi; b.grow = nullptr; b.post = 1.0; b.zmod = 1 << 30;
      b.pf_dist = c->pf_dist; b.ny = ng; b.rev = c->passb_rev;
      if (!dense) {
        BandArgs<T> ba{ddesc, spec, Bbuf, fam, N, cl.first + g0};
        if ((e = launch<BandBody<T>>(c, (K + NT * BandBody<T>::PER - 1) / (NT * BandBody<T>::PER), ng, ba)))
          return e;
      }
      if (c->fused == 2 && persistent) {
        e = dense ? dispatch_pipe<T, MODE_DENSE>(c, cl.log2K - 10, a, b, ng)
                  : dispatch_pipe<T, MODE_BAND>(c, cl.log2K - 10, a, b, ng);
        if (e) return e;
        continue;
      }
      if (c->fused == 1) {
        e = dense ? dispatch_fused<T, MODE_DENSE>(c, cl.log2K - 10, a, b, ng)
                  : dispatch_fused<T, MODE_BAND>(c, cl.log2K - 10, a, b, ng);
        if (e) return e;
        continue;
      }
      e = dense ? dispatch_passA<T, +1, MODE_DENSE>(c, cl.log2K - l2k, a, ng)
                : dispatch_passA<T, +1, MODE_BAND>(c, cl.log2K - l2k, a, ng);
      if (e) return e;
      if constexpr (k512_ok) {
        if (l2k == 9)
          e = launch<PassBBody<T, +1, 512>>(c, (N / 512 + Lay<T, 512>::P - 1) / Lay<T, 512>::P, ng, b);
      }
      if (l2k != 9)
        e = launch<PassBBody<T, +1>>(c, (N / K2C + Lay<T, K2C>::P - 1) / Lay<T, K2C>::P, ng, b);
      if (e) return e;
    }
    c->cur = c->stream;
  }
  (void)chain_no;
#ifndef CWTB_HOST_EMU
  if (split) {   // join: later work on the main stream sees every row of W
    RT(cudaEventRecord(c->ev_join, c->aux_stream));
    RT(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
    if (split2)
      for (int k = 1; k < c->n_chains; ++k) {
        RT(cudaEventRecord(c->ev_joinc[k - 1], c->chain_streams[k - 1]));
        RT(cudaStreamWaitEvent(c->stream, c->ev_joinc[k - 1], 0));
      }
  }
#endif
  return 0;
}

// band-buffer offsets of the two-kernel scales depend on the chunk position; set them here
static void assign_chunk_offsets(cwtb_ctx *c, Job &job) {
  const int G = chunk_rows(c, job.N, job.precision == CWTB_F64 ? sizeof(double2) : sizeof(float2));
  const size_t bchunk = band_chunk_elems(c, job, G);
  for (const ClassRun &cl : job.classes) {
    if (!class_two_kernel(c, job, cl) || cl.log2K == job.log2N) continue;
    const size_t region = (size_t)job_chain_region(c, job, cl) * bchunk;
    for (int i = 0; i < cl.count; ++i)
      job.descs[cl.first + i].boff =
          (long long)(job.b_single + region + (size_t)(class_persistent(c, cl) ? i : i % G) * ((size_t)1 << cl.log2K));
  }
}

static int upload_descs(cwtb_ctx *c, Job &job) {
  assign_chunk_offsets(c, job);
  if (c->wtab_host.size() > c->wtab_uploaded) {   // new expansion weight tables (appended)
    const size_t bytes = c->wtab_host.size() * sizeof(double);
    if (c->wtab.bytes < bytes) {
      RT(rt_sync(c->stream));
      int e2 = ensure(c, c->wtab, std::max(bytes, (size_t)2 * c->wtab.bytes));
      if (e2) return e2;
      c->wtab_uploaded = 0;   // a new allocation: everything again
    }
    RT(rt_h2d((char *)c->wtab.p + c->wtab_uploaded * sizeof(double), c->wtab_host.data() + c->wtab_uploaded,
              (c->wtab_host.size() - c->wtab_uploaded) * sizeof(double), c->stream));
    c->wtab_uploaded = c->wtab_host.size();
  }
  int e = ensure(c, c->descs, job.descs.size() * sizeof(ScaleDesc));
  if (e) return e;
  RT(rt_h2d(c->descs.p, job.descs.data(), job.descs.size() * sizeof(ScaleDesc), c->stream));
  RT(rt_sync(c->stream));  // job.descs is pageable host memory
  return 0;
}

static int timed_run(cwtb_ctx *c, const void *dsig, int iters, double *ms_out) {
  const Job &job = c->job;
  c->launches = 0;
#ifndef CWTB_HOST_EMU
  RT(cudaEventRecord(c->e0, c->stream));
#endif
  for (int it = 0; it < iters; ++it) {
    int e = job.precision == CWTB_F64 ? run_job<double>(c, job, (const double *)dsig)
                                      : run_job<float>(c, job, (const float *)dsig);
    if (e) return e;
  }
  float ms = 0;
#ifndef CWTB_HOST_EMU
  RT(cudaEventRecord(c->e1, c->stream));
  RT(cudaEventSynchronize(c->e1));
  RT(cudaEventElapsedTime(&ms, c->e0, c->e1));
#endif
  if (ms_out) *ms_out = (double)ms / iters;
  c->launches /= std::max(1, iters);
  return 0;
}

// ---- conversions ---------------------------------------------------------------------
template <typename TI, typename TO> struct CvtArgs { const TI *in; TO *out; long long n; };
template <typename TI, typename TO> struct CvtBody {
  using Args = CvtArgs<TI, TO>;
  static constexpr int NPHASE = 1;
  static constexpr size_t SMEM = 0;
  template <int PH> HD static void phase(const Args &a, int bx, int, int tid, void *) {
    long long i = (long long)bx * NT + tid;
    if (i < a.n) a.out[i] = (TO)a.in[i];
  }
};

// ======================================================================================
// C ABI
// ======================================================================================
extern "C" {

const char *cwtb_version(void) {
#ifdef CWTB_HOST_EMU
  return "cwt_b200 0.1 (host emulation build - tests only)";
#else
  return "cwt_b200 0.1 (sm_100a)";
#endif
}

int cwtb_device_count(void) {
#ifdef CWTB_HOST_EMU
  return 1;
#else
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
#endif
}

int cwtb_create(int device, cwtb_ctx **out) {
  if (!out) return CWTB_ERR_ARG;
  *out = nullptr;
  cwtb_ctx *c = new cwtb_ctx();
  c->device = device;
#ifndef CWTB_HOST_EMU
  if (cudaSetDevice(device) != cudaSuccess) { delete c; return CWTB_ERR_CUDA; }
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return CWTB_ERR_CUDA; }
  cudaEventCreate(&c->e0);
  cudaEventCreate(&c->e1);
  for (auto &st : c->copy_streams) cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
  cudaStreamCreateWithFlags(&c->aux_stream, cudaStreamNonBlocking);
  {
    int lo = 0, hi = 0;   // numerically lower = higher priority
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    cudaStreamCreateWithPriority(&c->prio_stream, cudaStreamNonBlocking, hi);
    for (auto &st : c->prio_aux) cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, hi);
  }
  cudaEventCreateWithFlags(&c->ev_xband, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&c->ev_angle, cudaEventDisableTiming);
  for (auto &ev : c->ev_pj) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  if (const char *g = getenv("CWTB_PRIO_FAN")) c->prio_fan = std::min(8, std::max(1, atoi(g)));
  cudaEventCreateWithFlags(&c->ev_coarse, cudaEventDisableTiming);
  for (auto &ev : c->ev_h2d) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  for (auto &ev : c->ev_used) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  if (const char *g = getenv("CWTB_BATCH_PIPELINE")) c->batch_pipeline = atoi(g) != 0;
  if (const char *g = getenv("CWTB_PRIO")) c->prio_mode = std::min(2, std::max(0, atoi(g)));
  for (auto &st : c->chain_streams) cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
  for (auto &ev : c->ev_joinc) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming);
  if (const char *g = getenv("CWTB_STREAMS")) { c->two_streams = atoi(g) >= 2; c->three_streams = atoi(g) >= 3; }
  if (const char *g = getenv("CWTB_D2H_SPLIT")) c->d2h_split = std::min(4, std::max(1, atoi(g)));
#endif
  c->cur = c->stream;
  if (const char *g = getenv("CWTB_GROUP")) c->group = std::max(0, atoi(g));
  if (const char *g = getenv("CWTB_GROUP_MB")) c->group_bytes = (size_t)std::max(1, atoi(g)) << 20;
  if (const char *g = getenv("CWTB_ROWS_CHUNK_MB")) c->rows_chunk_bytes = (size_t)std::max(1, atoi(g)) << 20;
  if (const char *g = getenv("CWTB_BAND_EPS")) c->band_eps = atof(g);
  if (const char *g = getenv("CWTB_BAND_EPS32")) c->band_eps32 = atof(g);
  if (const char *g = getenv("CWTB_EXPAND_EPS")) c->expand_eps = std::max(0.0, atof(g));
  if (const char *g = getenv("CWTB_EXPAND_EPS32")) c->expand_eps32 = std::max(0.0, atof(g));
  if (const char *g = getenv("CWTB_EXPAND_MIN_R")) c->expand_min_log2R = std::min(14, std::max(2, atoi(g)));
  if (const char *g = getenv("CWTB_EXPAND_MMA")) c->expand_mma = atoi(g) != 0;
  if (const char *g = getenv("CWTB_PLAN_REUSE")) c->plan_reuse = atoi(g) != 0;
  if (const char *g = getenv("CWTB_DENSE_MARGIN")) c->dense_margin = std::max(0, atoi(g));
  if (const char *g = getenv("CWTB_L2_PERSIST")) c->l2_persist = atoi(g);
  if (const char *g = getenv("CWTB_FUSED")) c->fused = atoi(g);
  if (const char *g = getenv("CWTB_PF_DIST")) c->pf_dist = std::max(0, atoi(g));
  if (const char *g = getenv("CWTB_CHAINS")) c->n_chains = std::min(4, std::max(1, atoi(g)));
  if (const char *g = getenv("CWTB_FFT_PAD")) c->pad_pow2 = atoi(g) != 0;
  if (const char *g = getenv("CWTB_PF_ROWS_A")) c->pf_rows_a = std::max(0, atoi(g));
  if (const char *g = getenv("CWTB_PF_ROWS_B")) c->pf_rows_b = std::max(0, atoi(g));
  if (const char *g = getenv("CWTB_PF_DIST_A")) c->pf_dist_a = std::max(0, atoi(g));
  if (const char *g = getenv("CWTB_K2_BAND")) c->k2_band_log2 = atoi(g) == 10 ? 10 : 9;
  if (const char *g = getenv("CWTB_K2_512_MAX")) c->k2_512_max_log2 = std::min(19, atoi(g));
  if (const char *g = getenv("CWTB_PASSB_REV")) c->passb_rev = atoi(g) != 0;
  if (const char *g = getenv("CWTB_GAUSS_REC")) c->gauss_rec = atoi(g);
  if (const char *g = getenv("CWTB_BATCH_MB")) c->batch_bytes = (size_t)std::max(1, atoi(g)) << 20;
  if (const char *g = getenv("CWTB_RING")) c->ring = std::max(1, atoi(g));
  else if (c->fused == 2) c->ring = 4;
  if (const char *g = getenv("CWTB_AHEAD")) c->pipe_ahead = std::max(1, atoi(g));
#ifndef CWTB_HOST_EMU
  cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, device);
#endif
  if (const char *g = getenv("CWTB_DIRECT_MAX")) c->direct_max_log2 = std::min(13, std::max(10, atoi(g)));
  int e = init_tables(c);
  if (e == 0) e = rt_sync(c->stream) ? CWTB_ERR_CUDA : 0;
  if (e) { delete c; return e; }
  *out = c;
  return CWTB_OK;
}

void cwtb_destroy(cwtb_ctx *c) {
  if (!c) return;
#ifndef CWTB_HOST_EMU
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
#endif
  cwtb_comm_destroy(c);
  for (Buf *b : {&c->Zxs[0], &c->Zxs[1], &c->Zxs[2], &c->Zxs[3], &c->Zxs[4], &c->Zxs[5], &c->Zxs[6], &c->stage_dev[0], &c->stage_dev[1], &c->batch_power, &c->filt, &c->comm_send, &c->comm_recv, &c->Zx, &c->Cin, &c->Cout, &c->wtab, &c->ctr, &c->sig, &c->sig2, &c->spec, &c->Z, &c->Zc[0], &c->Zc[1], &c->Zc[2], &c->Y, &c->B, &c->W, &c->W2, &c->descs, &c->table, &c->scratch,
                 &c->C, &c->A12, &c->F, &c->aux, &c->rowd, &c->win, &c->mask, &c->hist, &c->noise, &c->wide, &c->blueA, &c->blueX, &c->blueY})
    if (b->p) rt_free(b->p);
  for (auto &kv : c->ntabs) { rt_free(kv.second.hi); rt_free(kv.second.lo); }
  for (auto &kv : c->blue) { rt_free(kv.second.wm); rt_free(kv.second.bf[0]); rt_free(kv.second.bf[1]); }
  if (c->tw64) rt_free(c->tw64);
  if (c->tw32) rt_free(c->tw32);
  for (void *p : c->pinned) rt_host_free(p);
  for (void *p : c->devallocs) rt_free(p);
#ifndef CWTB_HOST_EMU
  cudaEventDestroy(c->e0);
  cudaEventDestroy(c->e1);
  cudaStreamDestroy(c->stream);
  for (auto &st : c->copy_streams) cudaStreamDestroy(st);
  cudaStreamDestroy(c->aux_stream);
  cudaStreamDestroy(c->prio_stream);
  for (auto &st : c->prio_aux) cudaStreamDestroy(st);
  cudaEventDestroy(c->ev_xband);
  cudaEventDestroy(c->ev_angle);
  for (auto &ev : c->ev_pj) cudaEventDestroy(ev);
  cudaEventDestroy(c->ev_coarse);
  for (auto &ev : c->ev_h2d) cudaEventDestroy(ev);
  for (auto &ev : c->ev_used) cudaEventDestroy(ev);
  for (void *p : c->stage_host) if (p) cudaFreeHost(p);
  for (auto &st : c->chain_streams) cudaStreamDestroy(st);
  for (auto &ev : c->ev_joinc) cudaEventDestroy(ev);
  cudaEventDestroy(c->ev_fork);
  cudaEventDestroy(c->ev_join);
#endif
  delete c;
}

const char *cwtb_last_error(cwtb_ctx *c) { return c ? c->err.c_str() : "null context"; }

int cwtb_set_band_eps(cwtb_ctx *c, double eps) {
  if (!c || !(eps >= 0) || eps >= 1e-6) return fail(c, CWTB_ERR_ARG, "band eps must be in [0, 1e-6)");
  c->band_eps = eps;
  return 0;
}

int cwtb_set_expand_eps(cwtb_ctx *c, double eps64, double eps32) {
  if (!c || !(eps64 >= 0) || !(eps32 >= 0) || eps64 > 1e-6 || eps32 > 1e-3)
    return fail(c, CWTB_ERR_ARG, "expansion tolerance must be in [0, 1e-6] (fp64) / [0, 1e-3] (fp32)");
  c->expand_eps = eps64;
  c->expand_eps32 = eps32;
  return 0;
}

int cwtb_host_alloc(cwtb_ctx *c, size_t bytes, void **out) {
  if (!c || !out) return CWTB_ERR_ARG;
  if (rt_host_alloc(out, bytes) != 0) return fail(c, CWTB_ERR_NOMEM, "pinned allocation failed");
  c->pinned.insert(*out);
  return 0;
}
int cwtb_host_free(cwtb_ctx *c, void *p) {
  if (!c || !c->pinned.count(p)) return CWTB_ERR_ARG;
  c->pinned.erase(p);
  rt_host_free(p);
  return 0;
}
int cwtb_dev_alloc(cwtb_ctx *c, size_t bytes, void **out) {
  if (!c || !out) return CWTB_ERR_ARG;
  if (rt_malloc(out, bytes) != 0) return fail(c, CWTB_ERR_NOMEM, "device allocation failed");
  c->devallocs.insert(*out);
  return 0;
}
int cwtb_dev_free(cwtb_ctx *c, void *p) {
  if (!c || !c->devallocs.count(p)) return CWTB_ERR_ARG;
  c->devallocs.erase(p);
  rt_free(p);
  return 0;
}
int cwtb_memcpy_h2d(cwtb_ctx *c, void *dst, const void *src, size_t bytes) {
  RT(rt_h2d(dst, src, bytes, c->stream));
  RT(rt_sync(c->stream));
  return 0;
}
int cwtb_memcpy_d2h(cwtb_ctx *c, void *dst, const void *src, size_t bytes) {
  RT(rt_d2h(dst, src, bytes, c->stream));
  RT(rt_sync(c->stream));
  return 0;
}
int cwtb_sync(cwtb_ctx *c) {
  RT(rt_sync(c->stream));
  return 0;
}

static int prepare(cwtb_ctx *c, long long n0, double dt, const double *scales, int S, int family,
                   double param, int precision, const void *table, int nbatch = 1) {
  if (!c) return CWTB_ERR_ARG;
  if (precision != CWTB_F64 && precision != CWTB_F32) return fail(c, CWTB_ERR_ARG, "bad precision");
  if (!scales) return fail(c, CWTB_ERR_ARG, "null scales");
#ifndef CWTB_HOST_EMU
  RT(cudaSetDevice(c->device));
#endif
  if (nbatch < 1 || (long long)nbatch * S > 60000) return fail(c, CWTB_ERR_ARG, "batch too large for one launch");
  ++c->serial;   // whatever was resident is about to be replaced
  cwtb_ctx::PlanKey key;
  key.n0 = n0; key.dt = dt; key.param = param; key.band_eps = c->band_eps; key.band_eps32 = c->band_eps32;
  key.expand_eps = c->expand_eps; key.expand_eps32 = c->expand_eps32; key.S = S; key.family = family;
  key.precision = precision; key.nbatch = nbatch; key.pad = c->pad_pow2;
  key.scales.assign(scales, scales + std::max(S, 0));
  if (c->plan_reuse && family != CWTB_TABLE && c->job.valid && key == c->plan_key) return 0;
  c->plan_key = cwtb_ctx::PlanKey();   // invalid until the new plan is complete
  int e = build_job(c, c->job, n0, dt, scales, S, family, param, precision, table != nullptr, nbatch);
  if (e) return e;
  if (family == CWTB_TABLE) {
    size_t bytes = (size_t)S * c->job.N * sizeof(double2);
    if ((e = ensure(c, c->table, bytes))) return e;
    RT(rt_h2d(c->table.p, table, bytes, c->stream));
  }
  if ((e = upload_descs(c, c->job))) return e;
  if (family != CWTB_TABLE) c->plan_key = std::move(key);
  return 0;
}

int cwtb_cwt_dev(cwtb_ctx *c, const void *d_signal, int signal_is_f32, int64_t n0, double dt,
                 const double *scales, int n_scales, int family, double param, int precision) {
  if (!c || !d_signal) return fail(c, CWTB_ERR_ARG, "null argument");
  if (family == CWTB_TABLE) return fail(c, CWTB_ERR_UNSUPPORTED, "use cwtb_cwt for CWTB_TABLE");
  int e = prepare(c, n0, dt, scales, n_scales, family, param, precision, nullptr);
  if (e) return e;
  const void *dsig = d_signal;
  const bool want_f32 = (precision == CWTB_F32);
  if ((signal_is_f32 != 0) != want_f32) {  // convert to the engine's real type
    if ((e = ensure(c, c->sig, (size_t)n0 * (want_f32 ? 4 : 8)))) return e;
    unsigned gx = (unsigned)((n0 + NT - 1) / NT);
    if (want_f32) {
      CvtArgs<double, float> a{(const double *)d_signal, (float *)c->sig.p, n0};
      e = launch<CvtBody<double, float>>(c, gx, 1, a);
    } else {
      CvtArgs<float, double> a{(const float *)d_signal, (double *)c->sig.p, n0};
      e = launch<CvtBody<float, double>>(c, gx, 1, a);
    }
    if (e) return e;
    dsig = c->sig.p;
  }
  c->job_dsig = dsig;
  c->job.sig_is_f32 = want_f32;
  return timed_run(c, dsig, 1, &c->last_ms);
}

int cwtb_cwt(cwtb_ctx *c, const void *signal, int signal_is_f32, int64_t n0, double dt,
             const double *scales, int n_scales, int family, double param, int precision,
             const void *table) {
  if (!c || !signal) return fail(c, CWTB_ERR_ARG, "null argument");
  int e = prepare(c, n0, dt, scales, n_scales, family, param, precision, table);
  if (e) return e;
  const bool want_f32 = (precision == CWTB_F32);
  const size_t esz = want_f32 ? 4 : 8;
  if ((e = ensure(c, c->sig, (size_t)n0 * esz))) return e;
  if ((signal_is_f32 != 0) == want_f32) {
    RT(rt_h2d(c->sig.p, signal, (size_t)n0 * esz, c->stream));
    RT(rt_sync(c->stream));
  } else {
    std::vector<unsigned char> tmp((size_t)n0 * esz);
    if (want_f32) for (int64_t i = 0; i < n0; ++i) ((float *)tmp.data())[i] = (float)((const double *)signal)[i];
    else for (int64_t i = 0; i < n0; ++i) ((double *)tmp.data())[i] = (double)((const float *)signal)[i];
    RT(rt_h2d(c->sig.p, tmp.data(), (size_t)n0 * esz, c->stream));
    RT(rt_sync(c->stream));
  }
  c->job_dsig = c->sig.p;
  c->job.sig_is_f32 = want_f32;
  return timed_run(c, c->sig.p, 1, &c->last_ms);
}

int cwtb_bench_last(cwtb_ctx *c, int iters, double *ms_out) {
  if (!c || !c->job.valid || !c->job_dsig) return fail(c, CWTB_ERR_STATE, "no transform to re-run");
  if (iters < 1) return fail(c, CWTB_ERR_ARG, "iters < 1");
  return timed_run(c, c->job_dsig, iters, ms_out);
}

double cwtb_last_kernel_ms(cwtb_ctx *c) { return c ? c->last_ms : -1; }
int cwtb_last_launch_count(cwtb_ctx *c) { return c ? c->launches : -1; }
int64_t cwtb_padded_length(cwtb_ctx *c) { return (c && c->job.valid) ? (int64_t)c->job.N : -1; }
int64_t cwtb_job_serial(cwtb_ctx *c) { return c ? c->serial : -1; }
void *cwtb_w_device_ptr(cwtb_ctx *c) { return (c && c->job.valid) ? c->W.p : nullptr; }

int cwtb_last_plan(cwtb_ctx *c, int *out, int n) {
  if (!c || !c->job.valid || !out) return CWTB_ERR_ARG;
  int m = std::min<int>(n, (int)c->job.plan_log2K.size());
  for (int i = 0; i < m; ++i) out[i] = c->job.plan_log2K[i];
  return m;
}

int cwtb_get_w(cwtb_ctx *c, void *out, int out_f64, int row0, int nrows) {
  if (!c || !c->job.valid || !out) return fail(c, CWTB_ERR_STATE, "no transform resident");
  const Job &job = c->job;
  if (row0 < 0 || nrows < 0 || row0 + nrows > job.S * job.nbatch) return fail(c, CWTB_ERR_ARG, "row range");
  const size_t cnt = (size_t)nrows * job.n0;
  if (job.precision == CWTB_F64) {
    const char *src = (const char *)((const double2 *)c->W.p + (size_t)row0 * job.n0);
    const size_t bytes = cnt * sizeof(double2);
#ifndef CWTB_HOST_EMU
    if (c->d2h_split > 1 && bytes >= ((size_t)64 << 20)) {
      RT(rt_sync(c->stream));   // kernels done
      const int ns = c->d2h_split;
      const size_t piece = ((bytes / ns) + 255) & ~(size_t)255;
      for (int i = 0; i < ns; ++i) {
        const size_t off = (size_t)i * piece;
        if (off >= bytes) break;
        RT(rt_d2h((char *)out + off, src + off, std::min(piece, bytes - off), c->copy_streams[i]));
      }
      for (int i = 0; i < ns; ++i) RT(rt_sync(c->copy_streams[i]));
      return 0;
    }
#endif
    RT(rt_d2h(out, src, bytes, c->stream));
    RT(rt_sync(c->stream));
  } else if (!out_f64) {
    RT(rt_d2h(out, (const float2 *)c->W.p + (size_t)row0 * job.n0, cnt * sizeof(float2), c->stream));
    RT(rt_sync(c->stream));
  } else {
    // complex64 on the device, complex128 for the caller: widen on the device in chunks and
    // copy each chunk out while the next one is converted (two staging halves, two streams).
    // 16 B per element over PCIe beats an 8 B copy plus a host-side conversion pass.
    const float2 *src = (const float2 *)c->W.p + (size_t)row0 * job.n0;
    const size_t chunk = std::min<size_t>(cnt, (size_t)8 << 20);   // elements per staging half
    int e;
    if ((e = ensure(c, c->wide, 2 * chunk * sizeof(double2)))) return e;
    RT(rt_sync(c->stream));   // kernels done
    int half = 0;
    for (size_t off = 0; off < cnt; off += chunk, half ^= 1) {
      const size_t m = std::min(chunk, cnt - off);
      double2 *stage = (double2 *)c->wide.p + (size_t)half * chunk;
      WidenArgs wa{src + off, stage, (long long)m};
      c->cur = c->copy_streams[half];
      e = launch<WidenBody>(c, (unsigned)((m + 4 * NT - 1) / (4 * NT)), 1, wa);
      c->cur = c->stream;
      if (e) return e;
      RT(rt_d2h((double2 *)out + off, stage, m * sizeof(double2), c->copy_streams[half]));
    }
    RT(rt_sync(c->copy_streams[0]));
    RT(rt_sync(c->copy_streams[1]));
  }
  return 0;
}

int cwtb_get_signal_fft(cwtb_ctx *c, void *out) {
  if (!c || !c->job.valid || !out) return fail(c, CWTB_ERR_STATE, "no transform resident");
  const Job &job = c->job;
  const size_t cnt = job.N / 2 > 0 ? job.N / 2 - 1 : 0;
  if (cnt == 0) return 0;
  const double sc = 1.0 / std::sqrt((double)job.N);
  double *o = (double *)out;
  if (job.precision == CWTB_F64) {
    // scaled on the device (the host loop cost as much as the 8 MB copy at N = 2^20)
    int e = ensure(c, c->aux, cnt * sizeof(double2));
    if (e) return e;
    ScaleCopyArgs sa{(const double *)((const double2 *)c->spec.p + 1), (double *)c->aux.p, (long long)(2 * cnt), sc};
    if ((e = launch<ScaleCopyBody>(c, (unsigned)((2 * cnt + NT - 1) / NT), 1, sa))) return e;
    RT(rt_d2h(out, c->aux.p, cnt * sizeof(double2), c->stream));
    RT(rt_sync(c->stream));
  } else {
    std::vector<float> tmp(cnt * 2);
    RT(rt_d2h(tmp.data(), (const float2 *)c->spec.p + 1, cnt * sizeof(float2), c->stream));
    RT(rt_sync(c->stream));
    for (size_t i = 0; i < cnt * 2; ++i) o[i] = (double)tmp[i] * sc;
  }
  return 0;
}

int cwtb_fft_c2c(cwtb_ctx *c, const void *in, void *out, int64_t n, int batch, int sign, int precision) {
  if (!c || !in || !out || n < 2 || batch < 1 || (sign != 1 && sign != -1))
    return fail(c, CWTB_ERR_ARG, "fft_c2c: bad argument");
  if (precision != CWTB_F64 && precision != CWTB_F32) return fail(c, CWTB_ERR_ARG, "bad precision");
  if (n > (1ll << 26)) return fail(c, CWTB_ERR_UNSUPPORTED, "fft_c2c: n > 2^26");
  const bool pow2 = (n & (n - 1)) == 0;
  if (!pow2 && precision != CWTB_F64) return fail(c, CWTB_ERR_UNSUPPORTED, "fft_c2c: lengths other than 2^k run in fp64");
  if (!pow2 && n > (1ll << 24)) return fail(c, CWTB_ERR_UNSUPPORTED, "fft_c2c: non power-of-two n > 2^24");
#ifndef CWTB_HOST_EMU
  RT(cudaSetDevice(c->device));
#endif
  const size_t cnt = (size_t)n * batch;
  const size_t esz = precision == CWTB_F64 ? sizeof(double2) : sizeof(float2);
  int e;
  // context-owned staging buffers (released with the context, also on error paths)
  if ((e = ensure(c, c->C, cnt * esz))) return e;
  if ((e = ensure(c, c->A12, cnt * esz))) return e;
  void *din = c->C.p, *dout = c->A12.p;
  if (!pow2) {   // any length: Bluestein on the power-of-two kernels
    RT(rt_h2d(din, in, cnt * esz, c->stream));
    if ((e = blue_rows(c, din, 0, n, (double2 *)dout, n, (unsigned)n, batch, sign, 1.0, n))) return e;
    RT(rt_d2h(out, dout, cnt * esz, c->stream));
    RT(rt_sync(c->stream));
    return 0;
  }
  if (precision == CWTB_F64) {
    RT(rt_h2d(din, in, cnt * esz, c->stream));
    e = sign < 0 ? fft_rows<double, -1>(c, din, 0, n, n, (double2 *)dout, n, (unsigned)n, batch)
                 : fft_rows<double, +1>(c, din, 0, n, n, (double2 *)dout, n, (unsigned)n, batch);
    if (e) return e;
    RT(rt_d2h(out, dout, cnt * esz, c->stream));
    RT(rt_sync(c->stream));
    return 0;
  }
  std::vector<float> tmp(cnt * 2);
  const double *src = (const double *)in;
  for (size_t i = 0; i < cnt * 2; ++i) tmp[i] = (float)src[i];
  RT(rt_h2d(din, tmp.data(), cnt * esz, c->stream));
  RT(rt_sync(c->stream));
  e = sign < 0 ? fft_rows<float, -1>(c, din, 0, n, n, (float2 *)dout, n, (unsigned)n, batch)
               : fft_rows<float, +1>(c, din, 0, n, n, (float2 *)dout, n, (unsigned)n, batch);
  if (e) return e;
  RT(rt_d2h(tmp.data(), dout, cnt * esz, c->stream));
  RT(rt_sync(c->stream));
  double *o = (double *)out;
  for (size_t i = 0; i < cnt * 2; ++i) o[i] = (double)tmp[i];
  return 0;
}

}  // extern "C"

extern "C" {

// device time of a kernel sequence on the engine's stream -> cwtb_last_kernel_ms
static int time_begin(cwtb_ctx *c) {
#ifndef CWTB_HOST_EMU
  RT(cudaEventRecord(c->e0, c->stream));
#endif
  c->last_ms = 0;
  return 0;
}
static int time_end(cwtb_ctx *c) {
#ifndef CWTB_HOST_EMU
  float ms = 0;
  RT(cudaEventRecord(c->e1, c->stream));
  RT(cudaEventSynchronize(c->e1));
  RT(cudaEventElapsedTime(&ms, c->e0, c->e1));
  c->last_ms = ms;
#endif
  return 0;
}

// ---- helpers for the post-processing entry points ---------------------------------------
static int upload_doubles(cwtb_ctx *c, Buf &b, const std::vector<double> &v) {
  int e = ensure(c, b, v.size() * sizeof(double));
  if (e) return e;
  RT(rt_h2d(b.p, v.data(), v.size() * sizeof(double), c->stream));
  RT(rt_sync(c->stream));
  return 0;
}

static int upload_signal_f64(cwtb_ctx *c, Buf &b, const double *y, long long n0) {
  int e = ensure(c, b, (size_t)n0 * sizeof(double));
  if (e) return e;
  RT(rt_h2d(b.p, y, (size_t)n0 * sizeof(double), c->stream));
  RT(rt_sync(c->stream));
  return 0;
}

// boxcar with half-weight end taps, normalised (helpers.py:176-191)
static int upload_window(cwtb_ctx *c, int K) {
  if (K < 1) return fail(c, CWTB_ERR_ARG, "boxcar length must be >= 1");
  std::vector<double> w(K, 1.0);
  w[0] = 0.5;
  w[K - 1] = 0.5;   // K == 1: single tap 0.5, normalised to 1
  double sum = 0;
  for (double v : w) sum += v;
  for (double &v : w) v /= sum;
  return upload_doubles(c, c->win, w);
}

// Morlet.smooth, time part (mothers.py:83-93), in place on X[S][n0] (complex128, device):
// forward transform of the zero-padded rows with the Gaussian folded into its output pass,
// inverse transform trimmed to n0.
static int smooth_time(cwtb_ctx *c, double2 *X, int S, long long n0, unsigned N, const double *d_g) {
  int e = ensure(c, c->F, (size_t)S * N * sizeof(double2));
  if (e) return e;
  double2 *F = (double2 *)c->F.p;
  if (N < 2) return 0;  // single sample: filter is exp(0) = 1
  const bool table = c->filt_rows > 0;     // caller-supplied responses instead of Morlet's Gaussian
  if (table && (c->filt_rows != S || c->filt_n != (long long)N))
    return fail(c, CWTB_ERR_STATE, "smoothing filter table does not match the rows / transform length of this call");
  if ((N & (N - 1)) != 0) {
    // un-padded mode: circular filter at the rows' own length (N == n0), Bluestein transforms
    if ((e = blue_rows(c, X, 0, n0, F, N, N, S, -1, 1.0, N))) return e;
    if (table) {
      FilterMulArgs fa{F, (const double *)c->filt.p, (long long)N, N, 1.0 / (double)N};
      if ((e = launch<FilterMulBody>(c, (N + NT - 1) / NT, S, fa))) return e;
    } else {
      BlueGaussArgs ga{F, d_g, (long long)N, N, 1.0 / (double)N};
      if ((e = launch<BlueGaussBody>(c, (N + NT - 1) / NT, S, ga))) return e;
    }
    return blue_rows(c, F, 0, N, X, n0, N, S, +1, 1.0, n0);
  }
  if (table) {
    if ((e = fft_rows<double, -1>(c, X, 0, n0, n0, F, N, N, S, N))) return e;
    FilterMulArgs fa{F, (const double *)c->filt.p, (long long)N, N, 1.0 / (double)N};
    if ((e = launch<FilterMulBody>(c, (N + NT - 1) / NT, S, fa))) return e;
  } else if ((e = fft_rows<double, -1>(c, X, 0, n0, n0, F, N, N, S, N, d_g, 1.0 / (double)N))) {
    return e;
  }
  return fft_rows<double, +1>(c, F, 0, N, N, X, n0, N, S, n0);
}

// two transforms + coherence pipeline; outputs are device pointers (any may be null)
static int wct_core(cwtb_ctx *c, const Job &job, const double *dsig1, const double *dsig2, int K,
                    double *dWCT, double *daWCT, const unsigned char *dmask, int maxscale, int nbins,
                    unsigned long long *dhist) {
  const int S = job.S;
  const long long n0 = job.n0;
  const size_t cnt = (size_t)S * n0;
  int e;
  if ((e = ensure(c, c->W, cnt * sizeof(double2)))) return e;
  if ((e = ensure(c, c->W2, cnt * sizeof(double2)))) return e;
  if ((e = ensure(c, c->C, cnt * sizeof(double2)))) return e;
  if ((e = ensure(c, c->A12, cnt * sizeof(double2)))) return e;
  if ((e = run_job<double>(c, job, dsig1, (double2 *)c->W.p, EPI_STORE))) return e;
  if ((e = run_job<double>(c, job, dsig2, (double2 *)c->W2.p, EPI_STORE))) return e;
  const double *d_scale = (const double *)c->rowd.p;      // [S] scales, then [S] g
  const double *d_g = d_scale + S;
  WctPrepArgs pa{(const double2 *)c->W.p, (const double2 *)c->W2.p, d_scale, (double2 *)c->C.p,
                 (double2 *)c->A12.p, daWCT, n0};
  const unsigned gx = (unsigned)((n0 + NT - 1) / NT);
  if ((e = launch<WctPrepBody>(c, gx, S, pa))) return e;
#ifndef CWTB_HOST_EMU
  if (c->angle_host && daWCT) {   // the angle is final here: its 8 B per point cross PCIe under the smoothing
    RT(cudaEventRecord(c->ev_angle, c->stream));
    RT(cudaStreamWaitEvent(c->copy_streams[0], c->ev_angle, 0));
    RT(cudaMemcpyAsync(c->angle_host, daWCT, cnt * sizeof(double), cudaMemcpyDeviceToHost, c->copy_streams[0]));
  }
#endif
  if ((e = smooth_time(c, (double2 *)c->C.p, S, n0, job.N, d_g))) return e;
  if ((e = smooth_time(c, (double2 *)c->A12.p, S, n0, job.N, d_g))) return e;
  WctFinalArgs fa{(const double2 *)c->C.p, (const double2 *)c->A12.p, (const double *)c->win.p, dWCT,
                  dmask, dhist, n0, S, K, maxscale, nbins};
  if (K > 64) return fail(c, CWTB_ERR_UNSUPPORTED, "scale boxcar longer than 64 taps");
  const int rows_out = dWCT ? S : maxscale;
  if (rows_out <= 0) return 0;
  using F16 = WctFinalBody<16>;
  const unsigned fx = (unsigned)((n0 + F16::CW - 1) / F16::CW), fy = (unsigned)((rows_out + F16::RS - 1) / F16::RS);
  return K <= 16 ? launch<F16>(c, fx, fy, fa) : launch<WctFinalBody<64>>(c, fx, fy, fa);
}

static int upload_row_tables(cwtb_ctx *c, const Job &job) {
  std::vector<double> v(2 * (size_t)job.S);
  for (int j = 0; j < job.S; ++j) {
    v[j] = job.scales[j];
    const double snorm = job.scales[j] / job.dt;
    v[job.S + j] = -0.5 * (snorm * snorm);
  }
  return upload_doubles(c, c->rowd, v);
}

// rows of W written by the single-kernel classes (the chain on aux_stream): true and *r0 set if
// they are exactly the rows [r0, S) -- the case for any ascending scale array
static bool single_kernel_rows(const cwtb_ctx *c, const Job &job, int *r0) {
  const int S = job.S;
  int lo = S, cnt = 0;
  for (const ClassRun &cl : job.classes) {
    if (!(cl.expand || class_single(c, job, cl))) continue;
    for (int i = cl.first; i < cl.first + cl.count; ++i) {
      lo = std::min(lo, job.descs[i].row);
      ++cnt;
    }
  }
  if (cnt == 0 || cnt == S || lo != S - cnt) return false;
  *r0 = lo;
  return true;
}

int cwtb_cwt_to_host(cwtb_ctx *c, const void *signal, int signal_is_f32, int64_t n0, double dt,
                     const double *scales, int n_scales, int family, double param, int precision,
                     void *out, int out_f64) {
  if (!c || !signal || !out) return fail(c, CWTB_ERR_ARG, "null argument");
#ifndef CWTB_HOST_EMU
  // fp64, analytic family, forked streams: the device->host copy of the rows the single-kernel
  // chain produced starts as soon as that chain is done, while the two-kernel chains still run
  if (precision == CWTB_F64 && family != CWTB_TABLE && c->two_streams && !c->profiling) {
    int e = prepare(c, n0, dt, scales, n_scales, family, param, precision, nullptr);
    if (e) return e;
    const Job &job = c->job;
    int r0 = 0;
    if (!job.exact && job.N >= 32 && job.nbatch == 1 && single_kernel_rows(c, job, &r0)) {
      if ((e = ensure(c, c->sig, (size_t)n0 * sizeof(double)))) return e;
      if (signal_is_f32) {
        std::vector<double> tmp((size_t)n0);
        for (int64_t i = 0; i < n0; ++i) tmp[i] = (double)((const float *)signal)[i];
        RT(rt_h2d(c->sig.p, tmp.data(), (size_t)n0 * sizeof(double), c->stream));
        RT(rt_sync(c->stream));
      } else {
        RT(rt_h2d(c->sig.p, signal, (size_t)n0 * sizeof(double), c->stream));
      }
      c->job_dsig = c->sig.p;
      c->job.sig_is_f32 = 0;
      c->launches = 0;
      RT(cudaEventRecord(c->e0, c->stream));
      if ((e = run_job<double>(c, job, (const double *)c->sig.p))) return e;
      RT(cudaEventRecord(c->e1, c->stream));
      const size_t rowb = (size_t)n0 * sizeof(double2);
      const char *W = (const char *)c->W.p;
      RT(cudaStreamWaitEvent(c->copy_streams[0], c->ev_join, 0));   // single-kernel chain done
      RT(rt_d2h((char *)out + (size_t)r0 * rowb, W + (size_t)r0 * rowb, (size_t)(n_scales - r0) * rowb, c->copy_streams[0]));
      RT(rt_d2h(out, W, (size_t)r0 * rowb, c->stream));               // after every chain has joined
      RT(rt_sync(c->copy_streams[0]));
      RT(rt_sync(c->stream));
      float ms = 0;
      RT(cudaEventElapsedTime(&ms, c->e0, c->e1));
      c->last_ms = ms;
      return 0;
    }
    // not eligible: fall through to the plain sequence (prepare runs again, cheap)
  }
#endif
  int e = cwtb_cwt(c, signal, signal_is_f32, n0, dt, scales, n_scales, family, param, precision, nullptr);
  if (e) return e;
  return cwtb_get_w(c, out, out_f64, 0, n_scales);
}

// rows per block of the column reductions: enough blocks to fill the machine, few enough that the
// atomics stay negligible
static int reduction_rows_per_block(int rows) { return rows <= 32 ? rows : 32; }

int cwtb_icwt_sum(cwtb_ctx *c, double *out) {
  if (!c || !c->job.valid || !out) return fail(c, CWTB_ERR_STATE, "no transform resident");
  const Job &job = c->job;
  if (job.nbatch != 1) return fail(c, CWTB_ERR_UNSUPPORTED, "icwt of a batched transform: fetch rows per channel");
  std::vector<double> rs(job.S);
  for (int j = 0; j < job.S; ++j) rs[j] = 1.0 / std::sqrt(job.scales[j]);
  int e = upload_doubles(c, c->rowd, rs);
  if (e) return e;
  if ((e = ensure(c, c->aux, (size_t)job.n0 * sizeof(double)))) return e;
  const unsigned gx = (unsigned)((job.n0 + NT - 1) / NT);
  const int rpb = reduction_rows_per_block(job.S);
  const unsigned gy = (unsigned)((job.S + rpb - 1) / rpb);
  if (gy > 1) RT(rt_memset(c->aux.p, 0, (size_t)job.n0 * sizeof(double), c->stream));
  if (job.precision == CWTB_F64) {
    IcwtArgs<double> a{(const double2 *)c->W.p, (const double *)c->rowd.p, (double *)c->aux.p, job.n0, job.n0, job.S, 0, rpb};
    e = launch<IcwtBody<double>>(c, gx, gy, a);
  } else {
    IcwtArgs<float> a{(const float2 *)c->W.p, (const double *)c->rowd.p, (double *)c->aux.p, job.n0, job.n0, job.S, 0, rpb};
    e = launch<IcwtBody<float>>(c, gx, gy, a);
  }
  if (e) return e;
  RT(rt_d2h(out, c->aux.p, (size_t)job.n0 * sizeof(double), c->stream));
  RT(rt_sync(c->stream));
  return 0;
}

int cwtb_icwt_sum_host(cwtb_ctx *c, const void *W, const double *scales, int n_scales, int64_t n, double *out) {
  if (!c || !W || !scales || !out || n_scales < 1 || n < 1) return fail(c, CWTB_ERR_ARG, "icwt: bad argument");
  std::vector<double> rs(n_scales);
  for (int j = 0; j < n_scales; ++j) rs[j] = 1.0 / std::sqrt(scales[j]);
  int e = upload_doubles(c, c->rowd, rs);
  if (e) return e;
  if ((e = ensure(c, c->aux, (size_t)n * sizeof(double)))) return e;
  const int chunk = (int)std::max<long long>(1, std::min<long long>(n_scales, (256ll << 20) / (n * 16)));
  if ((e = ensure(c, c->scratch, (size_t)chunk * n * sizeof(double2)))) return e;
  const unsigned gx = (unsigned)((n + NT - 1) / NT);
  for (int r0 = 0; r0 < n_scales; r0 += chunk) {
    const int nr = std::min(chunk, n_scales - r0);
    RT(rt_h2d(c->scratch.p, (const double2 *)W + (size_t)r0 * n, (size_t)nr * n * sizeof(double2), c->stream));
    IcwtArgs<double> a{(const double2 *)c->scratch.p, (const double *)c->rowd.p + r0, (double *)c->aux.p, n, n, nr, r0 > 0, nr};
    if ((e = launch<IcwtBody<double>>(c, gx, 1, a))) return e;
    RT(rt_sync(c->stream));
  }
  RT(rt_d2h(out, c->aux.p, (size_t)n * sizeof(double), c->stream));
  RT(rt_sync(c->stream));
  return 0;
}

static int power_common(cwtb_ctx *c, double *power_out, double *mean_out, const double *row_scale,
                        const int64_t *lo, const int64_t *hi) {
  if (!c || !c->job.valid) return fail(c, CWTB_ERR_STATE, "no transform resident");
  const Job &job = c->job;
  const int R = job.S * job.nbatch;
  const size_t cnt = (size_t)R * job.n0;
  // aux: [row sums R][row factors R][lo R][hi R][power cnt]
  int e = ensure(c, c->aux, (power_out ? cnt : 0) * sizeof(double) + (size_t)4 * R * sizeof(double));
  if (e) return e;
  double *dsum = (double *)c->aux.p;
  double *dmul = dsum + R;
  long long *dlo = (long long *)(dmul + R), *dhi = dlo + R;
  double *dpow = power_out ? (double *)(dhi + R) : nullptr;
  RT(rt_memset(dsum, 0, (size_t)R * sizeof(double), c->stream));
  if (row_scale) RT(rt_h2d(dmul, row_scale, (size_t)R * sizeof(double), c->stream));
  std::vector<long long> rng;
  if (lo && hi) {
    rng.resize(2 * (size_t)R);
    for (int j = 0; j < R; ++j) {
      rng[j] = std::max<long long>(0, lo[j]);
      rng[R + j] = std::min<long long>(job.n0, hi[j]);
    }
    RT(rt_h2d(dlo, rng.data(), rng.size() * sizeof(long long), c->stream));
  }
  const unsigned gx = (unsigned)((job.n0 + PowerBody<double>::PER * NT - 1) / (PowerBody<double>::PER * NT));
  if (job.precision == CWTB_F64) {
    PowerArgs<double> a{(const double2 *)c->W.p, dpow, dsum, job.n0, row_scale ? dmul : nullptr,
                        rng.empty() ? nullptr : dlo, rng.empty() ? nullptr : dhi};
    e = launch<PowerBody<double>>(c, gx, R, a);
  } else {
    PowerArgs<float> a{(const float2 *)c->W.p, dpow, dsum, job.n0, row_scale ? dmul : nullptr,
                       rng.empty() ? nullptr : dlo, rng.empty() ? nullptr : dhi};
    e = launch<PowerBody<float>>(c, gx, R, a);
  }
  if (e) return e;
  if (power_out) RT(rt_d2h(power_out, dpow, cnt * sizeof(double), c->stream));
  if (mean_out) RT(rt_d2h(mean_out, dsum, (size_t)R * sizeof(double), c->stream));
  RT(rt_sync(c->stream));   // also covers the pageable host sources above
  if (mean_out)
    for (int j = 0; j < R; ++j) {
      const long long cntj = rng.empty() ? (long long)job.n0 : rng[R + j] - rng[j];
      mean_out[j] = cntj > 0 ? mean_out[j] / (double)cntj : std::nan("");
    }
  return 0;
}
int cwtb_get_power(cwtb_ctx *c, double *out) { return power_common(c, out, nullptr, nullptr, nullptr, nullptr); }
int cwtb_global_power(cwtb_ctx *c, double *out) { return power_common(c, nullptr, out, nullptr, nullptr, nullptr); }
int cwtb_get_power_scaled(cwtb_ctx *c, const double *row_scale, double *out) {
  if (!out) return fail(c, CWTB_ERR_ARG, "null argument");
  return power_common(c, out, nullptr, row_scale, nullptr, nullptr);
}
int cwtb_global_power_ranges(cwtb_ctx *c, const int64_t *lo, const int64_t *hi, double *out) {
  if (!lo || !hi || !out) return fail(c, CWTB_ERR_ARG, "null argument");
  return power_common(c, nullptr, out, nullptr, lo, hi);
}

int cwtb_scale_avg_power(cwtb_ctx *c, const double *weights, double *out) {
  if (!c || !c->job.valid) return fail(c, CWTB_ERR_STATE, "no transform resident");
  if (!weights || !out) return fail(c, CWTB_ERR_ARG, "null argument");
  const Job &job = c->job;
  if (job.nbatch != 1) return fail(c, CWTB_ERR_UNSUPPORTED, "scale average of a batched transform: fetch rows per channel");
  // [weights S doubles][selected rows S ints]: rows with a zero weight are not read at all
  std::vector<double> w(weights, weights + job.S);
  std::vector<int> sel;
  for (int j = 0; j < job.S; ++j)
    if (w[j] != 0.0) sel.push_back(j);
  const int nsel = (int)sel.size();
  w.resize((size_t)job.S + ((size_t)job.S + 1) / 2);
  if (nsel) memcpy(w.data() + job.S, sel.data(), sizeof(int) * nsel);
  int e = upload_doubles(c, c->rowd, w);
  if (e) return e;
  if ((e = ensure(c, c->aux, (size_t)job.n0 * sizeof(double)))) return e;
  const unsigned gx = (unsigned)((job.n0 + NT - 1) / NT);
  const int spb = nsel <= 32 ? std::max(nsel, 1) : 32;
  const unsigned gy = (unsigned)std::max(1, (nsel + spb - 1) / spb);
  if (gy > 1) RT(rt_memset(c->aux.p, 0, (size_t)job.n0 * sizeof(double), c->stream));
  const int *dsel = (const int *)((const double *)c->rowd.p + job.S);
  if (job.precision == CWTB_F64) {
    ScaleAvgArgs<double> a{(const double2 *)c->W.p, (const double *)c->rowd.p, (double *)c->aux.p, job.n0, job.S, dsel, nsel, spb};
    e = launch<ScaleAvgBody<double>>(c, gx, gy, a);
  } else {
    ScaleAvgArgs<float> a{(const float2 *)c->W.p, (const double *)c->rowd.p, (double *)c->aux.p, job.n0, job.S, dsel, nsel, spb};
    e = launch<ScaleAvgBody<float>>(c, gx, gy, a);
  }
  if (e) return e;
  RT(rt_d2h(out, c->aux.p, (size_t)job.n0 * sizeof(double), c->stream));
  RT(rt_sync(c->stream));
  return 0;
}

int cwtb_xwt(cwtb_ctx *c, const double *y1, const double *y2, int64_t n0, double dt, const double *scales,
             int n_scales, int family, double param, void *W12_out) {
  if (!c || !y1 || !y2) return fail(c, CWTB_ERR_ARG, "null argument");
  if (family == CWTB_TABLE) return fail(c, CWTB_ERR_UNSUPPORTED, "xwt needs an analytic wavelet family");
  int e = prepare(c, n0, dt, scales, n_scales, family, param, CWTB_F64, nullptr);
  if (e) return e;
  if ((e = upload_signal_f64(c, c->sig, y1, n0))) return e;
  if ((e = upload_signal_f64(c, c->sig2, y2, n0))) return e;
  c->launches = 0;
  if ((e = time_begin(c))) return e;
  if ((e = run_job<double>(c, c->job, (const double *)c->sig.p, nullptr, EPI_STORE))) return e;
  if ((e = run_job<double>(c, c->job, (const double *)c->sig2.p, nullptr, EPI_MULCONJ))) return e;
  if ((e = time_end(c))) return e;
  c->job_dsig = nullptr;
  if (W12_out) return cwtb_get_w(c, W12_out, 1, 0, n_scales);
  RT(rt_sync(c->stream));
  return 0;
}

int cwtb_wct(cwtb_ctx *c, const double *y1, const double *y2, int64_t n0, double dt, double dj,
             const double *scales, int n_scales, int family, double param, int boxcar_len,
             double *WCT_out, double *aWCT_out) {
  (void)dj;
  if (!c || !y1 || !y2) return fail(c, CWTB_ERR_ARG, "null argument");
  if (family == CWTB_TABLE) return fail(c, CWTB_ERR_UNSUPPORTED, "wct needs an analytic wavelet family");
  int e = prepare(c, n0, dt, scales, n_scales, family, param, CWTB_F64, nullptr);
  if (e) return e;
  if ((e = upload_signal_f64(c, c->sig, y1, n0))) return e;
  if ((e = upload_signal_f64(c, c->sig2, y2, n0))) return e;
  if ((e = upload_window(c, boxcar_len))) return e;
  if ((e = upload_row_tables(c, c->job))) return e;
  const size_t cnt = (size_t)n_scales * n0;
  if ((e = ensure(c, c->aux, 2 * cnt * sizeof(double)))) return e;
  double *dW = (double *)c->aux.p, *dA = dW + cnt;
  c->launches = 0;
  if ((e = time_begin(c))) return e;
  bool early_angle = false;
#ifndef CWTB_HOST_EMU
  c->angle_host = aWCT_out;
  early_angle = aWCT_out != nullptr;
#endif
  e = wct_core(c, c->job, (const double *)c->sig.p, (const double *)c->sig2.p, boxcar_len, dW,
               aWCT_out ? dA : nullptr, nullptr, 0, 0, nullptr);
  c->angle_host = nullptr;
  if (e) return e;
  if ((e = time_end(c))) return e;
  c->job_dsig = nullptr;
  if (WCT_out) RT(rt_d2h(WCT_out, dW, cnt * sizeof(double), c->stream));
  if (aWCT_out && !early_angle) RT(rt_d2h(aWCT_out, dA, cnt * sizeof(double), c->stream));
  RT(rt_sync(c->stream));
#ifndef CWTB_HOST_EMU
  if (early_angle) RT(rt_sync(c->copy_streams[0]));
#endif
  return 0;
}

int cwtb_set_smooth_filter(cwtb_ctx *c, const double *table, int n_rows, int64_t n) {
  if (!c) return CWTB_ERR_ARG;
  if (!table || n_rows <= 0 || n <= 0) {   // back to Morlet's Gaussian (mothers.py:83-91)
    c->filt_rows = 0;
    c->filt_n = 0;
    return 0;
  }
#ifndef CWTB_HOST_EMU
  RT(cudaSetDevice(c->device));
#endif
  const size_t bytes = (size_t)n_rows * (size_t)n * sizeof(double);
  int e = ensure(c, c->filt, bytes);
  if (e) return e;
  RT(rt_h2d(c->filt.p, table, bytes, c->stream));
  RT(rt_sync(c->stream));
  c->filt_rows = n_rows;
  c->filt_n = n;
  return 0;
}

int cwtb_set_padding(cwtb_ctx *c, int pad_to_pow2) {
  if (!c) return CWTB_ERR_ARG;
  c->pad_pow2 = pad_to_pow2 != 0;
  return 0;
}

int cwtb_smooth(cwtb_ctx *c, const void *in, int is_complex, int n_scales, int64_t n, double dt,
                const double *scales, int boxcar_len, void *out) {
  if (!c || !in || !out || !scales || n_scales < 1 || n < 1 || !(dt > 0))
    return fail(c, CWTB_ERR_ARG, "smooth: bad argument");
  if (n > (1ll << 26)) return fail(c, CWTB_ERR_UNSUPPORTED, "smooth: rows longer than 2^26");
#ifndef CWTB_HOST_EMU
  RT(cudaSetDevice(c->device));
#endif
  const int S = n_scales;
  const size_t cnt = (size_t)S * n;
  if (!c->pad_pow2 && n > (1ll << 24)) return fail(c, CWTB_ERR_UNSUPPORTED, "smooth: un-padded rows longer than 2^24");
  const unsigned N = c->pad_pow2 ? 1u << ilog2((unsigned long long)n) : (unsigned)n;   // helpers.py:15-30
  int e = upload_window(c, boxcar_len);
  if (e) return e;
  std::vector<double> g(2 * (size_t)S);
  for (int j = 0; j < S; ++j) { g[j] = scales[j]; double sn = scales[j] / dt; g[S + j] = -0.5 * (sn * sn); }
  if ((e = upload_doubles(c, c->rowd, g))) return e;
  if ((e = ensure(c, c->C, cnt * sizeof(double2)))) return e;
  if ((e = ensure(c, c->A12, cnt * sizeof(double2)))) return e;
  double2 *X = (double2 *)c->C.p, *Y = (double2 *)c->A12.p;
  if (is_complex) {
    RT(rt_h2d(X, in, cnt * sizeof(double2), c->stream));
  } else {
    RT(rt_h2d(Y, in, cnt * sizeof(double), c->stream));   // stage the reals in Y, widen into X
    R2CArgs ra{(const double *)Y, X, (long long)cnt};
    if ((e = launch<R2CBody>(c, (unsigned)((cnt + NT - 1) / NT), 1, ra))) return e;
  }
  if ((e = smooth_time(c, X, S, n, N, (const double *)c->rowd.p + S))) return e;
  BoxcarArgs ba{X, Y, (const double *)c->win.p, n, S, boxcar_len};
  if ((e = launch<BoxcarBody>(c, (unsigned)((n + NT - 1) / NT), S, ba))) return e;
  if (is_complex) {
    RT(rt_d2h(out, Y, cnt * sizeof(double2), c->stream));
    RT(rt_sync(c->stream));
  } else {
    std::vector<double2> tmp(cnt);
    RT(rt_d2h(tmp.data(), Y, cnt * sizeof(double2), c->stream));
    RT(rt_sync(c->stream));
    double *o = (double *)out;
    for (size_t i = 0; i < cnt; ++i) o[i] = tmp[i].x;   // .real, mothers.py:95-96
  }
  return 0;
}

// common part of the two Monte-Carlo entry points: `noise` host surrogates [n_pairs][2][n0], or
// null -> drawn on the device from (seed, pair0 + i)
static int wct_mc_core(cwtb_ctx *c, const double *noise, unsigned long long seed, long long pair0, int n_pairs,
                       int64_t n0, double dt, const double *scales, int n_scales, int family, double param,
                       int boxcar_len, const uint8_t *mask, int maxscale, int nbins, int64_t *hist) {
  if (!c || !mask || !hist || n_pairs < 0 || nbins < 1 || maxscale < 0 || maxscale > n_scales)
    return fail(c, CWTB_ERR_ARG, "wct_mc: bad argument");
  if (family == CWTB_TABLE) return fail(c, CWTB_ERR_UNSUPPORTED, "wct_mc needs an analytic wavelet family");
  int e = prepare(c, n0, dt, scales, n_scales, family, param, CWTB_F64, nullptr);
  if (e) return e;
  if ((e = upload_window(c, boxcar_len))) return e;
  if ((e = upload_row_tables(c, c->job))) return e;
  const size_t cnt = (size_t)n_scales * n0;
  if ((e = ensure(c, c->mask, cnt))) return e;
  RT(rt_h2d(c->mask.p, mask, cnt, c->stream));
  const size_t hb = (size_t)n_scales * nbins * sizeof(unsigned long long);
  if ((e = ensure(c, c->hist, hb))) return e;
  RT(rt_memset(c->hist.p, 0, hb, c->stream));
  // surrogates of at most `batch` pairs are resident at a time
  const int batch = noise ? n_pairs : (int)std::max<size_t>(1, std::min<size_t>((size_t)n_pairs, ((size_t)256 << 20) / ((size_t)2 * n0 * sizeof(double))));
  if ((e = ensure(c, c->noise, (size_t)std::max(batch, 1) * 2 * n0 * sizeof(double)))) return e;
  if (noise) RT(rt_h2d(c->noise.p, noise, (size_t)n_pairs * 2 * n0 * sizeof(double), c->stream));
  RT(rt_sync(c->stream));
  c->launches = 0;
  if ((e = time_begin(c))) return e;
  for (int i0 = 0; i0 < n_pairs; i0 += batch) {
    const int nb = std::min(batch, n_pairs - i0);
    if (!noise) {
      NoiseArgs na{(double *)c->noise.p, seed, pair0 + i0, (long long)n0, nb};
      if ((e = launch<NoiseBody>(c, (unsigned)(((n0 + 1) / 2 + NT - 1) / NT), (unsigned)(2 * nb), na))) return e;
    }
    for (int i = 0; i < nb; ++i) {
      const double *a = (const double *)c->noise.p + (size_t)i * 2 * n0;
      if ((e = wct_core(c, c->job, a, a + n0, boxcar_len, nullptr, nullptr, (const unsigned char *)c->mask.p,
                        maxscale, nbins, (unsigned long long *)c->hist.p)))
        return e;
    }
  }
  if ((e = time_end(c))) return e;
  c->job_dsig = nullptr;
  std::vector<unsigned long long> h((size_t)n_scales * nbins);
  RT(rt_d2h(h.data(), c->hist.p, hb, c->stream));
  RT(rt_sync(c->stream));
  for (size_t i = 0; i < h.size(); ++i) hist[i] += (int64_t)h[i];
  return 0;
}

int cwtb_wct_mc(cwtb_ctx *c, const double *noise, int n_pairs, int64_t n0, double dt, double dj,
                const double *scales, int n_scales, int family, double param, int boxcar_len,
                const uint8_t *mask, int maxscale, int nbins, int64_t *hist) {
  (void)dj;
  if (!noise) return fail(c, CWTB_ERR_ARG, "wct_mc: null surrogates");
  return wct_mc_core(c, noise, 0, 0, n_pairs, n0, dt, scales, n_scales, family, param, boxcar_len, mask,
                     maxscale, nbins, hist);
}

int cwtb_wct_mc_seeded(cwtb_ctx *c, uint64_t seed, int64_t first_pair, int n_pairs, int64_t n0, double dt,
                       const double *scales, int n_scales, int family, double param, int boxcar_len,
                       const uint8_t *mask, int maxscale, int nbins, int64_t *hist) {
  return wct_mc_core(c, nullptr, seed, first_pair, n_pairs, n0, dt, scales, n_scales, family, param, boxcar_len,
                     mask, maxscale, nbins, hist);
}

// test hook: the surrogates of the seeded mode, [n_pairs][2][n0] to the host
int cwtb_mc_surrogates(cwtb_ctx *c, uint64_t seed, int64_t first_pair, int n_pairs, int64_t n0, double *out) {
  if (!c || !out || n_pairs < 1 || n0 < 1) return fail(c, CWTB_ERR_ARG, "mc_surrogates: bad argument");
  int e = ensure(c, c->noise, (size_t)n_pairs * 2 * n0 * sizeof(double));
  if (e) return e;
  NoiseArgs na{(double *)c->noise.p, seed, first_pair, (long long)n0, n_pairs};
  if ((e = launch<NoiseBody>(c, (unsigned)(((n0 + 1) / 2 + NT - 1) / NT), (unsigned)(2 * n_pairs), na))) return e;
  RT(rt_d2h(out, c->noise.p, (size_t)n_pairs * 2 * n0 * sizeof(double), c->stream));
  RT(rt_sync(c->stream));
  return 0;
}

// One pass of the last cwtb_cwt_dev transform with a CUDA event pair around every launch.
// Writes one line per kernel type: "name,launches,total_ms,rows" (rows = sum of gridDim.y, i.e.
// scale rows processed) into `out`.  Returns the number of bytes written (<= cap-1) or < 0.
static int profile_report(cwtb_ctx *c, char *out, size_t cap) {
#ifdef CWTB_HOST_EMU
  (void)c;
  if (cap) out[0] = 0;
  return 0;
#else
  RT(rt_sync(c->stream));
  std::map<std::string, std::array<double, 3>> agg;
  std::vector<std::string> order;
  for (auto &r : c->prof) {
    float ms = 0;
    RT(cudaEventElapsedTime(&ms, c->prof_events[r.ev], c->prof_events[r.ev + 1]));
    if (!agg.count(r.name)) order.push_back(r.name);
    auto &a = agg[r.name];
    a[0] += 1; a[1] += ms; a[2] += r.gy;
  }
  std::string txt;
  char line[512];
  for (auto &n : order) {
    auto &a = agg[n];
    snprintf(line, sizeof line, "%s|%d|%.6f|%d\n", n.c_str(), (int)a[0], a[1], (int)a[2]);
    txt += line;
  }
  size_t m = std::min(cap - 1, txt.size());
  memcpy(out, txt.data(), m);
  out[m] = 0;
  return (int)m;
#endif
}

int cwtb_profile_last(cwtb_ctx *c, char *out, size_t cap) {
  if (!c || !c->job.valid || !c->job_dsig || !out || cap < 2) return fail(c, CWTB_ERR_STATE, "no transform to profile");
#ifdef CWTB_HOST_EMU
  out[0] = 0;
  return 0;
#else
  c->prof.clear();
  c->profiling = true;
  const int ts = c->two_streams;
  c->two_streams = 0;   // kernels one after the other: per-kernel times are not blurred by overlap
  int e = timed_run(c, c->job_dsig, 1, nullptr);
  c->two_streams = ts;
  c->profiling = false;
  if (e) return e;
  return profile_report(c, out, cap);
#endif
}

// Profile ANY sequence of calls (xwt, wct, wct_mc, smooth ...): between begin and end every kernel
// launch is bracketed by an event pair and the independent chains run on one stream.
int cwtb_profile_begin(cwtb_ctx *c) {
  if (!c) return CWTB_ERR_ARG;
  c->prof.clear();
  c->profiling = true;
  c->prof_saved_streams = c->two_streams;
  c->two_streams = 0;
  return 0;
}
int cwtb_profile_end(cwtb_ctx *c, char *out, size_t cap) {
  if (!c || !out || cap < 2) return CWTB_ERR_ARG;
  if (!c->profiling) return fail(c, CWTB_ERR_STATE, "profile_end without profile_begin");
  c->profiling = false;
  c->two_streams = c->prof_saved_streams;
  return profile_report(c, out, cap);
}

// Batched transform of independent channels: chunks of channels share every kernel launch
// (one descriptor row per (channel, scale)).  X: host [n_chan][n0].
#ifndef CWTB_HOST_EMU
// Per-row sums of |W|^2 of the resident chunk into dsum (device, R doubles, zeroed by the caller), on
// the engine's stream, no synchronisation.
static int launch_row_power(cwtb_ctx *c, double *dsum) {
  const Job &job = c->job;
  const int R = job.S * job.nbatch;
  const unsigned gx = (unsigned)((job.n0 + PowerBody<double>::PER * NT - 1) / (PowerBody<double>::PER * NT));
  if (job.precision == CWTB_F64) {
    PowerArgs<double> a{(const double2 *)c->W.p, nullptr, dsum, job.n0, nullptr, nullptr, nullptr};
    return launch<PowerBody<double>>(c, gx, R, a);
  }
  PowerArgs<float> a{(const float2 *)c->W.p, nullptr, dsum, job.n0, nullptr, nullptr, nullptr};
  return launch<PowerBody<float>>(c, gx, R, a);
}

// Spectra-only batch: chunk k+1 is copied into page-locked memory and sent to the device while the
// kernels of chunk k run; nothing synchronises until the per-row power of all chunks is read back.
static int cwt_batch_pipelined(cwtb_ctx *c, const void *X, int x_is_f32, int n_chan, int64_t n0, double dt,
                               const double *scales, int n_scales, int family, double param, int precision,
                               double *power_out, int nb) {
  const bool f32 = (precision == CWTB_F32);
  const size_t esz_in = x_is_f32 ? 4 : 8, esz = f32 ? 4 : 8;
  const size_t chunk_bytes = (size_t)nb * n0 * esz;
  int e;
  if (c->stage_bytes < chunk_bytes) {
    RT(rt_sync(c->stream));
    for (auto &p : c->stage_host) {
      if (p) RT(cudaFreeHost(p));
      p = nullptr;
      RT(cudaHostAlloc(&p, chunk_bytes, cudaHostAllocDefault));
    }
    c->stage_bytes = chunk_bytes;
  }
  for (auto &b : c->stage_dev)
    if ((e = ensure(c, b, chunk_bytes))) return e;
  if ((e = ensure(c, c->batch_power, (size_t)n_chan * n_scales * sizeof(double)))) return e;
  double *dpow = (double *)c->batch_power.p;
  rt_stream copy = c->copy_streams[0];
  RT(rt_memset(dpow, 0, (size_t)n_chan * n_scales * sizeof(double), c->stream));
  c->launches = 0;
  bool timing = false;
  int k = 0;
  for (int ch0 = 0; ch0 < n_chan; ch0 += nb, ++k) {
    const int nc = std::min(nb, n_chan - ch0), slot = k & 1;
    // (re-plans only when the chunk geometry changes: first and a shorter last chunk)
    if ((e = prepare(c, n0, dt, scales, n_scales, family, param, precision, nullptr, nc))) return e;
    if (!timing) { RT(cudaEventRecord(c->e0, c->stream)); timing = true; }
    const char *src = (const char *)X + (size_t)ch0 * n0 * esz_in;
    const size_t cnt = (size_t)nc * n0;
    const void *from = src;
    if ((x_is_f32 != 0) != f32) {   // conversion: through the page-locked staging buffer
      if (k >= 2) RT(cudaEventSynchronize(c->ev_h2d[slot]));   // the staging buffer is free again
      if (f32) for (size_t i = 0; i < cnt; ++i) ((float *)c->stage_host[slot])[i] = (float)((const double *)src)[i];
      else for (size_t i = 0; i < cnt; ++i) ((double *)c->stage_host[slot])[i] = (double)((const float *)src)[i];
      from = c->stage_host[slot];
    }
    // (input of the engine's type: straight from the caller's pageable array -- the driver's own staged
    // copy is faster than a host memcpy into page-locked memory plus a DMA, and while it blocks this
    // thread the kernels of the previous chunk keep running)
    if (k >= 2) RT(cudaStreamWaitEvent(copy, c->ev_used[slot], 0));   // chunk k-2 has consumed this device buffer
    RT(cudaMemcpyAsync(c->stage_dev[slot].p, from, cnt * esz, cudaMemcpyHostToDevice, copy));
    RT(cudaEventRecord(c->ev_h2d[slot], copy));
    RT(cudaStreamWaitEvent(c->stream, c->ev_h2d[slot], 0));
    c->job_dsig = c->stage_dev[slot].p;
    c->job.sig_is_f32 = f32;
    e = f32 ? run_job<float>(c, c->job, (const float *)c->stage_dev[slot].p)
            : run_job<double>(c, c->job, (const double *)c->stage_dev[slot].p);
    if (e) return e;
    if ((e = launch_row_power(c, dpow + (size_t)ch0 * n_scales))) return e;
    RT(cudaEventRecord(c->ev_used[slot], c->stream));
  }
  RT(cudaEventRecord(c->e1, c->stream));
  RT(rt_d2h(power_out, dpow, (size_t)n_chan * n_scales * sizeof(double), c->stream));
  RT(rt_sync(c->stream));
  RT(rt_sync(copy));
  float ms = 0;
  RT(cudaEventElapsedTime(&ms, c->e0, c->e1));
  c->last_ms = ms;
  for (size_t i = 0; i < (size_t)n_chan * n_scales; ++i) power_out[i] /= (double)n0;
  return 0;
}
#endif

int cwtb_cwt_batch(cwtb_ctx *c, const void *X, int x_is_f32, int n_chan, int64_t n0, double dt,
                   const double *scales, int n_scales, int family, double param, int precision,
                   double *power_out, void *W_out) {
  if (!c || !X || n_chan < 1 || n0 < 1 || n_scales < 1) return fail(c, CWTB_ERR_ARG, "cwt_batch: bad argument");
  if (family == CWTB_TABLE) return fail(c, CWTB_ERR_UNSUPPORTED, "cwt_batch needs an analytic wavelet family");
  const bool f32 = (precision == CWTB_F32);
  const size_t esz_in = x_is_f32 ? 4 : 8, esz = f32 ? 4 : 8;
  const size_t wrow = (f32 ? 8 : 16) * (size_t)n0;
  // channels per chunk: coefficients of a chunk <= batch_bytes, rows <= 32768
  size_t per_chan = wrow * n_scales;
  int nb = (int)std::max<size_t>(1, std::min<size_t>(c->batch_bytes / std::max<size_t>(per_chan, 1), 32768 / n_scales));
  nb = std::max(1, std::min(nb, n_chan));
#ifndef CWTB_HOST_EMU
  if (c->batch_pipeline && power_out && !W_out && (c->pad_pow2 || (n0 & (n0 - 1)) == 0))
    return cwt_batch_pipelined(c, X, x_is_f32, n_chan, n0, dt, scales, n_scales, family, param, precision, power_out, nb);
#endif
  std::vector<unsigned char> conv;
  for (int ch0 = 0; ch0 < n_chan; ch0 += nb) {
    const int nc = std::min(nb, n_chan - ch0);
    int e = prepare(c, n0, dt, scales, n_scales, family, param, precision, nullptr, nc);
    if (e) return e;
    if ((e = ensure(c, c->sig, (size_t)nc * n0 * esz))) return e;
    const char *src = (const char *)X + (size_t)ch0 * n0 * esz_in;
    if ((x_is_f32 != 0) == f32) {
      RT(rt_h2d(c->sig.p, src, (size_t)nc * n0 * esz, c->stream));
    } else {
      conv.resize((size_t)nc * n0 * esz);
      const size_t cnt = (size_t)nc * n0;
      if (f32) for (size_t i = 0; i < cnt; ++i) ((float *)conv.data())[i] = (float)((const double *)src)[i];
      else for (size_t i = 0; i < cnt; ++i) ((double *)conv.data())[i] = (double)((const float *)src)[i];
      RT(rt_h2d(c->sig.p, conv.data(), conv.size(), c->stream));
    }
    RT(rt_sync(c->stream));
    c->job_dsig = c->sig.p;
    c->job.sig_is_f32 = f32;
    if ((e = timed_run(c, c->sig.p, 1, &c->last_ms))) return e;
    if (power_out && (e = cwtb_global_power(c, power_out + (size_t)ch0 * n_scales))) return e;
    if (W_out && (e = cwtb_get_w(c, (char *)W_out + (size_t)ch0 * per_chan, 0, 0, nc * n_scales))) return e;
  }
  return 0;
}

// Device-resident batched transform for benchmarks: d_X [n_chan][n0] of the engine's real
// type; all channels in one chunk (rows = n_chan * n_scales <= 60000).  W stays on the device
// (cwtb_w_device_ptr), per-row mean power is optionally copied to power_out.
int cwtb_cwt_batch_dev(cwtb_ctx *c, const void *d_X, int n_chan, int64_t n0, double dt, const double *scales,
                       int n_scales, int family, double param, int precision, double *power_out) {
  if (!c || !d_X || n_chan < 1) return fail(c, CWTB_ERR_ARG, "cwt_batch_dev: bad argument");
  if (family == CWTB_TABLE) return fail(c, CWTB_ERR_UNSUPPORTED, "cwt_batch needs an analytic wavelet family");
  int e = prepare(c, n0, dt, scales, n_scales, family, param, precision, nullptr, n_chan);
  if (e) return e;
  c->job_dsig = d_X;
  c->job.sig_is_f32 = (precision == CWTB_F32);
  if ((e = timed_run(c, d_X, 1, &c->last_ms))) return e;
  if (power_out) return cwtb_global_power(c, power_out);
  return 0;
}


// ======================================================================================
// Multi-GPU collectives (SURVEY 8b vii / 8e): one context per GPU and process, an NCCL
// communicator owned by the context.  NCCL is bound at run time (dlopen of libnccl.so.2), so the
// library has no link-time dependency and single-GPU users never touch it.  The data path of the
// transform needs no collective (channels / scales / surrogate pairs are independent); what
// crosses NVLink are the REDUCED products: per-row spectra (all-gather), Monte-Carlo histograms
// (all-reduce), timings (max).  Buffers are host arrays staged through context-owned device
// memory: sizes are O(channels x scales), a few MB.
// ======================================================================================
#ifndef CWTB_HOST_EMU
namespace {
typedef struct { char internal[128]; } nccl_uid;
struct NcclApi {
  void *h = nullptr;
  int (*GetUniqueId)(nccl_uid *) = nullptr;
  int (*CommInitRank)(void **, int, nccl_uid, int) = nullptr;
  int (*CommDestroy)(void *) = nullptr;
  int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
  int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
  int (*Broadcast)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
  bool ok = false;
};
NcclApi &nccl_api() {
  static NcclApi a;
  static std::mutex m;   // contexts of several host threads may bind NCCL at the same time
  std::lock_guard<std::mutex> lock(m);
  if (a.h) return a;
  for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
    a.h = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
    if (a.h) break;
  }
  if (!a.h) return a;
  a.GetUniqueId = (int (*)(nccl_uid *))dlsym(a.h, "ncclGetUniqueId");
  a.CommInitRank = (int (*)(void **, int, nccl_uid, int))dlsym(a.h, "ncclCommInitRank");
  a.CommDestroy = (int (*)(void *))dlsym(a.h, "ncclCommDestroy");
  a.AllGather = (int (*)(const void *, void *, size_t, int, void *, cudaStream_t))dlsym(a.h, "ncclAllGather");
  a.AllReduce = (int (*)(const void *, void *, size_t, int, int, void *, cudaStream_t))dlsym(a.h, "ncclAllReduce");
  a.Broadcast = (int (*)(const void *, void *, size_t, int, int, void *, cudaStream_t))dlsym(a.h, "ncclBroadcast");
  a.GetErrorString = (const char *(*)(int))dlsym(a.h, "ncclGetErrorString");
  a.ok = a.GetUniqueId && a.CommInitRank && a.CommDestroy && a.AllGather && a.AllReduce && a.Broadcast;
  return a;
}
enum { NCCL_CHAR = 0, NCCL_INT64 = 4, NCCL_FLOAT64 = 8, NCCL_SUM = 0, NCCL_MAX = 2 };
}  // namespace
#define NCCLCHK(call)                                                                               \
  do {                                                                                              \
    int r_ = (call);                                                                                \
    if (r_ != 0)                                                                                    \
      return fail(c, CWTB_ERR_COMM, std::string(#call) + ": " +                                     \
                                        (nccl_api().GetErrorString ? nccl_api().GetErrorString(r_) : "NCCL error")); \
  } while (0)
#endif

int cwtb_comm_unique_id(void *id128) {
  if (!id128) return CWTB_ERR_ARG;
#ifdef CWTB_HOST_EMU
  memset(id128, 0, 128);
  return 0;
#else
  NcclApi &a = nccl_api();
  if (!a.ok) return CWTB_ERR_COMM;
  return a.GetUniqueId((nccl_uid *)id128) == 0 ? 0 : CWTB_ERR_COMM;
#endif
}

int cwtb_comm_init(cwtb_ctx *c, int world, int rank, const void *id128) {
  if (!c || !id128 || world < 1 || rank < 0 || rank >= world) return fail(c, CWTB_ERR_ARG, "comm_init: bad argument");
  cwtb_comm_destroy(c);
  c->comm_world = world;
  c->comm_rank = rank;
#ifndef CWTB_HOST_EMU
  if (world == 1) return 0;
  NcclApi &a = nccl_api();
  if (!a.ok) return fail(c, CWTB_ERR_COMM, "libnccl.so.2 could not be loaded");
  RT(cudaSetDevice(c->device));
  nccl_uid id;
  memcpy(&id, id128, sizeof id);
  NCCLCHK(a.CommInitRank(&c->comm, world, id, rank));
#else
  if (world != 1) return fail(c, CWTB_ERR_UNSUPPORTED, "the emulation build has no communicator");
#endif
  return 0;
}

int cwtb_comm_destroy(cwtb_ctx *c) {
  if (!c) return CWTB_ERR_ARG;
#ifndef CWTB_HOST_EMU
  if (c->comm) {
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    nccl_api().CommDestroy(c->comm);
    c->comm = nullptr;
  }
#endif
  c->comm_world = 1;
  c->comm_rank = 0;
  return 0;
}

int cwtb_comm_world(cwtb_ctx *c) { return c ? c->comm_world : -1; }
int cwtb_comm_rank(cwtb_ctx *c) { return c ? c->comm_rank : -1; }

// recv[r * bytes .. (r+1) * bytes) = rank r's send, for every rank (host buffers)
int cwtb_comm_allgather(cwtb_ctx *c, const void *send, void *recv, size_t bytes) {
  if (!c || !send || !recv) return fail(c, CWTB_ERR_ARG, "allgather: null argument");
  if (c->comm_world == 1) { memmove(recv, send, bytes); return 0; }
#ifndef CWTB_HOST_EMU
  int e;
  RT(cudaSetDevice(c->device));
  if ((e = ensure(c, c->comm_send, bytes))) return e;
  if ((e = ensure(c, c->comm_recv, bytes * c->comm_world))) return e;
  RT(rt_h2d(c->comm_send.p, send, bytes, c->stream));
  NCCLCHK(nccl_api().AllGather(c->comm_send.p, c->comm_recv.p, bytes, NCCL_CHAR, c->comm, c->stream));
  RT(rt_d2h(recv, c->comm_recv.p, bytes * c->comm_world, c->stream));
  RT(rt_sync(c->stream));
  return 0;
#else
  return fail(c, CWTB_ERR_UNSUPPORTED, "no communicator");
#endif
}

static int comm_allreduce(cwtb_ctx *c, void *buf, size_t count, int dtype, int op) {
  if (!c || !buf) return fail(c, CWTB_ERR_ARG, "allreduce: null argument");
  if (c->comm_world == 1) return 0;
#ifndef CWTB_HOST_EMU
  int e;
  RT(cudaSetDevice(c->device));
  if ((e = ensure(c, c->comm_send, count * 8))) return e;
  RT(rt_h2d(c->comm_send.p, buf, count * 8, c->stream));
  NCCLCHK(nccl_api().AllReduce(c->comm_send.p, c->comm_send.p, count, dtype, op, c->comm, c->stream));
  RT(rt_d2h(buf, c->comm_send.p, count * 8, c->stream));
  RT(rt_sync(c->stream));
  return 0;
#else
  (void)count; (void)dtype; (void)op;
  return fail(c, CWTB_ERR_UNSUPPORTED, "no communicator");
#endif
}
int cwtb_comm_allreduce_sum_i64(cwtb_ctx *c, int64_t *buf, size_t count) {
#ifndef CWTB_HOST_EMU
  return comm_allreduce(c, buf, count, NCCL_INT64, NCCL_SUM);
#else
  return comm_allreduce(c, buf, count, 0, 0);
#endif
}
int cwtb_comm_allreduce_max_f64(cwtb_ctx *c, double *buf, size_t count) {
#ifndef CWTB_HOST_EMU
  return comm_allreduce(c, buf, count, NCCL_FLOAT64, NCCL_MAX);
#else
  return comm_allreduce(c, buf, count, 0, 0);
#endif
}
int cwtb_comm_broadcast(cwtb_ctx *c, void *buf, size_t bytes, int root) {
  if (!c || !buf || root < 0 || root >= c->comm_world) return fail(c, CWTB_ERR_ARG, "broadcast: bad argument");
  if (c->comm_world == 1) return 0;
#ifndef CWTB_HOST_EMU
  int e;
  RT(cudaSetDevice(c->device));
  if ((e = ensure(c, c->comm_send, bytes))) return e;
  if (c->comm_rank == root) RT(rt_h2d(c->comm_send.p, buf, bytes, c->stream));
  NCCLCHK(nccl_api().Broadcast(c->comm_send.p, c->comm_send.p, bytes, NCCL_CHAR, root, c->comm, c->stream));
  RT(rt_d2h(buf, c->comm_send.p, bytes, c->stream));
  RT(rt_sync(c->stream));
  return 0;
#else
  return fail(c, CWTB_ERR_UNSUPPORTED, "no communicator");
#endif
}

}  // extern "C"
