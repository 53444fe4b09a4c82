// pixsht.cu -- plan object, C ABI (include/pixsht.h) and launch logic of libpixsht.so.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -shared -Xcompiler -fPIC (see build.sh).
#include "common.cuh"
#include "tables.cuh"
#include "legendre.cuh"
#include "legendre_batch.cuh"
#include "legendre_2s.cuh"
#include "fft.cuh"
#include "fft_edge.cuh"
#include "../../include/pixsht.h"

#include <algorithm>
#include <array>
#include <chrono>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>
#ifndef PIXSHT_EMU
#include <sys/mman.h>
#include <sys/syscall.h>
#include <unistd.h>
#endif

using namespace pixsht;

// ---------------------------------------------------------------------------------------------------------------
// error plumbing: every entry point returns a status, the text is kept per host thread; nothing aborts.
// ---------------------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CU(call)                                                                                                      \
    do {                                                                                                              \
        cudaError_t e__ = (call);                                                                                     \
        if (e__ != cudaSuccess)                                                                                       \
            return fail(PIXSHT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));                        \
    } while (0)

// Owner of one device allocation (move-only; freed on destruction).  Allocation happens on the CURRENT device; cudaFree
// finds the owning device through the unified address space.
template <class T>
struct DevBuf {
    T* p = nullptr; size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept { if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; } return *this; }
    ~DevBuf() { release(); }
    int alloc(size_t count)
    {
        release();
        if (count == 0) return PIXSHT_OK;
        if (cudaMalloc((void**)&p, count * sizeof(T)) != cudaSuccess) { p = nullptr; (void)cudaGetLastError(); return PIXSHT_ERR_NOMEM; }
        n = count; return PIXSHT_OK;
    }
    int upload(const std::vector<T>& h)
    {
        int rc = alloc(h.size()); if (rc) return rc;
        if (h.empty()) return PIXSHT_OK;
        return cudaMemcpy(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice) == cudaSuccess ? PIXSHT_OK : PIXSHT_ERR_CUDA;
    }
    void release() { if (p) { if (cudaFree(p) != cudaSuccess) (void)cudaGetLastError(); } p = nullptr; n = 0; }
};

constexpr int PIXSHT_NDEP = 128;
struct pixsht_plan {
    int device = 0, dtype = PIXSHT_F64, sm_count = 0;
    int nphi = 0, nrings = 0, lmax = 0, mmax = 0;
    int nx = 0, ny = 0, flipx = 0, flipy = 0;
    double phi0 = 0;
    long long nalm = 0;
    int npairs = 0;
    int R0 = 4, R2 = 4, R0a = 4, R2a = 4;   // ring pairs per thread in the spin-0 / spin-2 synthesis and analysis kernels
    // FFT
    int nfft = 0, nfac = 0, fac[FFT_MAXFAC] = {0}, fft_threads = 256;
    unsigned fft_magic[FFT_MAXFAC] = {0};
    int nsp = 0; unsigned char sp_first[FFT_MAXFAC] = {0}, sp_count[FFT_MAXFAC] = {0};   // fused super-passes (fft.cuh)
    int nsp_plain = 0; unsigned char sp_first_plain[FFT_MAXFAC] = {0}, sp_count_plain[FFT_MAXFAC] = {0};   // grouping of the launches that run the plain kernels
    size_t fft_smem = 0;
    int fft_packed = 1, fft_pt = FFT_PT;   // even nphi: real ring packed into nphi/2 complex samples; entries per pass table
    int fft_rows = 0;                      // > 0: ring work buffers in global memory, this many CTAs per component (fft.cuh FftParams::gbuf)
    int fft_edge_multi = 0;                // edge-fused kernels also for the m-sharded phase layout (PIXSHT_FFT_EDGE_MULTI)
    int fft_edge = 0;                      // 1: the kernels of fft_edge.cuh (outer super-passes fused into the row I/O; PIXSHT_FFT_EDGE=0 turns it off)
    int fft_persist = 0;                   // > 0 (default; PIXSHT_FFT_PERSIST=0 turns it off): shared-memory FFT CTAs loop over rings, this many
                                           //      resident per SM, and prefetch the next ring's input row into L2 during the passes
    long long fft_gslot = 0; int fft_galt = 0;
    DevBuf<unsigned char> d_fftbuf;
    int seek_thr_log2 = SEEK_THR_LOG2;   // PIXSHT_ACT_LOG2 (experimental) = log2 of the activation threshold, default -90; libsharp2 uses -60
    int batch_overlap = 1;   // host-pointer batches double-buffer their staging so that copies overlap the kernels (PIXSHT_BATCH_OVERLAP=0: one group at a time;
                             // measured on C2x64: 350 -> 193 ms end to end, bit-identical results, profiles/r02)
    bool stage_fam0 = true, stage_fam2 = true;   // spin families the pixsht_stage_* calls process (pixsht_plan_set_stage_families)
    long long MP = 0;             // phase row length (mmax+1 rounded up to a multiple of 8 complex = 128 B)
    // geometry (host copies kept for introspection)
    std::vector<double> h_theta, h_wgt;
    // device tables
    DevBuf<double> d_x, d_lsh_hi, d_lsh_lo, d_lch_hi, d_lch_lo, d_mlim, d_wgt;
    DevBuf<int> d_ringN, d_ringS;
    DevBuf<double> d_lg0_hi, d_lg0_lo, d_lg2_hi, d_lg2_lo;
    DevBuf<double2> d_ad0, d_ad2;          // (alpha, delta) per (l,m)
    DevBuf<double> d_gamma0, d_gamma2;
    DevBuf<double> d_rec0, d_rec2;         // synthesis records, written per call by k_prep_synth
    DevBuf<int> d_lact0, d_lact2;          // activation table: first contributing l per (m, ring pair), built lazily per spin family
    DevBuf<double> d_st0, d_st2;           // recurrence state at l_act
    bool have_seek0 = false, have_seek2 = false;
    // two-step spin-0 sequence (legendre_2s.cuh): tables built on first use
    int twostep = 1;                       // PIXSHT_TWOSTEP=0 turns it off
    int p_eq = 0;                          // first ring pair (pole -> equator) with |cos theta| < TWOSTEP_XMIN: from its chunk on, the standard kernels
    int p_pole = 0;                        // ring pairs within TWOSTEP_POLE_DEG of a pole: their chunks stay with the standard kernels too
    DevBuf<double> d_lg1_hi, d_lg1_lo;     // log2 of the seed prefactor sqrt(2m+3) lambda_mm
    DevBuf<double2> d_ad1, d_wg1;          // (alpha_k, beta_k), (gamma_k c_{l_k+1}, gamma_k c_{l_k+2}) at alm_index(lmax, 0, m) + m + k
    DevBuf<double> d_gam1, d_rec1;         // gamma_k; synthesis records (6 doubles per k)
    DevBuf<int> d_lact1; DevBuf<double> d_st1;
    bool have_seek1 = false;
    DevBuf<double2> d_tw, d_phi0tw;
    DevBuf<unsigned short> d_perm;
    // work buffers (grown on demand)
    DevBuf<double2> d_phase; int phase_ncomp = 0;
    DevBuf<unsigned char> d_map[8], d_alm[8];   // staging of the host paths: components / batch members, two sets for the overlapped batch path
    DevBuf<double2> d_alm64[8];
    cudaStream_t stream = nullptr, own_stream = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t dep[PIXSHT_NDEP] = {nullptr};   // dependency events of the pipelined host path (at most ~45 per call with 8 splits)
    std::vector<int> h_ringN, h_ringS;
    int nsplit = 8;
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t kev[4] = {nullptr, nullptr, nullptr, nullptr};   // around the spin-0 / spin-2 Legendre kernel of the device path
    bool kev_on = false;
    int leg_order = 1;                     // grid order of the Legendre work units (legendre.cuh: leg_unit; PIXSHT_LEG_ORDER)
    int polconv_iau = 0;                   // 1: the caller's U maps follow the IAU sign convention (pixsht_plan_set_polconv)
    double timings[8] = {0};
    int launches = 0;
    std::mutex mu;
    struct pixsht_multi* multi = nullptr;   // non-null: a multi-GPU plan (multi.inl); this object then carries the geometry only
    void* stager = nullptr;                 // pixsht_stage::Stager, created when a call first sees a pageable host array (host_stage.inl)
};
struct pixsht_multi;
static void multi_destroy(pixsht_multi* M);
static void multi_quiesce(pixsht_multi* M);
static pixsht_plan* multi_first_sub(pixsht_multi* M);
static int multi_ndev(const pixsht_multi* M);
static void multi_set_polconv(pixsht_multi* M, int iau);
static int execute_multi(pixsht_plan* P, int direction, int ncomp, void* const* alms, void* const* maps, bool sharded);
static int execute_batch_multi(pixsht_plan* P, int direction, int nbatch, void* const* alms, void* const* maps, int location);

// ---------------------------------------------------------------------------------------------------------------
// small conversion / utility kernels
// ---------------------------------------------------------------------------------------------------------------
__global__ void k_cvt_f32_to_f64(const float* __restrict__ in, double* __restrict__ out, long long n)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long step = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += step) out[i] = (double)in[i];
}
__global__ void k_cvt_f64_to_f32(const double* __restrict__ in, float* __restrict__ out, long long n)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long step = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += step) out[i] = (float)in[i];
}

// the same over the alm columns of the m values m_list[0..nm) (blockIdx.y = position in the list); ZERO: out = 0
template <class TI, class TO, bool ZERO>
__global__ void k_cvt_rows(const int* __restrict__ m_list, int lmax, const TI* __restrict__ in, TO* __restrict__ out)
{
    const int m = m_list[blockIdx.y];
    const long long base = 2 * alm_index(lmax, 0, m);
    for (int i = 2 * m + blockIdx.x * blockDim.x + threadIdx.x; i < 2 * (lmax + 1); i += gridDim.x * blockDim.x)
        out[base + i] = ZERO ? (TO)0 : (TO)in[base + i];
}

#ifndef PIXSHT_EMU
// FMA peak probe: 16 independent accumulators per thread, acc[a][j] += p[j] * g[a] with warp-uniform g (uniform-register
// operand) -> two vector-register reads per FMA, the shape that reaches the pipe's issue rate (tools/dfma_mix.cu: chains with
// constant operands stop at ~34 TFLOP/s FP64 on B200, this shape reaches ~36.7 of the 37.2 TFLOP/s datasheet figure).
// ITER*64 FMAs per thread.
template <class T>
__global__ void __launch_bounds__(256) k_fma_peak(T* out, int iters, const T* __restrict__ in)
{
    T p[4], g[4], acc[4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) p[j] = in[j] + (T)threadIdx.x * (T)1e-9;
#pragma unroll
    for (int a = 0; a < 4; ++a) g[a] = in[8 + a];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[a][j] = (T)0;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[a][j] = fma(p[j], g[a], acc[a][j]);
    }
    T s = (T)0;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int j = 0; j < 4; ++j) s += acc[a][j];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}
#endif

// ---------------------------------------------------------------------------------------------------------------
// plan construction
// ---------------------------------------------------------------------------------------------------------------
static const long double LPI = 3.14159265358979323846264338327950288L;

static void split_dd(long double v, double& hi, double& lo)
{
    if (std::isinf((double)v) || v != v) { hi = (double)v; lo = 0.0; return; }
    hi = (double)v; lo = (double)(v - (long double)hi);
}

static int factorize(int n, int* fac, int& nfac)
{
    nfac = 0;
    if (n == 1) { fac[nfac++] = 1; return 0; }   // a two-sample ring: one trivial pass (handled by the generic-radix branch)
    // pass order = order of fac[] (fft.cuh): odd radices first (largest first), then 4s, then a single 2
    int n2 = 0;
    while (n % 2 == 0) { ++n2; n /= 2; }
    int odd[FFT_MAXFAC], nodd = 0;
    for (int p = 3; n > 1; p += 2) {
        while (n % p == 0) {
            if (nodd >= FFT_MAXFAC) return 1;
            odd[nodd++] = p; n /= p;
        }
        if ((long long)p * p > n && n > 1) {
            if (nodd >= FFT_MAXFAC) return 1;
            odd[nodd++] = n; n = 1;
        }
    }
    // odd radices alternate large / small (5,3,5,3,...) so that neighbours fuse into super-passes of <= 16 points
    for (int lo = 0, hi = nodd - 1; lo <= hi;) { fac[nfac++] = odd[hi--]; if (lo <= hi) fac[nfac++] = odd[lo++]; }
    for (; n2 >= 2; n2 -= 2) { if (nfac >= FFT_MAXFAC) return 1; fac[nfac++] = 4; }
    if (n2 == 1) { if (nfac >= FFT_MAXFAC) return 1; fac[nfac++] = 2; }
    return 0;
}

static int env_int(const char* name, int dflt)
{
    const char* s = getenv(name);
    if (!s || !*s) return dflt;
    return atoi(s);
}

#include "host_stage.inl"

// ---- host-side copies of the host-pointer calls: page-locked arrays go straight to cudaMemcpyAsync, pageable ones through the
// plan's stager (host_stage.inl).  Enqueued on `s` either way. ----
static bool host_is_pageable(const void* p)
{
#ifndef PIXSHT_EMU
    static const int on = env_int("PIXSHT_STAGE", 1);
    return on && pixsht_stage::is_pageable(p);
#else
    (void)p; return false;
#endif
}
constexpr size_t STAGE_MIN_BYTES = 4u << 20;   // smaller copies are left to the driver's own pageable path
static cudaError_t host_copy_in(pixsht_plan* P, bool pageable, void* dst_dev, const void* src_host, size_t n, cudaStream_t s)
{
#ifndef PIXSHT_EMU
    if (pageable && n >= STAGE_MIN_BYTES) {
        if (!P->stager) P->stager = new pixsht_stage::Stager();
        return static_cast<pixsht_stage::Stager*>(P->stager)->h2d(dst_dev, src_host, n, s);
    }
#endif
    (void)P; (void)pageable;
    return cudaMemcpyAsync(dst_dev, src_host, n, cudaMemcpyDefault, s);
}
static cudaError_t host_copy_out(pixsht_plan* P, bool pageable, void* dst_host, const void* src_dev, size_t n, cudaStream_t s)
{
#ifndef PIXSHT_EMU
    if (pageable && n >= STAGE_MIN_BYTES) {
        if (!P->stager) P->stager = new pixsht_stage::Stager();
        return static_cast<pixsht_stage::Stager*>(P->stager)->d2h(dst_host, src_dev, n, s);
    }
#endif
    (void)P; (void)pageable;
    return cudaMemcpyAsync(dst_host, src_dev, n, cudaMemcpyDefault, s);
}
// after the plan's streams have been synchronised: the copy threads have drained everything into the caller's arrays
static void host_copies_done(pixsht_plan* P)
{
#ifndef PIXSHT_EMU
    if (P->stager) static_cast<pixsht_stage::Stager*>(P->stager)->drain_wait();
#else
    (void)P;
#endif
}
static void stager_destroy(pixsht_plan* P)
{
#ifndef PIXSHT_EMU
    if (P->stager) delete static_cast<pixsht_stage::Stager*>(P->stager);
#endif
    P->stager = nullptr;
}

static int plan_build(pixsht_plan* P, const std::vector<double>& theta, const std::vector<double>& wgt_or_empty, int N_cc, int ring_first,
                      int ring_scheme = 0)
{
    const int nr = P->nrings, lmax = P->lmax, mmax = P->mmax;
    P->nalm = pixsht_nalm(lmax, mmax);
    P->h_theta = theta;
    {
        // ring pairs per thread: more pairs amortise the per-step operand loads (DESIGN.md "operand bandwidth") but widen a
        // warp's spread of activation degrees; the wide setting pays off once a chunk is < 5 % of the pairs
        // (with the chunk-major grid order of round 2 the wide setting also wins at 2701 pairs: C3 78.3 -> 77.1 ms)
        const bool wide = (nr + 1) / 2 >= 2048;
        int v = env_int("PIXSHT_R0", wide ? 8 : 4); P->R0 = (v == 1 || v == 2 || v == 3 || v == 4 || v == 6 || v == 8) ? v : 4;
        v = env_int("PIXSHT_R2", wide ? 4 : 2); P->R2 = (v == 1 || v == 2 || v == 3 || v == 4 || v == 6) ? v : 2;
        v = env_int("PIXSHT_R0A", P->R0); P->R0a = (v == 1 || v == 2 || v == 3 || v == 4 || v == 6 || v == 8) ? v : 4;
        v = env_int("PIXSHT_R2A", 4); P->R2a = (v == 1 || v == 2 || v == 3 || v == 4 || v == 6) ? v : 4;
    }

    // ---- north/south pairing (equatorial symmetry): pair rings whose cos(theta) are opposite ----
    std::vector<long double> xs(nr);
    for (int i = 0; i < nr; ++i) xs[i] = cosl((long double)theta[i]);
    std::vector<int> ringN, ringS; std::vector<long double> thn;   // per pair: members and the north colatitude
    {
        std::vector<int> order(nr);
        for (int i = 0; i < nr; ++i) order[i] = i;
        std::sort(order.begin(), order.end(), [&](int a, int b) { return xs[a] > xs[b]; });   // north pole first
        int lo = 0, hi = nr - 1;
        std::vector<char> used(nr, 0);
        while (lo <= hi) {
            const int a = order[lo], b = order[hi];
            if (lo == hi) {
                if (xs[a] >= 0) { ringN.push_back(a); ringS.push_back(-1); thn.push_back((long double)theta[a]); }
                else { ringN.push_back(-1); ringS.push_back(a); thn.push_back(LPI - (long double)theta[a]); }
                break;
            }
            const long double s = xs[a] + xs[b];
            if (fabsl(s) < 1e-12L && xs[a] > 0) { ringN.push_back(a); ringS.push_back(b); thn.push_back((long double)theta[a]); ++lo; --hi; }
            else if (xs[a] >= 0 && (s > 0 || xs[b] >= 0)) { ringN.push_back(a); ringS.push_back(-1); thn.push_back((long double)theta[a]); ++lo; }
            else { ringN.push_back(-1); ringS.push_back(b); thn.push_back(LPI - (long double)theta[b]); --hi; }
        }
        // order pairs by north colatitude so that a warp's pairs are neighbours on the sky
        std::vector<int> po(ringN.size());
        for (size_t i = 0; i < po.size(); ++i) po[i] = (int)i;
        std::sort(po.begin(), po.end(), [&](int a, int b) { return thn[a] < thn[b]; });
        std::vector<int> rn2, rs2; std::vector<long double> th2;
        for (int i : po) { rn2.push_back(ringN[i]); rs2.push_back(ringS[i]); th2.push_back(thn[i]); }
        ringN.swap(rn2); ringS.swap(rs2); thn.swap(th2);
    }
    const int np = (int)ringN.size();
    P->npairs = np;
    std::vector<double> hx(np), lsh_hi(np), lsh_lo(np), lch_hi(np), lch_lo(np), mlim(np);
    const double ofs = std::max(100.0, 0.01 * lmax) + 4.0;
    for (int i = 0; i < np; ++i) {
        const long double t = thn[i];
        hx[i] = (double)cosl(t);
        const long double sh = sinl(0.5L * t), ch = cosl(0.5L * t);
        split_dd(sh > 0 ? log2l(sh) : -HUGE_VALL, lsh_hi[i], lsh_lo[i]);
        split_dd(ch > 0 ? log2l(ch) : -HUGE_VALL, lch_hi[i], lch_lo[i]);
        mlim[i] = (double)lmax * (double)sinl(t) + ofs;   // pairs with m > mlim never reach 2^-90 for l <= lmax (DESIGN.md)
    }

    // ---- seed prefactors per m (long double running sums) ----
    std::vector<double> lg0_hi(mmax + 1), lg0_lo(mmax + 1), lg2_hi(mmax + 1), lg2_lo(mmax + 1);
    {
        // spin 0: lambda_mm = (-1)^m sqrt((2m+1)/(4 pi) prod_{k<=m} (2k-1)/(2k)) (2 sh ch)^m
        long double acc = 0.0L;
        for (int m = 0; m <= mmax; ++m) {
            if (m > 0) acc += log2l((2.0L * m - 1.0L) / (2.0L * m));
            const long double v = 0.5L * (log2l((2.0L * m + 1.0L) / (4.0L * LPI)) + acc) + (long double)m;
            split_dd(v, lg0_hi[m], lg0_lo[m]);
        }
        // spin 2: sqrt((2 l0+1)/(4 pi) (2 l0)!/((l0-q)!(l0+q)!)), l0 = max(m,2), q = min(m,2)
        long double cacc = 0.0L;  // log2 C(2m, m+2), m >= 2
        for (int m = 0; m <= mmax; ++m) {
            long double v;
            if (m < 2) v = 0.5L * (log2l(5.0L / (4.0L * LPI)) + log2l(m == 0 ? 6.0L : 4.0L));
            else {
                if (m > 2) cacc += log2l((2.0L * m) * (2.0L * m - 1.0L) / ((m + 2.0L) * (m - 2.0L)));
                v = 0.5L * (log2l((2.0L * m + 1.0L) / (4.0L * LPI)) + cacc);
            }
            split_dd(v, lg2_hi[m], lg2_lo[m]);
        }
    }

    // two-step spin-0 sequence: seed h_0 = sqrt(2m+3) lambda_mm; chunks that hold pairs with |cos theta| < TWOSTEP_XMIN stay standard
    std::vector<double> lg1_hi(mmax + 1), lg1_lo(mmax + 1);
    for (int m = 0; m <= mmax; ++m) {
        const long double v = (long double)lg0_hi[m] + (long double)lg0_lo[m] + 0.5L * log2l(2.0L * m + 3.0L);
        split_dd(v, lg1_hi[m], lg1_lo[m]);
    }
    P->p_eq = P->npairs;
    for (int i = 0; i < P->npairs; ++i) if (std::fabs(hx[i]) < TWOSTEP_XMIN) { P->p_eq = i; break; }
    for (int i = P->p_eq; i < P->npairs; ++i) if (std::fabs(hx[i]) >= TWOSTEP_XMIN) { P->p_eq = 0; break; }   // pairs not ordered pole -> equator: no two-step chunks
    P->p_pole = 0;
    while (P->p_pole < P->npairs && thn[P->p_pole] < (long double)TWOSTEP_POLE_DEG * LPI / 180.0L) ++P->p_pole;
    P->twostep = env_int("PIXSHT_TWOSTEP", 1) ? 1 : 0;

    // ---- e^{+i m phi0} ----
    std::vector<double2> ph0(mmax + 1);
    for (int m = 0; m <= mmax; ++m) {
        const long double ang = fmodl((long double)m * (long double)P->phi0, 2.0L * LPI);
        ph0[m] = make_double2((double)cosl(ang), (double)sinl(ang));
    }

    // ---- FFT plan ----
    // even nphi: the real ring is one complex FFT of nphi/2 packed samples; odd nphi: a complex FFT of nphi samples with
    // zero imaginary part (no Nyquist mode, no even/odd split)
    P->fft_packed = (P->nphi % 2 == 0) ? 1 : 0;
    P->nfft = P->fft_packed ? P->nphi / 2 : P->nphi;
    if (P->nfft > 65535) return fail(PIXSHT_ERR_UNSUPPORTED, "ring too long: the FFT index tables are 16 bit (nphi <= 131070 even, <= 65535 odd)");
    if (factorize(P->nfft, P->fac, P->nfac)) return fail(PIXSHT_ERR_UNSUPPORTED, "ring length has too many prime factors");
    const size_t elem = (P->dtype == PIXSHT_F64) ? 16 : 8;
    {
        // super-passes: neighbouring radices from {2,3,4,5} whose product is <= PIXSHT_FFT_FUSE (default 16) share one
        // shared-memory round trip
        const int lim = std::min(env_int("PIXSHT_FFT_FUSE", FFT_FUSE_MAX), FFT_FUSE_MAX);
        // Edge-fused kernels (fft_edge.cuh): the last pass stays a single radix (it is done on butterfly pairs in the phase-row
        // I/O), the first super-pass is done in the map-row I/O.  Needs an even ring, radices 2..5 at both ends, no aliasing.
        // Rings below 32 KB (several CTAs of 128 threads per SM) measured no gain (C2, Float32: 0.191 against 0.185 ms): plain kernels,
        // unless PIXSHT_FFT_EDGE=2 forces the edge-fused ones (the emulation tests do, to cover every plan shape at small sizes).
        const int edge_env = env_int("PIXSHT_FFT_EDGE", 1);
        bool edge = P->fft_packed && P->nfac >= 2 && P->mmax <= P->nfft && edge_env != 0 && ((size_t)P->nfft * elem >= 32768 || edge_env == 2)
                    && P->fac[0] >= 2 && P->fac[0] <= 5 && P->fac[P->nfac - 1] >= 2 && P->fac[P->nfac - 1] <= 5;
        const int ngroup = edge ? P->nfac - 1 : P->nfac;   // factors grouped greedily; the edge plan keeps the last one apart
        P->nsp = 0;
        for (int t = 0; t < ngroup;) {
            const bool small = P->fac[t] <= 5 && t + 1 < ngroup && P->fac[t + 1] <= 5;
            const int cnt = (small && P->fac[t] * P->fac[t + 1] <= lim && P->fac[t] * P->fac[t + 1] <= FFT_CST_MAX) ? 2 : 1;
            P->sp_first[P->nsp] = (unsigned char)t; P->sp_count[P->nsp] = (unsigned char)cnt; ++P->nsp; t += cnt;
        }
        if (edge) { P->sp_first[P->nsp] = (unsigned char)(P->nfac - 1); P->sp_count[P->nsp] = 1; ++P->nsp; }
        // launches of an edge plan that run the plain kernels (m-sharded phase layout) group all factors greedily, exactly as a
        // plan created with PIXSHT_FFT_EDGE=0 does: their results are then the same bits
        P->nsp_plain = 0;
        for (int t = 0; t < P->nfac;) {
            const bool small = P->fac[t] <= 5 && t + 1 < P->nfac && P->fac[t + 1] <= 5;
            const int cnt = (small && P->fac[t] * P->fac[t + 1] <= lim && P->fac[t] * P->fac[t + 1] <= FFT_CST_MAX) ? 2 : 1;
            P->sp_first_plain[P->nsp_plain] = (unsigned char)t; P->sp_count_plain[P->nsp_plain] = (unsigned char)cnt; ++P->nsp_plain; t += cnt;
        }
        P->fft_edge = edge ? 1 : 0;
        P->fft_edge_multi = env_int("PIXSHT_FFT_EDGE_MULTI", 0) ? 1 : 0;
        std::vector<double2> cst((FFT_CST_MAX + 1) * FFT_CST_MAX);
        for (int S = 1; S <= FFT_CST_MAX; ++S)
            for (int k = 0; k < S; ++k) { const long double a = 2.0L * LPI * k / S; cst[S * FFT_CST_MAX + k] = make_double2((double)cosl(a), (double)(-sinl(a))); }
        CU(cudaMemcpyToSymbol(c_fft_cst, cst.data(), sizeof(double2) * cst.size()));
    }
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, P->device));
    P->sm_count = prop.multiProcessorCount;
    {
        // Where the ring lives during its FFT.  Default: shared memory (n + 1 samples + tables).  Rings that do not fit, or
        // lengths with a prime factor > FFT_MAXRADIX (whose direct pass works out of place), use per-CTA work buffers in
        // global memory instead: one CTA per SM loops over the rings, the buffers stay L2-resident.
        bool big_prime = false; int Lmax = 1, L = 1;
        for (int i = 0; i < P->nfac; ++i) { if (P->fac[i] > FFT_MAXRADIX) big_prime = true; if (P->fac[i] <= 5) Lmax = std::max(Lmax, L); L *= P->fac[i]; }
        P->fft_smem = (size_t)(P->nfft + 1 + fft_tw_entries(P->nphi) + 4 * FFT_PT) * elem;
        const bool in_smem = !big_prime && P->fft_smem <= prop.sharedMemPerBlockOptin && Lmax <= 128 * (FFT_PT - 128) && !env_int("PIXSHT_FFT_GLOBAL", 0);
        if (!in_smem) P->fft_edge = 0;
        else if (P->fft_edge) {
            const size_t tot = (elem == 16 ? ef_rot_offset<double>(P->nfft, P->nphi, FFT_PT) : ef_rot_offset<float>(P->nfft, P->nphi, FFT_PT))
                               + (size_t)ef_rot_entries(P->mmax) * sizeof(double2);
            if (tot <= prop.sharedMemPerBlockOptin) P->fft_smem = tot;
            else P->fft_edge = 0;
        }
        if (!in_smem) {
            P->fft_pt = 128 + std::max(FFT_PT - 128, (Lmax + 127) / 128);
            P->fft_smem = (size_t)(fft_tw_entries(P->nphi) + 4 * P->fft_pt) * elem;
            P->fft_rows = std::max(1, std::min(nr, P->sm_count));
            P->fft_gslot = ((long long)P->nfft + 1 + 7) / 8 * 8;
            P->fft_galt = big_prime ? 1 : 0;
            const size_t bytes = (size_t)P->fft_rows * 4 * P->fft_gslot * (P->fft_galt ? 2 : 1) * elem;   // up to 4 components per launch
            if (P->d_fftbuf.alloc(bytes)) return fail(PIXSHT_ERR_NOMEM, "FFT work buffer allocation failed");
        }
    }
    {
        // threads per CTA: the multiple of 32 that wastes the fewest thread-iterations over the passes
        // as many CTAs per SM as the shared memory allows (their load / compute / store phases then overlap), threads per CTA
        // scaled down accordingly; among the candidates the multiple of 32 that wastes the fewest thread-iterations
        int ctas = (int)(prop.sharedMemPerMultiprocessor / (P->fft_smem + 1024));
        ctas = std::max(1, std::min(ctas, 4));
        if (P->fft_rows) ctas = 1;   // global-memory work buffers: one large CTA per SM
        else if (env_int("PIXSHT_FFT_PERSIST", 1)) P->fft_persist = ctas;
        const int maxthreads = P->fft_edge ? EF_MAXTHREADS : FFT_MAXTHREADS;
        const int tcap = std::max(64, std::min(maxthreads, (maxthreads / ctas) / 32 * 32));
        const int tmax = std::max(64, std::min(tcap, (P->nfft / 2 + 31) / 32 * 32));
        const int tmin = std::max(64, tmax * 3 / 4 / 32 * 32);
        long long best = -1; int bt = tmax;
        for (int t = tmin; t <= tmax; t += 32) {
            long long cost = 0;
            const int nspc = P->fft_edge ? P->nsp : P->nsp_plain;
            const unsigned char* spf = P->fft_edge ? P->sp_first : P->sp_first_plain;
            const unsigned char* spc = P->fft_edge ? P->sp_count : P->sp_count_plain;
            for (int i = 0; i < nspc; ++i) {
                int pts = P->fac[spf[i]]; if (spc[i] == 2) pts *= P->fac[spf[i] + 1];
                int nb = P->nfft / pts;
                if (P->fft_edge && i == nspc - 1) { nb = (nb - 1) / 2 + 2; pts *= 2; }   // butterfly pairs kk, L - kk
                cost += (long long)((nb + t - 1) / t) * (pts + 2);
            }
            cost = cost * 64 + (tmax - t) / 32;   // ties: prefer more threads
            if (best < 0 || cost < best) { best = cost; bt = t; }
        }
        P->fft_threads = env_int("PIXSHT_FFT_THREADS", bt);
        if (P->fft_threads < 32 || P->fft_threads > maxthreads || P->fft_threads % 32) P->fft_threads = bt;
    }
    std::vector<unsigned short> perm(P->nfft);
    for (int i = 0; i < P->nfft; ++i) perm[i] = (unsigned short)fft_digit_reverse(P->fac, P->nfac, P->nfft, i);
    {
        long long L = 1;
        for (int i = 0; i < P->nfac; ++i) { P->fft_magic[i] = (L == 1) ? 0u : (unsigned)((1ULL << 32) / (unsigned long long)L + 1ULL); L *= P->fac[i]; }
    }
    P->MP = ((long long)P->mmax + 1 + 7) / 8 * 8;

    // ---- upload ----
    int rc = 0;
    rc |= P->d_x.upload(hx); rc |= P->d_lsh_hi.upload(lsh_hi); rc |= P->d_lsh_lo.upload(lsh_lo);
    rc |= P->d_lch_hi.upload(lch_hi); rc |= P->d_lch_lo.upload(lch_lo); rc |= P->d_mlim.upload(mlim);
    rc |= P->d_ringN.upload(ringN); rc |= P->d_ringS.upload(ringS);
    rc |= P->d_lg0_hi.upload(lg0_hi); rc |= P->d_lg0_lo.upload(lg0_lo); rc |= P->d_lg2_hi.upload(lg2_hi); rc |= P->d_lg2_lo.upload(lg2_lo);
    rc |= P->d_lg1_hi.upload(lg1_hi); rc |= P->d_lg1_lo.upload(lg1_lo);
    rc |= P->d_phi0tw.upload(ph0); rc |= P->d_perm.upload(perm);
    rc |= P->d_wgt.alloc(nr); rc |= P->d_tw.alloc(P->nphi);
    rc |= P->d_ad0.alloc(P->nalm); rc |= P->d_gamma0.alloc(P->nalm);
    rc |= P->d_ad2.alloc(P->nalm); rc |= P->d_gamma2.alloc(P->nalm);
    if (rc) return fail(PIXSHT_ERR_NOMEM, "device allocation of plan tables failed");

    CU(cudaStreamCreateWithFlags(&P->own_stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&P->s_h2d, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&P->s_d2h, cudaStreamNonBlocking));
    for (auto& e : P->dep) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    P->h_ringN = ringN; P->h_ringS = ringS;
    { int v = env_int("PIXSHT_SPLITS", 8); P->nsplit = (v >= 1 && v <= 8) ? v : 8; }
    P->batch_overlap = env_int("PIXSHT_BATCH_OVERLAP", 1) ? 1 : 0;
    { const int v = env_int("PIXSHT_LEG_ORDER", 1); P->leg_order = v >= 0 ? v : 1; }   // chunk-major by default (measured, profiles/r02/legbench_order*.txt)
    { const int a = env_int("PIXSHT_ACT_LOG2", ACT_LOG2); P->seek_thr_log2 = (a <= -40 && a >= -200) ? a + SEEK_QUANT : SEEK_THR_LOG2; }
    P->stream = P->own_stream;
    for (auto& e : P->ev) CU(cudaEventCreate(&e));
    for (auto& e : P->kev) CU(cudaEventCreate(&e));

    // ---- device-side precompute ----
    if (wgt_or_empty.empty()) {
        if (ring_scheme == PIXSHT_RINGS_FEJER1) PIXSHT_LAUNCH(k_fejer1_weights, (nr + 127) / 128, 128, 0, P->stream, N_cc, P->nphi, ring_first, nr, P->d_wgt.p);
        else PIXSHT_LAUNCH(k_cc_weights, (nr + 127) / 128, 128, 0, P->stream, N_cc, P->nphi, ring_first, nr, P->d_wgt.p);
    } else {
        CU(cudaMemcpyAsync(P->d_wgt.p, wgt_or_empty.data(), sizeof(double) * nr, cudaMemcpyHostToDevice, P->stream));
    }
    PIXSHT_LAUNCH(k_twiddles, (P->nphi + 127) / 128, 128, 0, P->stream, P->nphi, P->d_tw.p);
    PIXSHT_LAUNCH(k_coef_tables, (mmax + 64) / 64, 64, 0, P->stream, lmax, mmax, 0, P->d_ad0.p, P->d_gamma0.p);
    PIXSHT_LAUNCH(k_coef_tables, (mmax + 64) / 64, 64, 0, P->stream, lmax, mmax, 2, P->d_ad2.p, P->d_gamma2.p);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(P->stream));
    P->h_wgt.resize(nr);
    CU(cudaMemcpy(P->h_wgt.data(), P->d_wgt.p, sizeof(double) * nr, cudaMemcpyDeviceToHost));

#ifndef PIXSHT_EMU
    // Opt in to large dynamic shared memory: the cap is a per-function attribute shared by every plan of the process, so it is
    // set to the device maximum once and for all (a plan-sized cap would be lowered by the next, smaller plan and break the
    // launches of the larger one); what a launch actually reserves is its own fft_smem.
    {
        const int cap = (int)prop.sharedMemPerBlockOptin;
        CU(cudaFuncSetAttribute(fft_phase2map<double, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
        CU(cudaFuncSetAttribute(fft_map2phase<double, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
        CU(cudaFuncSetAttribute(fft_phase2map<double, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
        CU(cudaFuncSetAttribute(fft_map2phase<double, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
        CU(cudaFuncSetAttribute(fft_phase2map<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
        CU(cudaFuncSetAttribute(fft_map2phase<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
        CU(cudaFuncSetAttribute(fft_phase2map<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
        CU(cudaFuncSetAttribute(fft_map2phase<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
        CU(cudaFuncSetAttribute(fft_phase2map_edge<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
        CU(cudaFuncSetAttribute(fft_map2phase_edge<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
        CU(cudaFuncSetAttribute(fft_phase2map_edge<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
        CU(cudaFuncSetAttribute(fft_map2phase_edge<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
    }
#endif
    return PIXSHT_OK;
}

static int check_device(int device)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        (void)cudaGetLastError();
        return fail(PIXSHT_ERR_NODEVICE, "no CUDA device available: libpixsht has no CPU fallback");
    }
    if (device < 0 || device >= n) return fail(PIXSHT_ERR_ARG, "device index out of range");
    if (cudaSetDevice(device) != cudaSuccess) return fail(PIXSHT_ERR_CUDA, "cudaSetDevice failed");
    return PIXSHT_OK;
}

extern "C" int64_t pixsht_nalm(int lmax, int mmax)
{
    return (int64_t)(mmax + 1) * (lmax + 1) - (int64_t)mmax * (mmax + 1) / 2;
}

extern "C" int pixsht_plan_create(pixsht_plan** out, const pixsht_geom* g, int lmax, int mmax, int dtype, int device)
{
    if (!out || !g) return fail(PIXSHT_ERR_ARG, "null argument");
    *out = nullptr;
    if (lmax < 0 || mmax < 0 || mmax > lmax) return fail(PIXSHT_ERR_ARG, "need 0 <= mmax <= lmax");
    if (dtype != PIXSHT_F64 && dtype != PIXSHT_F32) return fail(PIXSHT_ERR_ARG, "dtype must be PIXSHT_F64 or PIXSHT_F32");
    if (g->nphi < 2 || g->nrings_total < 2 || g->nrings < 1 || g->ring_first < 0 || g->ring_first + g->nrings > g->nrings_total)
        return fail(PIXSHT_ERR_ARG, "inconsistent ring geometry");
    if (g->ring_scheme != PIXSHT_RINGS_CC && g->ring_scheme != PIXSHT_RINGS_FEJER1) return fail(PIXSHT_ERR_ARG, "unknown ring scheme");
    if (g->nx < 1 || g->nx > g->nphi) return fail(PIXSHT_ERR_ARG, "need 1 <= nx <= nphi");
    int rc = check_device(device); if (rc) return rc;
    pixsht_plan* P = new pixsht_plan();
    P->device = device; P->dtype = dtype; P->nphi = g->nphi; P->nrings = g->nrings; P->lmax = lmax; P->mmax = mmax;
    P->nx = g->nx; P->ny = g->nrings; P->flipx = g->flipx != 0; P->flipy = g->flipy != 0; P->phi0 = g->phi0;
    // theta_k = pi k/(N-1) rounded to double, as range(0, pi, length=N)[k] gives the reference (src/transforms.jl:46)
    // Fejer-1: theta_k = pi (k + 1/2)/N, no ring on the poles
    std::vector<double> theta(g->nrings);
    for (int i = 0; i < g->nrings; ++i)
        theta[i] = g->ring_scheme == PIXSHT_RINGS_FEJER1
                       ? (double)(LPI * ((long double)(g->ring_first + i) + 0.5L) / (long double)g->nrings_total)
                       : (double)(LPI * (long double)(g->ring_first + i) / (long double)(g->nrings_total - 1));
    rc = plan_build(P, theta, std::vector<double>(), g->nrings_total, g->ring_first, g->ring_scheme);
    if (rc) { std::string keep = g_err; pixsht_plan_destroy(P); g_err = keep; return rc; }
    *out = P;
    return PIXSHT_OK;
}

extern "C" int pixsht_plan_create_rings(pixsht_plan** out, int nrings, const double* theta, const double* weight, int nphi,
                                        double phi0, int lmax, int mmax, int dtype, int device)
{
    if (!out || !theta || !weight) return fail(PIXSHT_ERR_ARG, "null argument");
    *out = nullptr;
    if (lmax < 0 || mmax < 0 || mmax > lmax) return fail(PIXSHT_ERR_ARG, "need 0 <= mmax <= lmax");
    if (dtype != PIXSHT_F64 && dtype != PIXSHT_F32) return fail(PIXSHT_ERR_ARG, "dtype must be PIXSHT_F64 or PIXSHT_F32");
    if (nrings < 1 || nphi < 2) return fail(PIXSHT_ERR_ARG, "inconsistent ring geometry");
    for (int i = 0; i < nrings; ++i)
        if (!(theta[i] >= 0.0 && theta[i] <= 3.1415926535897936)) return fail(PIXSHT_ERR_ARG, "theta outside [0, pi]");
    int rc = check_device(device); if (rc) return rc;
    pixsht_plan* P = new pixsht_plan();
    P->device = device; P->dtype = dtype; P->nphi = nphi; P->nrings = nrings; P->lmax = lmax; P->mmax = mmax;
    P->nx = nphi; P->ny = nrings; P->flipx = 0; P->flipy = 0; P->phi0 = phi0;
    std::vector<double> th(theta, theta + nrings), w(weight, weight + nrings);
    rc = plan_build(P, th, w, 0, 0);
    if (rc) { std::string keep = g_err; pixsht_plan_destroy(P); g_err = keep; return rc; }
    *out = P;
    return PIXSHT_OK;
}

extern "C" void pixsht_plan_destroy(pixsht_plan* P)
{
    if (!P) return;
    if (P->multi) { multi_destroy(P->multi); P->multi = nullptr; delete P; return; }
    // may run from a GC finalizer thread, possibly after the CUDA context is gone: every call below tolerates failure
    (void)cudaSetDevice(P->device);
    if (P->s_h2d) (void)cudaStreamSynchronize(P->s_h2d);
    if (P->s_d2h) (void)cudaStreamSynchronize(P->s_d2h);
    stager_destroy(P);
    P->d_x.release(); P->d_lsh_hi.release(); P->d_lsh_lo.release(); P->d_lch_hi.release(); P->d_lch_lo.release();
    P->d_mlim.release(); P->d_wgt.release(); P->d_ringN.release(); P->d_ringS.release();
    P->d_lg0_hi.release(); P->d_lg0_lo.release(); P->d_lg2_hi.release(); P->d_lg2_lo.release();
    P->d_ad0.release(); P->d_gamma0.release(); P->d_ad2.release(); P->d_gamma2.release(); P->d_rec0.release(); P->d_rec2.release();
    P->d_tw.release(); P->d_phi0tw.release(); P->d_phase.release(); P->d_perm.release(); P->d_fftbuf.release();
    P->d_lact0.release(); P->d_lact2.release(); P->d_st0.release(); P->d_st2.release();
    P->d_lg1_hi.release(); P->d_lg1_lo.release(); P->d_ad1.release(); P->d_wg1.release(); P->d_gam1.release(); P->d_rec1.release();
    P->d_lact1.release(); P->d_st1.release();
    for (int c = 0; c < 8; ++c) { P->d_map[c].release(); P->d_alm[c].release(); P->d_alm64[c].release(); }
    for (auto& e : P->ev) if (e) cudaEventDestroy(e);
    for (auto& e : P->kev) if (e) cudaEventDestroy(e);
    for (auto& e : P->dep) if (e) cudaEventDestroy(e);
    if (P->s_h2d) cudaStreamDestroy(P->s_h2d);
    if (P->s_d2h) cudaStreamDestroy(P->s_d2h);
    if (P->own_stream) cudaStreamDestroy(P->own_stream);
    (void)cudaGetLastError();
    delete P;
}

// ---------------------------------------------------------------------------------------------------------------
// stage launches
// ---------------------------------------------------------------------------------------------------------------
// The activation table of one spin family (legendre.cuh, k_seek_table): built on first use, kept for the plan's lifetime.
static int ensure_seek(pixsht_plan* P, int spin, cudaStream_t st)
{
    bool& have = spin == 0 ? P->have_seek0 : P->have_seek2;
    if (have) return PIXSHT_OK;
    DevBuf<int>& lact = spin == 0 ? P->d_lact0 : P->d_lact2;
    DevBuf<double>& stt = spin == 0 ? P->d_st0 : P->d_st2;
    const size_t n = (size_t)(P->mmax + 1) * P->npairs;
    if (lact.alloc(n) || stt.alloc(n * (spin == 0 ? 2 : 4))) return fail(PIXSHT_ERR_NOMEM, "activation table allocation failed");
    SeekParams K;
    memset(&K, 0, sizeof(K));
    K.lmax = P->lmax; K.mmax = P->mmax; K.npairs = P->npairs; K.x = P->d_x.p;
    K.lsh_hi = P->d_lsh_hi.p; K.lsh_lo = P->d_lsh_lo.p; K.lch_hi = P->d_lch_hi.p; K.lch_lo = P->d_lch_lo.p; K.mlim = P->d_mlim.p;
    if (spin == 0) { K.lgpref_hi = P->d_lg0_hi.p; K.lgpref_lo = P->d_lg0_lo.p; K.ad = P->d_ad0.p; }
    else { K.lgpref_hi = P->d_lg2_hi.p; K.lgpref_lo = P->d_lg2_lo.p; K.ad = P->d_ad2.p; }
    K.lact = lact.p; K.st = stt.p;
    K.thr_log2 = P->seek_thr_log2;
    dim3 grid((P->npairs + 127) / 128, P->mmax + 1);
    if (spin == 0) PIXSHT_LAUNCH(k_seek_table<0>, grid, 128, 0, st, K);
    else PIXSHT_LAUNCH(k_seek_table<2>, grid, 128, 0, st, K);
    CU(cudaGetLastError());
    have = true;
    return PIXSHT_OK;
}

// Tables of the two-step spin-0 sequence (legendre_2s.cuh): coefficients and activation table, built on first use.
static int ensure_twostep(pixsht_plan* P, cudaStream_t st)
{
    if (P->have_seek1) return PIXSHT_OK;
    const size_t n = (size_t)(P->mmax + 1) * P->npairs;
    if (P->d_ad1.alloc(P->nalm) || P->d_wg1.alloc(P->nalm) || P->d_gam1.alloc(P->nalm) || P->d_lact1.alloc(n) || P->d_st1.alloc(n * 2))
        return fail(PIXSHT_ERR_NOMEM, "two-step table allocation failed");
    PIXSHT_LAUNCH(k_coef_tables_2s, (P->mmax + 64) / 64, 64, 0, st, P->lmax, P->mmax, P->d_ad1.p, P->d_wg1.p, P->d_gam1.p);
    SeekParams K;
    memset(&K, 0, sizeof(K));
    K.lmax = P->lmax; K.mmax = P->mmax; K.npairs = P->npairs; K.x = P->d_x.p;
    K.lsh_hi = P->d_lsh_hi.p; K.lsh_lo = P->d_lsh_lo.p; K.lch_hi = P->d_lch_hi.p; K.lch_lo = P->d_lch_lo.p; K.mlim = P->d_mlim.p;
    K.lgpref_hi = P->d_lg1_hi.p; K.lgpref_lo = P->d_lg1_lo.p; K.ad = P->d_ad1.p;
    K.lact = P->d_lact1.p; K.st = P->d_st1.p;
    K.thr_log2 = P->seek_thr_log2;
    dim3 grid((P->npairs + 127) / 128, P->mmax + 1);
    PIXSHT_LAUNCH(k_seek_table_2s, grid, 128, 0, st, K);
    CU(cudaGetLastError());
    P->have_seek1 = true;
    return PIXSHT_OK;
}
// Chunks [lo, hi) (of 32 R pairs, pole -> equator) take the two-step spin-0 kernels; the polar chunk(s) and the equatorial one(s)
// stay with the standard kernels (accuracy, legendre_2s.cuh).  hi <= lo: no two-step chunks (small maps).
static void twostep_range(const pixsht_plan* P, int R, int& lo, int& hi)
{
    lo = (P->p_pole + 32 * R - 1) / (32 * R);
    hi = P->twostep ? P->p_eq / (32 * R) : 0;
    if (hi <= lo) { lo = 0; hi = 0; }
}
static bool twostep_any(const pixsht_plan* P, int R) { int lo, hi; twostep_range(P, R, lo, hi); return hi > lo; }

// where the phase rows of a Legendre launch live: ring r at phase + r*ncomp*MP; columns are m (single GPU) or launch rows (m-sharded)
struct PhaseRef { double2* phase; long long MP; int col_is_row; };   // MP = 0: the plan's own row length

// one Legendre launch: m values [m_begin, m_begin+nm) (or m_list[0..nm)), chunks [chunk_begin, chunk_begin+nchunks) of 32*R pairs
struct LegJob { int spin, ncomp, c0; int m_begin, nm; const int* m_list; int chunk_begin, nchunks; PhaseRef ph; };

static int leg_R(const pixsht_plan* P, int spin, bool anal) { return spin == 0 ? (anal ? P->R0a : P->R0) : (anal ? P->R2a : P->R2); }
static int leg_total_chunks(const pixsht_plan* P, int R) { return (P->npairs + 32 * R - 1) / (32 * R); }

static LegParams leg_params(pixsht_plan* P, const LegJob& J, int R)
{
    LegParams L;
    memset(&L, 0, sizeof(L));
    L.lmax = P->lmax; L.mmax = P->mmax; L.nm = J.nm; L.m_list = J.m_list; L.m_begin = J.m_begin;
    L.npairs = P->npairs; L.nchunks = J.nchunks; L.chunk_begin = J.chunk_begin;
    L.x = P->d_x.p; L.ringN = P->d_ringN.p; L.ringS = P->d_ringS.p;
    if (J.spin == 0) { L.lact = P->d_lact0.p; L.st = P->d_st0.p; L.ad = P->d_ad0.p; L.gamma = P->d_gamma0.p; L.rec = P->d_rec0.p; }
    else { L.lact = P->d_lact2.p; L.st = P->d_st2.p; L.ad = P->d_ad2.p; L.gamma = P->d_gamma2.p; L.rec = P->d_rec2.p; }
    L.MP = J.ph.MP > 0 ? J.ph.MP : P->MP; L.col_is_row = J.ph.col_is_row;
    L.phase = J.ph.phase; L.ring_stride = (long long)J.ncomp * L.MP; L.c0 = J.c0;
    L.order = P->leg_order;
    return L;
}
// the same launch on the tables of the two-step spin-0 sequence (legendre_2s.cuh); anal: `rec` carries the output weights
static LegParams leg_params_2s(pixsht_plan* P, const LegJob& J, int R, bool anal)
{
    LegParams L = leg_params(P, J, R);
    L.lact = P->d_lact1.p; L.st = P->d_st1.p; L.ad = P->d_ad1.p; L.gamma = P->d_gam1.p;
    L.rec = anal ? reinterpret_cast<const double*>(P->d_wg1.p) : P->d_rec1.p;
    return L;
}
template <int R> static void launch_2s(bool anal, int grid, const LegParams& L, cudaStream_t st)
{
    if (anal) PIXSHT_LAUNCH(leg_anal_2s<R>, grid, LEG_NT, 0, st, L);
    else PIXSHT_LAUNCH(leg_synth_2s<R>, grid, LEG_NT, 0, st, L);
}
static void launch_twostep(pixsht_plan* P, bool anal, int R, const LegParams& L, cudaStream_t st)
{
    const int grid = L.nm * L.nchunks;
    if (grid <= 0) return;
    switch (R) {
        case 1: launch_2s<1>(anal, grid, L, st); break;
        case 2: launch_2s<2>(anal, grid, L, st); break;
        case 3: launch_2s<3>(anal, grid, L, st); break;
        case 6: launch_2s<6>(anal, grid, L, st); break;
        case 8: launch_2s<8>(anal, grid, L, st); break;
        default: launch_2s<4>(anal, grid, L, st); break;
    }
    P->launches++;
}
// m range [ma, mb) whose alm columns are exactly the index range [first, first + count) (the callers pass whole columns)
static void alm_range_to_m(const pixsht_plan* P, long long first, long long count, int& ma, int& mb)
{
    auto col = [&](int m) { return m > P->mmax ? P->nalm : alm_index(P->lmax, m, m); };
    ma = 0;
    while (ma <= P->mmax && col(ma) < first) ++ma;
    mb = ma;
    while (mb <= P->mmax && col(mb) < first + count) ++mb;
}

template <int SPIN>
static void launch_synth(pixsht_plan* P, int R, const LegParams& L, cudaStream_t st)
{
    const int grid = L.nm * L.nchunks;
    if (grid <= 0) return;
    void (*k)(const LegParams) = (R == 1) ? leg_synth<SPIN, 1> : (R == 2 ? leg_synth<SPIN, 2> : (R == 3 ? leg_synth<SPIN, 3> :
                                 (R == 8 && SPIN == 0 ? leg_synth<0, 8> : (R == 6 ? leg_synth<SPIN, 6> : leg_synth<SPIN, 4>))));
    PIXSHT_LAUNCH(k, grid, LEG_NT, 0, st, L);
    P->launches++;
}
template <int SPIN>
static void launch_anal(pixsht_plan* P, int R, const LegParams& L, cudaStream_t st)
{
    const int grid = L.nm * L.nchunks;
    if (grid <= 0) return;
    void (*k)(const LegParams) = (R == 1) ? leg_anal<SPIN, 1> : (R == 2 ? leg_anal<SPIN, 2> : (R == 3 ? leg_anal<SPIN, 3> :
                                 (R == 8 && SPIN == 0 ? leg_anal<0, 8> : (R == 6 ? leg_anal<SPIN, 6> : leg_anal<SPIN, 4>))));
    PIXSHT_LAUNCH(k, grid, LEG_NT, 0, st, L);
    P->launches++;
}

// per-call pre-scaling of the alm of one spin family into the synthesis records: over the alm index range [first, first+count)
// (m_list == nullptr), or over the columns of the m values m_list[0..nm) -- the m-sharded pipelines prepare only the columns a
// launch owns and that have arrived
static int synth_prep(pixsht_plan* P, int spin, const double2* a0, const double2* a1, cudaStream_t st, long long first = 0, long long count = -1,
                      const int* m_list = nullptr, int nm = 0)
{
    if (!m_list) {
        if (count < 0) count = P->nalm - first;
        if (count <= 0) return PIXSHT_OK;
    } else if (nm <= 0) return PIXSHT_OK;
    const int prep_grid = P->sm_count > 0 ? P->sm_count * 8 : 256;
    const dim3 row_grid((unsigned)std::max(1, std::min(8, (P->lmax + 256) / 256)), (unsigned)std::max(nm, 1));
    int rc = ensure_seek(P, spin, st); if (rc) return rc;
    if (spin == 0) {
        if (P->d_rec0.n < (size_t)P->nalm * 4 && P->d_rec0.alloc((size_t)P->nalm * 4)) return fail(PIXSHT_ERR_NOMEM, "record buffer allocation failed");
        if (m_list) PIXSHT_LAUNCH(k_prep_synth_rows<0>, row_grid, 256, 0, st, m_list, P->lmax, P->d_ad0.p, P->d_gamma0.p, a0, a0, P->d_rec0.p);
        else PIXSHT_LAUNCH(k_prep_synth<0>, prep_grid, 256, 0, st, first, count, P->lmax, P->d_ad0.p, P->d_gamma0.p, a0, a0, P->d_rec0.p);
        if (twostep_any(P, P->R0)) {
            // the records of the two-step kernels for the same columns
            rc = ensure_twostep(P, st); if (rc) return rc;
            if (P->d_rec1.n < (size_t)P->nalm * 6 && P->d_rec1.alloc((size_t)P->nalm * 6)) return fail(PIXSHT_ERR_NOMEM, "record buffer allocation failed");
            int ma = 0, mb = nm;
            if (!m_list) alm_range_to_m(P, first, count, ma, mb);
            if (mb > ma) {
                const dim3 g2((unsigned)std::max(1, std::min(8, (P->lmax / 2 + 256) / 256)), (unsigned)(mb - ma));
                PIXSHT_LAUNCH(k_prep_synth_2s, g2, 256, 0, st, m_list, ma, P->lmax, P->d_ad1.p, P->d_wg1.p, P->d_gam1.p, a0, P->d_rec1.p);
                P->launches++;
            }
        }
    } else {
        if (P->d_rec2.n < (size_t)P->nalm * 6 && P->d_rec2.alloc((size_t)P->nalm * 6)) return fail(PIXSHT_ERR_NOMEM, "record buffer allocation failed");
        if (m_list) PIXSHT_LAUNCH(k_prep_synth_rows<2>, row_grid, 256, 0, st, m_list, P->lmax, P->d_ad2.p, P->d_gamma2.p, a0, a1, P->d_rec2.p);
        else PIXSHT_LAUNCH(k_prep_synth<2>, prep_grid, 256, 0, st, first, count, P->lmax, P->d_ad2.p, P->d_gamma2.p, a0, a1, P->d_rec2.p);
    }
    P->launches++;
    CU(cudaGetLastError());
    return PIXSHT_OK;
}
// Profiling aid for tools/loop_eff.py, compiled in only with -DPIXSHT_PROBES (results are then WRONG by design):
// PIXSHT_DBG_NM / PIXSHT_DBG_CHUNKS restrict a launch to the first NM m values and the CHUNKS equator-most chunks, where
// every ring is active for almost the whole l range -> pure inner-loop throughput.
static void dbg_restrict(LegParams& L)
{
#ifdef PIXSHT_PROBES
    const int nm = env_int("PIXSHT_DBG_NM", 0), nc = env_int("PIXSHT_DBG_CHUNKS", 0);
    if (nm > 0 && nm < L.nm) L.nm = nm;
    if (nc > 0 && nc < L.nchunks) { L.chunk_begin += L.nchunks - nc; L.nchunks = nc; }
#else
    (void)L;
#endif
}

static int synth_launch(pixsht_plan* P, const LegJob& J, cudaStream_t st)
{
    if (J.nm <= 0 || J.nchunks <= 0) return PIXSHT_OK;   // an empty piece of a split
    const int R = leg_R(P, J.spin, false);
    LegParams L = leg_params(P, J, R);
    dbg_restrict(L);
    if (P->kev_on) CU(cudaEventRecord(P->kev[J.spin == 0 ? 0 : 2], st));
    if (J.spin == 0) {
        // the chunks of the launch that lie in [lo, hi) go through the two-step kernels, the polar and equatorial rest through the standard ones
        int lo, hi; twostep_range(P, R, lo, hi);
        const int cb = L.chunk_begin, ce = L.chunk_begin + L.nchunks;
        const int t0 = std::max(cb, lo), t1 = std::min(ce, hi);
        if (t1 > t0) {
            LegParams L2 = leg_params_2s(P, J, R, false);
            L2.nm = L.nm; L2.chunk_begin = t0; L2.nchunks = t1 - t0;
            launch_twostep(P, false, R, L2, st);
            if (t0 > cb) { LegParams La = L; La.chunk_begin = cb; La.nchunks = t0 - cb; launch_synth<0>(P, R, La, st); }
            if (ce > t1) { LegParams Lb = L; Lb.chunk_begin = t1; Lb.nchunks = ce - t1; launch_synth<0>(P, R, Lb, st); }
        } else launch_synth<0>(P, R, L, st);
    } else launch_synth<2>(P, R, L, st);
    if (P->kev_on) CU(cudaEventRecord(P->kev[J.spin == 0 ? 1 : 3], st));
    CU(cudaGetLastError());
    return PIXSHT_OK;
}
static int anal_launch(pixsht_plan* P, const LegJob& J, double2* out0, double2* out1, cudaStream_t st)
{
    if (J.nm <= 0 || J.nchunks <= 0) return PIXSHT_OK;   // an empty piece of a split
    int rc = ensure_seek(P, J.spin, st); if (rc) return rc;
    const int R = leg_R(P, J.spin, true);
    LegParams L = leg_params(P, J, R);
    dbg_restrict(L);
    L.alm_out0 = out0; L.alm_out1 = out1;
    if (P->kev_on) CU(cudaEventRecord(P->kev[J.spin == 0 ? 0 : 2], st));
    if (J.spin == 0) {
        int lo, hi; twostep_range(P, R, lo, hi);
        const int cb = L.chunk_begin, ce = L.chunk_begin + L.nchunks;
        const int t0 = std::max(cb, lo), t1 = std::min(ce, hi);
        if (t1 > t0) {
            rc = ensure_twostep(P, st); if (rc) return rc;
            LegParams L2 = leg_params_2s(P, J, R, true);
            L2.alm_out0 = out0;
            L2.nm = L.nm; L2.chunk_begin = t0; L2.nchunks = t1 - t0;
            launch_twostep(P, true, R, L2, st);
            if (t0 > cb) { LegParams La = L; La.chunk_begin = cb; La.nchunks = t0 - cb; launch_anal<0>(P, R, La, st); }
            if (ce > t1) { LegParams Lb = L; Lb.chunk_begin = t1; Lb.nchunks = ce - t1; launch_anal<0>(P, R, Lb, st); }
        } else launch_anal<0>(P, R, L, st);
    } else launch_anal<2>(P, R, L, st);
    if (P->kev_on) CU(cudaEventRecord(P->kev[J.spin == 0 ? 1 : 3], st));
    CU(cudaGetLastError());
    return PIXSHT_OK;
}

// alm component layout per ncomp: ncomp 1: [T]; 2: [E,B]; 3: [T,E,B].  phase/map components likewise [T] / [Q,U] / [T,Q,U].
static int stage_alm2phase(pixsht_plan* P, int ncomp, const double2* const* alm, int nm, const int* d_m_list, PhaseRef ph, cudaStream_t st,
                           bool fam0 = true, bool fam2 = true)
{
    if ((ncomp == 1 || ncomp == 3) && fam0) {
        int rc = synth_prep(P, 0, alm[0], alm[0], st, 0, d_m_list ? -1 : alm_index(P->lmax, nm, nm), d_m_list, nm); if (rc) return rc;
        const LegJob J = {0, ncomp, 0, 0, nm, d_m_list, 0, leg_total_chunks(P, P->R0), ph};
        rc = synth_launch(P, J, st); if (rc) return rc;
    }
    if (ncomp >= 2 && fam2) {
        const int c0 = ncomp == 3 ? 1 : 0;
        int rc = synth_prep(P, 2, alm[c0], alm[c0 + 1], st, 0, d_m_list ? -1 : alm_index(P->lmax, nm, nm), d_m_list, nm); if (rc) return rc;
        const LegJob J = {2, ncomp, c0, 0, nm, d_m_list, 0, leg_total_chunks(P, P->R2), ph};
        rc = synth_launch(P, J, st); if (rc) return rc;
    }
    return PIXSHT_OK;
}

static int stage_phase2alm(pixsht_plan* P, int ncomp, PhaseRef ph, int nm, const int* d_m_list, double2* const* alm, cudaStream_t st,
                           bool fam0 = true, bool fam2 = true)
{
    if ((ncomp == 1 || ncomp == 3) && fam0) {
        const LegJob J = {0, ncomp, 0, 0, nm, d_m_list, 0, leg_total_chunks(P, P->R0a), ph};
        int rc = anal_launch(P, J, alm[0], nullptr, st); if (rc) return rc;
    }
    if (ncomp >= 2 && fam2) {
        const int c0 = ncomp == 3 ? 1 : 0;
#ifdef PIXSHT_PROBES
        // profiling aid: the spin-2 analysis as Q launches over chunk ranges (equator first), as the multi-GPU ring pieces do
        if (const int Q = env_int("PIXSHT_DBG_ANAL_SPLIT", 0); Q > 1) {
            const int nch = leg_total_chunks(P, P->R2a);
            for (int k = Q - 1; k >= 0; --k) {
                const int a = (int)((long long)nch * k / Q), b = (int)((long long)nch * (k + 1) / Q);
                const LegJob J = {2, ncomp, c0, 0, nm, d_m_list, a, b - a, ph};
                int rc = anal_launch(P, J, alm[c0], alm[c0 + 1], st); if (rc) return rc;
            }
            return PIXSHT_OK;
        }
#endif
        const LegJob J = {2, ncomp, c0, 0, nm, d_m_list, 0, leg_total_chunks(P, P->R2a), ph};
        int rc = anal_launch(P, J, alm[c0], alm[c0 + 1], st); if (rc) return rc;
    }
    return PIXSHT_OK;
}

// FFT stage for components [c_begin, c_begin+c_count) of band rings [ring_begin, ring_begin+ring_count); `phase` points at the
// row of (ring_begin, component 0) in a buffer with ncomp components per ring
static int stage_fft(pixsht_plan* P, int dir, int ncomp, int c_begin, int c_count, double2* phase, int ring_begin, int ring_count,
                     void* const* maps, cudaStream_t st, const long long* mtab = nullptr, bool stokes = true)
{
    if (ring_count <= 0 || c_count <= 0) return PIXSHT_OK;
    FftParams F;
    memset(&F, 0, sizeof(F));
    F.nphi = P->nphi; F.n = P->nfft; F.nfac = P->nfac;
    for (int i = 0; i < P->nfac; ++i) { F.fac[i] = P->fac[i]; F.magic[i] = P->fft_magic[i]; }
    F.tw = P->d_tw.p; F.phi0tw = P->d_phi0tw.p; F.wgt = P->d_wgt.p; F.perm = P->d_perm.p; F.mmax = P->mmax;
    F.phase = phase; F.mtab = mtab; F.MP = P->MP; F.ncomp = ncomp; F.c_begin = c_begin;
    F.ring_begin = ring_begin; F.ring_count = ring_count;
    F.nx = P->nx; F.ny = P->ny; F.flipx = P->flipx; F.flipy = P->flipy;
    for (int c = 0; c < ncomp; ++c) F.maps[c] = maps[c];
    F.neg_mask = (stokes && P->polconv_iau && ncomp >= 2) ? (1 << (ncomp - 1)) : 0;   // U is the last Stokes component
    {
        // the row start (rowy * nx elements past the base) is pair-aligned when the base is and nx is even (nx == nphi, packed)
        const size_t al = 2 * (P->dtype == PIXSHT_F64 ? sizeof(double) : sizeof(float));
        F.vec_ok = 1;
        for (int c = c_begin; c < c_begin + c_count; ++c) if (reinterpret_cast<uintptr_t>(maps[c]) % al != 0) F.vec_ok = 0;
    }
    F.packed = P->fft_packed; F.pt = P->fft_pt;
    if (P->fft_rows) {
        if (c_count > 4) return fail(PIXSHT_ERR_ARG, "at most 4 components per FFT launch");
        F.gbuf = P->d_fftbuf.p; F.gslot = P->fft_gslot; F.galt = P->fft_galt;
    }
    int gx = P->fft_rows ? std::min(ring_count, P->fft_rows) : ring_count;
    if (!P->fft_rows && P->fft_persist > 0) {
        gx = std::min(ring_count, std::max(1, P->sm_count * P->fft_persist / c_count));
        F.prefetch = gx < ring_count ? 1 : 0;
    }
    dim3 grid(gx, c_count);
    const bool glob = P->fft_rows > 0, fwd = dir != PIXSHT_ALM2MAP;
    // m-sharded (multi-GPU) phase layout: the row I/O is the NVLink transpose; PIXSHT_FFT_EDGE_MULTI picks the kernels for it
    F.edge = (P->fft_edge && !glob && (mtab == nullptr || P->fft_edge_multi)) ? 1 : 0;
    if (F.edge) { F.nsp = P->nsp; for (int i = 0; i < P->nsp; ++i) { F.sp_first[i] = P->sp_first[i]; F.sp_count[i] = P->sp_count[i]; } }
    else { F.nsp = P->nsp_plain; for (int i = 0; i < P->nsp_plain; ++i) { F.sp_first[i] = P->sp_first_plain[i]; F.sp_count[i] = P->sp_count_plain[i]; } }
    if (F.edge) {
        if (P->dtype == PIXSHT_F64) { if (!fwd) PIXSHT_LAUNCH((fft_phase2map_edge<double>), grid, P->fft_threads, P->fft_smem, st, F); else PIXSHT_LAUNCH((fft_map2phase_edge<double>), grid, P->fft_threads, P->fft_smem, st, F); }
        else { if (!fwd) PIXSHT_LAUNCH((fft_phase2map_edge<float>), grid, P->fft_threads, P->fft_smem, st, F); else PIXSHT_LAUNCH((fft_map2phase_edge<float>), grid, P->fft_threads, P->fft_smem, st, F); }
    } else if (P->dtype == PIXSHT_F64) {
        if (!glob) { if (!fwd) PIXSHT_LAUNCH((fft_phase2map<double, false>), grid, P->fft_threads, P->fft_smem, st, F); else PIXSHT_LAUNCH((fft_map2phase<double, false>), grid, P->fft_threads, P->fft_smem, st, F); }
        else { if (!fwd) PIXSHT_LAUNCH((fft_phase2map<double, true>), grid, P->fft_threads, P->fft_smem, st, F); else PIXSHT_LAUNCH((fft_map2phase<double, true>), grid, P->fft_threads, P->fft_smem, st, F); }
    } else {
        if (!glob) { if (!fwd) PIXSHT_LAUNCH((fft_phase2map<float, false>), grid, P->fft_threads, P->fft_smem, st, F); else PIXSHT_LAUNCH((fft_map2phase<float, false>), grid, P->fft_threads, P->fft_smem, st, F); }
        else { if (!fwd) PIXSHT_LAUNCH((fft_phase2map<float, true>), grid, P->fft_threads, P->fft_smem, st, F); else PIXSHT_LAUNCH((fft_map2phase<float, true>), grid, P->fft_threads, P->fft_smem, st, F); }
    }
    P->launches++;
    CU(cudaGetLastError());
    return PIXSHT_OK;
}

static int ensure_phase(pixsht_plan* P, int ncomp)
{
    if (P->phase_ncomp >= ncomp) return PIXSHT_OK;
    if (P->d_phase.alloc((size_t)ncomp * P->MP * P->nrings)) return fail(PIXSHT_ERR_NOMEM, "phase buffer allocation failed");
    P->phase_ncomp = ncomp;
    return PIXSHT_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// pixsht_execute
// ---------------------------------------------------------------------------------------------------------------
// Band-ring ranges covered by the pair range [p0, p1): at most one range of northern and one of southern members when
// the pairs are contiguous on the sky (always the case for CAR bands).  Returns false when they are not.
static bool pair_range_rings(const pixsht_plan* P, int p0, int p1, int rng[2][2])
{
    for (int h = 0; h < 2; ++h) {
        const std::vector<int>& v = h == 0 ? P->h_ringN : P->h_ringS;
        int lo = 1 << 30, hi = -1, cnt = 0;
        for (int p = p0; p < p1; ++p) if (v[p] >= 0) { lo = std::min(lo, v[p]); hi = std::max(hi, v[p]); ++cnt; }
        if (cnt == 0) { rng[h][0] = 0; rng[h][1] = 0; continue; }
        if (hi - lo + 1 != cnt) return false;
        rng[h][0] = lo; rng[h][1] = hi + 1;
    }
    return true;
}

// rows of the caller's map for band rings [r0, r1): one contiguous block (the y flip only mirrors it)
static void ring_rows(const pixsht_plan* P, int r0, int r1, size_t esz, size_t& off_bytes, size_t& nbytes)
{
    const int row0 = P->flipy ? (P->ny - r1) : r0;
    off_bytes = (size_t)row0 * P->nx * esz; nbytes = (size_t)(r1 - r0) * P->nx * esz;
}

// PIXSHT_PIECE_SHAPE=0 makes every pipeline of the host path use equal pieces (read once per process).
static bool graded_pieces()
{
    static const bool on = env_int("PIXSHT_PIECE_SHAPE", 1) != 0;
    return on;
}

// Cumulative piece boundaries 0 = f_0 < ... < f_s = 1 of the pipelined host path.  The first piece of an input and the last piece
// of an output are exposed (nothing runs before the one has arrived / while the other leaves); the pieces in between only have to
// be short enough for their copy to hide under the neighbouring piece's kernels.
//   shape 1 (alm2map: the T alm that arrive in m ranges, the polarisation rows that leave in ring ranges): sizes grow by factors
//            of two from both ends (s = 8: 1 2 4 8 8 4 2 1 thirtieths) -- measured at C4: exposed head + tail 3.3 -> 0.3 ms, call
//            254.7 -> 250.9 ms;
//   shape 0 (map2alm): equal pieces -- larger middle pieces measured 8 ms of extra gaps in its ring-range inputs, a tapered end
//            of its alm outputs 1.6 ms more tail (profiles/r02/e2e_probe_pieces*.txt).
static std::vector<double> piece_fractions(int nsplit, int limit, int shape = 0)
{
    std::vector<double> f;
    const int s = std::max(1, std::min(nsplit, limit));
    if (shape == 0 || !graded_pieces() || s < 4) { for (int k = 0; k <= s; ++k) f.push_back((double)k / s); return f; }
    std::vector<double> w(s);
    double tot = 0.0;
    for (int k = 0; k < s; ++k) {
        w[k] = (double)(1 << std::min(std::min(k, s - 1 - k), 20));
        tot += w[k];
    }
    double acc = 0.0;
    f.push_back(0.0);
    for (int k = 0; k < s; ++k) { acc += w[k]; f.push_back(k == s - 1 ? 1.0 : acc / tot); }
    return f;
}

// m boundaries 0 = mb[0] <= ... <= mb[K] = mmax + 1 of equal Legendre work at the cumulative fractions f (work per m ~ lmax - m + 1)
static std::vector<int> m_bounds(const pixsht_plan* P, const std::vector<double>& f)
{
    const int K = (int)f.size() - 1, n = P->mmax + 1;
    std::vector<int> mb(K + 1);
    for (int k = 0; k <= K; ++k) mb[k] = (int)std::lround(n * (1.0 - std::sqrt(1.0 - f[k])));
    mb[0] = 0; mb[K] = n;
    for (int k = 1; k <= K; ++k) mb[k] = std::max(mb[k], mb[k - 1]);
    return mb;
}

// boundaries 0 = cb[0] <= ... <= cb[K] = nch of `nch` ring-pair chunks (pole to equator) of equal Legendre work at the cumulative
// fractions f (work per pair ~ sin(theta))
static std::vector<int> chunk_bounds(int nch, const std::vector<double>& f)
{
    const int K = (int)f.size() - 1;
    std::vector<int> cb(K + 1);
    for (int k = 0; k <= K; ++k) cb[k] = (int)std::lround(nch * (2.0 / 3.14159265358979323846) * std::acos(1.0 - f[k]));
    cb[0] = 0; cb[K] = nch;
    for (int k = 1; k <= K; ++k) cb[k] = std::max(cb[k], cb[k - 1]);
    return cb;
}

// A piece of the ring pairs: chunks [c0, c1) and the band rings [rings[h][0], rings[h][1]) of their northern (h = 0) and southern
// members.  A piece of whole components: all chunks, rings {{0, nrings}, {0, 0}}.
struct Piece { int c0, c1; int rings[2][2]; };

// The pieces between the chunk boundaries cb (chunks of 32 R pairs); false when the pairs of a piece are not contiguous on the sky
static bool chunk_pieces(const pixsht_plan* P, int R, const std::vector<int>& cb, std::vector<Piece>& pcs)
{
    pcs.resize(cb.size() - 1);
    for (size_t k = 0; k < pcs.size(); ++k) {
        pcs[k].c0 = cb[k]; pcs[k].c1 = cb[k + 1];
        if (!pair_range_rings(P, std::min(P->npairs, cb[k] * 32 * R), std::min(P->npairs, cb[k + 1] * 32 * R), pcs[k].rings)) return false;
    }
    return true;
}

// f(r0, r1) for the band-ring range of each hemisphere of a piece that is not empty, north first
template <class F>
static int each_hemisphere(const Piece& pc, F&& f)
{
    for (int h = 0; h < 2; ++h)
        if (pc.rings[h][1] > pc.rings[h][0]) { const int rc = f(pc.rings[h][0], pc.rings[h][1]); if (rc) return rc; }
    return PIXSHT_OK;
}

// first alm index of column m (nalm past the last column)
static long long col_begin(const pixsht_plan* P, int m) { return m > P->mmax ? P->nalm : alm_index(P->lmax, m, m); }

// The Float64 alm of component (or batch member) c that the Legendre kernels read and write: `alm` itself in a Float64 plan,
// the plan's work buffer d_alm64[c] in a Float32 plan.
static int work_alm(pixsht_plan* P, int c, void* alm, double2** out)
{
    if (P->dtype != PIXSHT_F32) { *out = static_cast<double2*>(alm); return PIXSHT_OK; }
    if (P->d_alm64[c].n < (size_t)P->nalm && P->d_alm64[c].alloc(P->nalm)) return fail(PIXSHT_ERR_NOMEM, "alm work buffer allocation failed");
    *out = P->d_alm64[c].p;
    return PIXSHT_OK;
}

// Float32 plan: converts the alm elements [i0, i1) from the Float32 array `alm` to its work buffer `alm64` (to64) or back, one
// launch on `st`; nothing in a Float64 plan, whose work buffer is the array
static void convert_alm(pixsht_plan* P, bool to64, void* alm, double2* alm64, long long i0, long long i1, cudaStream_t st)
{
    if (P->dtype != PIXSHT_F32) return;
    const int grid = P->sm_count > 0 ? P->sm_count * 8 : 256;
    if (to64) PIXSHT_LAUNCH(k_cvt_f32_to_f64, grid, 256, 0, st, (const float*)alm + 2 * i0, (double*)(alm64 + i0), 2 * (i1 - i0));
    else PIXSHT_LAUNCH(k_cvt_f64_to_f32, grid, 256, 0, st, (const double*)(alm64 + i0), (float*)alm + 2 * i0, 2 * (i1 - i0));
    P->launches++;
}

// every stream of the plan idle, errors swallowed (failure paths: the error text of the original failure is kept by the caller)
static void quiesce(pixsht_plan* P)
{
    const std::string keep = g_err;
    if (P->s_h2d) (void)cudaStreamSynchronize(P->s_h2d);
    if (P->stream) (void)cudaStreamSynchronize(P->stream);
    if (P->s_d2h) (void)cudaStreamSynchronize(P->s_d2h);
    (void)cudaGetLastError();
    host_copies_done(P);
    g_err = keep;
}

// One call of the pipelined host path: its streams, the device staging of each component, whether each of the caller's arrays
// is pageable (staged by the plan's copy threads) and the dependency events, handed out in order.
struct HostCall {
    pixsht_plan* P;
    int ncomp;
    void* const* alms; void* const* maps;     // the caller's arrays
    cudaStream_t sc, sh, sd;                  // compute, host -> device, device -> host
    size_t esz;
    void* dmap[3]; void* dalm[3];             // staging, boundary dtype
    double2* dalm64[3];                       // what the Legendre kernels see
    bool pg_alm[3], pg_map[3];
    int ndep;
    // <= ~45 per call; the batch path recycles entries only after their waits were enqueued
    cudaEvent_t next_ev() { return P->dep[ndep++ % PIXSHT_NDEP]; }
    // FFT of components [cb, cb+cn) for band rings [r0, r1)
    int fft(int dir, int cb, int cn, int r0, int r1)
    {
        return stage_fft(P, dir, ncomp, cb, cn, P->d_phase.p + (long long)r0 * ncomp * P->MP, r0, r1 - r0, dmap, sc);
    }
    // H2D of the rows of component c for band rings [r0, r1)
    int rows_in(int c, int r0, int r1)
    {
        size_t off, nb; ring_rows(P, r0, r1, esz, off, nb);
        CU(host_copy_in(P, pg_map[c], (char*)dmap[c] + off, (const char*)maps[c] + off, nb, sh));
        return PIXSHT_OK;
    }
    // FFT + D2H of components [cb, cb+cn) for band rings [r0, r1)
    int emit_rings(int cb, int cn, int r0, int r1)
    {
        int rc = fft(PIXSHT_ALM2MAP, cb, cn, r0, r1); if (rc) return rc;
        cudaEvent_t e = next_ev();
        CU(cudaEventRecord(e, sc));
        CU(cudaStreamWaitEvent(sd, e, 0));
        size_t off, nb; ring_rows(P, r0, r1, esz, off, nb);
        for (int c = cb; c < cb + cn; ++c)
            CU(host_copy_out(P, pg_map[c], (char*)maps[c] + off, (char*)dmap[c] + off, nb, sd));
        return PIXSHT_OK;
    }
    // conversion + D2H of the alm columns of m in [m0, m1) for components [cb, cb+cn)
    int emit_alm(int cb, int cn, int m0, int m1)
    {
        if (m1 <= m0) return PIXSHT_OK;
        const long long i0 = col_begin(P, m0), i1 = col_begin(P, m1);
        for (int c = cb; c < cb + cn; ++c) convert_alm(P, false, dalm[c], dalm64[c], i0, i1, sc);
        cudaEvent_t e = next_ev();
        CU(cudaEventRecord(e, sc));
        CU(cudaStreamWaitEvent(sd, e, 0));
        for (int c = cb; c < cb + cn; ++c)
            CU(host_copy_out(P, pg_alm[c], (char*)alms[c] + (size_t)i0 * 2 * esz, (char*)dalm[c] + (size_t)i0 * 2 * esz, (size_t)(i1 - i0) * 2 * esz, sd));
        return PIXSHT_OK;
    }
};

static int host_alm2map(HostCall& H)
{
    pixsht_plan* P = H.P;
    cudaStream_t sc = H.sc;
    const int ncomp = H.ncomp, c0 = ncomp == 3 ? 1 : 0;   // c0: first spin-2 component
    const bool has0 = ncomp != 2, has2 = ncomp >= 2;
    const PhaseRef ph = {P->d_phase.p, 0, 0};
    int rc;
    // Synthesis of m in [m0, m1) of components [cb, cb+cn) in ring-pair ranges of equal Legendre work, polar side first, so that
    // the last (exposed) piece of the map copy is the one with the fewest rings; each range's rows leave after its FFT.
    auto synth_in_ring_pieces = [&](int spin, int cb, int cn, int m0, int m1) -> int {
        const int R = spin == 0 ? P->R0 : P->R2, nch = leg_total_chunks(P, R);
        std::vector<Piece> pcs;
        if (!chunk_pieces(P, R, chunk_bounds(nch, piece_fractions(P->nsplit, nch, 1)), pcs)) pcs.assign(1, {0, nch, {{0, P->nrings}, {0, 0}}});
        for (const Piece& pc : pcs) {
            const LegJob J = {spin, ncomp, cb, m0, m1 - m0, nullptr, pc.c0, pc.c1 - pc.c0, ph};
            int rc2 = synth_launch(P, J, sc); if (rc2) return rc2;
            rc2 = each_hemisphere(pc, [&](int r0, int r1) { return H.emit_rings(cb, cn, r0, r1); }); if (rc2) return rc2;
        }
        return PIXSHT_OK;
    };

    // input copies: the spin-0 alm goes first, in m ranges of equal Legendre work, so that its synthesis starts after a
    // fraction of one component has arrived; the polarisation alm follow and arrive under the spin-0 work
    // A single spin-0 map has no polarisation work for its rows to leave under: its LAST m piece then carries half of the
    // work and is synthesised in ring ranges whose rows leave one by one (pieces 1 2 4 8 15 thirtieths; tonly_rings).
    const bool tonly_rings = has0 && !has2 && graded_pieces() && P->nsplit >= 5 && P->mmax + 1 >= 64 && leg_total_chunks(P, P->R0) >= env_int("PIXSHT_TONLY_MINCHUNKS", 16);   // large plans only: the pieces must outweigh their launches
    const std::vector<int> mb0 = m_bounds(P, tonly_rings ? std::vector<double>{0.0, 1.0 / 30, 3.0 / 30, 7.0 / 30, 15.0 / 30, 1.0}
                                                         : piece_fractions(P->nsplit, P->mmax + 1, 1));
    const int K0 = has0 ? (int)mb0.size() - 1 : 0;
    std::vector<cudaEvent_t> e_t(K0);
    for (int k = 0; k < K0; ++k) {
        const long long i0 = col_begin(P, mb0[k]), i1 = col_begin(P, mb0[k + 1]);
        if (i1 > i0) CU(host_copy_in(P, H.pg_alm[0], (char*)H.dalm[0] + (size_t)i0 * 2 * H.esz, (const char*)H.alms[0] + (size_t)i0 * 2 * H.esz, (size_t)(i1 - i0) * 2 * H.esz, H.sh));
        e_t[k] = H.next_ev(); CU(cudaEventRecord(e_t[k], H.sh));
    }
    cudaEvent_t e_in[3] = {nullptr, nullptr, nullptr};
    for (int c = (has0 ? 1 : 0); c < ncomp; ++c) {
        CU(host_copy_in(P, H.pg_alm[c], H.dalm[c], H.alms[c], (size_t)P->nalm * 2 * H.esz, H.sh));
        e_in[c] = H.next_ev(); CU(cudaEventRecord(e_in[c], H.sh));
    }
    if (has0) {
        rc = ensure_seek(P, 0, sc); if (rc) return rc;
        for (int k = 0; k < K0; ++k) {
            const long long i0 = col_begin(P, mb0[k]), i1 = col_begin(P, mb0[k + 1]);
            CU(cudaStreamWaitEvent(sc, e_t[k], 0));
            if (i1 <= i0) continue;
            convert_alm(P, true, H.dalm[0], H.dalm64[0], i0, i1, sc);
            rc = synth_prep(P, 0, H.dalm64[0], H.dalm64[0], sc, i0, i1 - i0); if (rc) return rc;
            if (tonly_rings && k == K0 - 1) break;   // the last m piece goes in ring ranges, below
            const LegJob J = {0, ncomp, 0, mb0[k], mb0[k + 1] - mb0[k], nullptr, 0, leg_total_chunks(P, P->R0), ph};
            rc = synth_launch(P, J, sc); if (rc) return rc;
        }
        rc = tonly_rings ? synth_in_ring_pieces(0, 0, 1, mb0[K0 - 1], mb0[K0]) : H.emit_rings(0, 1, 0, P->nrings); if (rc) return rc;
    }
    if (has2) {
        CU(cudaStreamWaitEvent(sc, e_in[c0], 0));
        CU(cudaStreamWaitEvent(sc, e_in[c0 + 1], 0));
        convert_alm(P, true, H.dalm[c0], H.dalm64[c0], 0, P->nalm, sc);
        convert_alm(P, true, H.dalm[c0 + 1], H.dalm64[c0 + 1], 0, P->nalm, sc);
        rc = synth_prep(P, 2, H.dalm64[c0], H.dalm64[c0 + 1], sc); if (rc) return rc;
        rc = synth_in_ring_pieces(2, c0, 2, 0, P->mmax + 1); if (rc) return rc;
    }
    return PIXSHT_OK;
}

static int host_map2alm(HostCall& H)
{
    pixsht_plan* P = H.P;
    cudaStream_t sc = H.sc;
    const int ncomp = H.ncomp, c0 = ncomp == 3 ? 1 : 0;   // c0: first spin-2 component
    const bool has0 = ncomp != 2, has2 = ncomp >= 2;
    const PhaseRef ph = {P->d_phase.p, 0, 0};
    int rc;
    // Analysis of chunks [ch0, ch0+nch) of components [cb, cb+cn) in m ranges of equal Legendre work, ascending (the last piece is
    // the smallest); each range's alm columns leave after its launch.
    auto anal_in_m_pieces = [&](int spin, int cb, int cn, int ch0, int nch) -> int {
        const std::vector<int> mb = m_bounds(P, piece_fractions(P->nsplit, P->mmax + 1));
        for (size_t q = 0; q + 1 < mb.size(); ++q) {
            const LegJob J = {spin, ncomp, cb, mb[q], mb[q + 1] - mb[q], nullptr, ch0, nch, ph};
            int rc2 = anal_launch(P, J, H.dalm64[cb], cn == 2 ? H.dalm64[cb + 1] : nullptr, sc); if (rc2) return rc2;
            rc2 = H.emit_alm(cb, cn, mb[q], mb[q + 1]); if (rc2) return rc2;
        }
        return PIXSHT_OK;
    };

    // input copies: the spin-0 map goes first, in ring-pair ranges (north rows + mirrored south rows), so that its FFTs
    // and analysis start after a fraction of one component has arrived; the polarisation maps follow
    const int Ra = P->R0a, nch0 = leg_total_chunks(P, Ra);
    // The pieces go EQUATOR FIRST (the last of the pole-to-equator chunk ranges is copied and analysed first): the equatorial
    // chunks carry most of the Legendre work (every m is active there), so the compute stream has a backlog after the first
    // piece and every later copy hides under it; pole first, the bulk of the spin-0 analysis waited for the end of the whole
    // component's copy.  Sizes from the equator: 1, 2, 3, 3, ... chunks (the first piece is the exposed head of the call).
    // PIXSHT_PIECE_SHAPE=0: equal pieces, pole first (round-1 order).
    const bool eq_first = has0 && graded_pieces() && nch0 >= 4 && P->nsplit >= 4;
    const bool tonly_m = has0 && !has2 && nch0 >= env_int("PIXSHT_TONLY_MINCHUNKS", 16);   // single spin-0 map of a large plan, see below
    std::vector<Piece> pcs0;   // in the order they are copied and analysed
    if (has0) {
        std::vector<int> cb0;
        if (eq_first) {
            cb0.push_back(nch0);
            for (int k = 0; cb0.back() > 0; ++k) {
                const int left = cb0.back();
                int take = (k == 0) ? 1 : (k == 1 ? 2 : std::max(3, (nch0 - 3 + P->nsplit - 3) / std::max(1, P->nsplit - 2)));
                if ((int)cb0.size() == P->nsplit || take > left) take = left;
                // a single spin-0 map: the polar 40 % of the chunks (a fifth of the work) stay together as the last piece, which is
                // analysed in m ranges whose alm columns leave one by one (nothing else would cover that copy)
                if (tonly_m && k > 0 && nch0 - left >= (nch0 * 3 + 4) / 5) take = left;
                cb0.push_back(left - take);
            }
            std::reverse(cb0.begin(), cb0.end());
        } else {
            for (double f : piece_fractions(P->nsplit, nch0)) cb0.push_back((int)std::lround(nch0 * f));
            cb0.back() = nch0;
            for (size_t k = 1; k < cb0.size(); ++k) cb0[k] = std::max(cb0[k], cb0[k - 1]);
        }
        if (!chunk_pieces(P, Ra, cb0, pcs0)) pcs0.assign(1, {0, nch0, {{0, P->nrings}, {0, 0}}});
        if (eq_first) std::reverse(pcs0.begin(), pcs0.end());
    }
    const int K0 = (int)pcs0.size();
    std::vector<cudaEvent_t> e_t(K0);
    for (int k = 0; k < K0; ++k) {
        rc = each_hemisphere(pcs0[k], [&](int r0, int r1) { return H.rows_in(0, r0, r1); }); if (rc) return rc;
        e_t[k] = H.next_ev(); CU(cudaEventRecord(e_t[k], H.sh));
    }
    // The polarisation maps follow in two parts: the equatorial third of the rings (half of the spin-2 Legendre work), then
    // the polar rest.  The analysis of the first part (all m) starts as soon as it has arrived -- about when the spin-0 work
    // ends -- and covers the arrival of the second, which is then analysed in m ranges whose alm columns leave one by one.
    const int nch2 = leg_total_chunks(P, P->R2a);
    const int cA = has2 ? (int)std::lround(nch2 * (2.0 / 3.0)) : 0;      // chunks [cA, nch2): the equatorial part
    std::vector<Piece> parts;                                             // [0]: the polar part, [1]: the equatorial part
    const bool two_part = has2 && cA > 0 && cA < nch2 && chunk_pieces(P, P->R2a, {0, cA, nch2}, parts);
    cudaEvent_t e_in[3] = {nullptr, nullptr, nullptr}, e_partA = nullptr;
    if (two_part) {
        for (int part : {1, 0}) {
            for (int c = c0; c < c0 + 2; ++c) {
                rc = each_hemisphere(parts[part], [&](int r0, int r1) { return H.rows_in(c, r0, r1); }); if (rc) return rc;
            }
            cudaEvent_t e = H.next_ev(); CU(cudaEventRecord(e, H.sh));
            if (part == 1) e_partA = e; else e_in[c0] = e_in[c0 + 1] = e;
        }
    } else {
        for (int c = (has0 ? 1 : 0); c < ncomp; ++c) {
            CU(host_copy_in(P, H.pg_map[c], H.dmap[c], H.maps[c], (size_t)P->nx * P->ny * H.esz, H.sh));
            e_in[c] = H.next_ev(); CU(cudaEventRecord(e_in[c], H.sh));
        }
    }
    for (int c = 0; c < ncomp; ++c) CU(cudaMemsetAsync(H.dalm64[c], 0, (size_t)P->nalm * sizeof(double2), sc));
    if (has0) {
        // a single spin-0 map: its last (polar) piece is analysed in m ranges, each followed by the copy of its alm columns
        const bool last_in_m = tonly_m && eq_first && K0 > 1;
        for (int k = 0; k < K0; ++k) {
            const Piece& pc = pcs0[k];
            CU(cudaStreamWaitEvent(sc, e_t[k], 0));
            rc = each_hemisphere(pc, [&](int r0, int r1) { return H.fft(PIXSHT_MAP2ALM, 0, 1, r0, r1); }); if (rc) return rc;
            if (last_in_m && k == K0 - 1) rc = anal_in_m_pieces(0, 0, 1, pc.c0, pc.c1 - pc.c0);
            else {
                const LegJob J = {0, ncomp, 0, 0, P->mmax + 1, nullptr, pc.c0, pc.c1 - pc.c0, ph};
                rc = anal_launch(P, J, H.dalm64[0], nullptr, sc);
            }
            if (rc) return rc;
        }
        if (!last_in_m) { rc = H.emit_alm(0, 1, 0, P->mmax + 1); if (rc) return rc; }
    }
    if (has2) {
        int chunksB = nch2;   // chunks left for the m-range launches below
        if (two_part) {
            CU(cudaStreamWaitEvent(sc, e_partA, 0));
            rc = each_hemisphere(parts[1], [&](int r0, int r1) { return H.fft(PIXSHT_MAP2ALM, c0, 2, r0, r1); }); if (rc) return rc;
            const LegJob JA = {2, ncomp, c0, 0, P->mmax + 1, nullptr, cA, nch2 - cA, ph};
            rc = anal_launch(P, JA, H.dalm64[c0], H.dalm64[c0 + 1], sc); if (rc) return rc;
            chunksB = cA;
        }
        CU(cudaStreamWaitEvent(sc, e_in[c0], 0));
        CU(cudaStreamWaitEvent(sc, e_in[c0 + 1], 0));
        if (two_part) rc = each_hemisphere(parts[0], [&](int r0, int r1) { return H.fft(PIXSHT_MAP2ALM, c0, 2, r0, r1); });
        else rc = H.fft(PIXSHT_MAP2ALM, c0, 2, 0, P->nrings);
        if (rc) return rc;
        rc = anal_in_m_pieces(2, c0, 2, 0, chunksB); if (rc) return rc;
    }
    return PIXSHT_OK;
}

// Host-pointer transform: copies, Legendre and FFT launches are pipelined over three streams so that most of the PCIe
// time hides under the Legendre kernels (spin-0 work runs while the polarisation inputs arrive; results leave in
// split-sized pieces while the next split computes).
static int execute_host(pixsht_plan* P, int direction, int ncomp, void* const* alms, void* const* maps)
{
    HostCall H = {P, ncomp, alms, maps, P->stream, P->s_h2d, P->s_d2h, P->dtype == PIXSHT_F32 ? sizeof(float) : sizeof(double)};
    const size_t map_bytes = (size_t)P->nx * P->ny * H.esz, alm_bytes = (size_t)P->nalm * 2 * H.esz;
    for (int c = 0; c < ncomp; ++c) {
        if (P->d_map[c].n < map_bytes && P->d_map[c].alloc(map_bytes)) return fail(PIXSHT_ERR_NOMEM, "map staging allocation failed");
        if (P->d_alm[c].n < alm_bytes && P->d_alm[c].alloc(alm_bytes)) return fail(PIXSHT_ERR_NOMEM, "alm staging allocation failed");
        H.dmap[c] = P->d_map[c].p; H.dalm[c] = P->d_alm[c].p;
        int rc = work_alm(P, c, H.dalm[c], &H.dalm64[c]); if (rc) return rc;
        H.pg_alm[c] = host_is_pageable(alms[c]); H.pg_map[c] = host_is_pageable(maps[c]);
    }

    // the copy streams start after whatever the caller queued on the compute stream
    cudaEvent_t e_start = H.next_ev();
    CU(cudaEventRecord(e_start, H.sc));
    CU(cudaStreamWaitEvent(H.sh, e_start, 0));
    CU(cudaStreamWaitEvent(H.sd, e_start, 0));
    CU(cudaEventRecord(P->ev[0], H.sc));
    const int rc = direction == PIXSHT_ALM2MAP ? host_alm2map(H) : host_map2alm(H);
    if (rc) return rc;
    CU(cudaEventRecord(P->ev[1], H.sc));
    CU(cudaStreamSynchronize(H.sh));
    CU(cudaStreamSynchronize(H.sc));
    CU(cudaStreamSynchronize(H.sd));
    CU(cudaGetLastError());
    host_copies_done(P);
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, P->ev[0], P->ev[1]));
    for (auto& t : P->timings) t = 0;
    P->timings[5] = ms;   // compute stream busy span (copies overlap it)
    return PIXSHT_OK;
}

extern "C" int pixsht_execute(pixsht_plan* P, int direction, int ncomp, void* const* alms, void* const* maps, int location)
{
    if (!P || !alms || !maps) return fail(PIXSHT_ERR_ARG, "null argument");
    if (direction != PIXSHT_MAP2ALM && direction != PIXSHT_ALM2MAP) return fail(PIXSHT_ERR_ARG, "bad direction");
    if (ncomp < 1 || ncomp > 3) return fail(PIXSHT_ERR_ARG, "SHTs require 1 <= ncomp <= 3, for I, QU, and IQU.");
    if (location != PIXSHT_HOST && location != PIXSHT_DEVICE) return fail(PIXSHT_ERR_ARG, "bad location");
    for (int c = 0; c < ncomp; ++c) if (!alms[c] || !maps[c]) return fail(PIXSHT_ERR_ARG, "null component pointer");
    std::lock_guard<std::mutex> lock(P->mu);
    if (P->multi) {
        // multi-GPU plan: whole arrays in host memory, or anywhere the GPUs can copy from (the copies use cudaMemcpyDefault)
        const int rcm = execute_multi(P, direction, ncomp, alms, maps, false);
        if (rcm) multi_quiesce(P->multi);
        return rcm;
    }
    int rc = check_device(P->device); if (rc) return rc;
    const auto t_begin = std::chrono::steady_clock::now();
    P->launches = 0;
    rc = ensure_phase(P, ncomp); if (rc) return rc;
    if (location == PIXSHT_HOST) {
        rc = execute_host(P, direction, ncomp, alms, maps);
        if (rc) quiesce(P);   // nothing may still reference the caller's buffers when a failed call returns
        P->timings[4] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
        return rc;
    }
    cudaStream_t st = P->stream;
    double2* dalm64[3] = {nullptr, nullptr, nullptr}; // what the Legendre kernels see
    for (int c = 0; c < ncomp; ++c) { rc = work_alm(P, c, alms[c], &dalm64[c]); if (rc) return rc; }
    const PhaseRef ph = {P->d_phase.p, 0, 0};

    CU(cudaEventRecord(P->ev[0], st));
    CU(cudaEventRecord(P->ev[1], st));
    P->kev_on = true;
    struct KevOff { pixsht_plan* p; ~KevOff() { p->kev_on = false; } } kev_off{P};
    if (direction == PIXSHT_ALM2MAP) {
        for (int c = 0; c < ncomp; ++c) convert_alm(P, true, alms[c], dalm64[c], 0, P->nalm, st);
        rc = stage_alm2phase(P, ncomp, dalm64, P->mmax + 1, nullptr, ph, st); if (rc) return rc;
        CU(cudaEventRecord(P->ev[2], st));
        rc = stage_fft(P, PIXSHT_ALM2MAP, ncomp, 0, ncomp, P->d_phase.p, 0, P->nrings, maps, st); if (rc) return rc;
        CU(cudaEventRecord(P->ev[3], st));
    } else {
        rc = stage_fft(P, PIXSHT_MAP2ALM, ncomp, 0, ncomp, P->d_phase.p, 0, P->nrings, maps, st); if (rc) return rc;
        CU(cudaEventRecord(P->ev[2], st));
        for (int c = 0; c < ncomp; ++c) CU(cudaMemsetAsync(dalm64[c], 0, (size_t)P->nalm * sizeof(double2), st));
        rc = stage_phase2alm(P, ncomp, ph, P->mmax + 1, nullptr, dalm64, st); if (rc) return rc;
        for (int c = 0; c < ncomp; ++c) convert_alm(P, false, alms[c], dalm64[c], 0, P->nalm, st);
        CU(cudaEventRecord(P->ev[3], st));
    }
    CU(cudaEventRecord(P->ev[4], st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    float ms[4] = {0, 0, 0, 0};
    for (int i = 0; i < 4; ++i) CU(cudaEventElapsedTime(&ms[i], P->ev[i], P->ev[i + 1]));
    for (auto& t : P->timings) t = 0;
    P->timings[0] = ms[0];
    if (direction == PIXSHT_ALM2MAP) { P->timings[1] = ms[1]; P->timings[2] = ms[2]; }
    else { P->timings[2] = ms[1]; P->timings[1] = ms[2]; }
    P->timings[3] = ms[3];
    P->timings[4] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    if (ncomp != 2) { float k; CU(cudaEventElapsedTime(&k, P->kev[0], P->kev[1])); P->timings[6] = k; }
    if (ncomp >= 2) { float k; CU(cudaEventElapsedTime(&k, P->kev[2], P->kev[3])); P->timings[7] = k; }
    return PIXSHT_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// batched spin-0 transforms (legendre_batch.cuh): nbatch independent T maps / alm on one geometry, NB at a time
// ---------------------------------------------------------------------------------------------------------------
template <int NB>
static int batch_group(pixsht_plan* P, int direction, double2* const* alm64, void* const* dmap, cudaStream_t st)
{
    // ring pairs per thread: synthesis keeps 4 NB accumulators per ring (R = 2 at NB = 4); analysis wants many rings per
    // lane because its per-step cross-lane reduction grows with NB
    constexpr int RS = (NB == 4) ? 2 : 4, RA = 4;
    const int R = direction == PIXSHT_ALM2MAP ? RS : RA;
    const int prep_grid = P->sm_count > 0 ? P->sm_count * 8 : 256;
    int rc = ensure_seek(P, 0, st); if (rc) return rc;
    const LegJob J = {0, NB, 0, 0, P->mmax + 1, nullptr, 0, leg_total_chunks(P, R), {P->d_phase.p, 0, 0}};
    LegParams L = leg_params(P, J, R);
    BatchPtrs A;
    memset(&A, 0, sizeof(A));
    for (int b = 0; b < NB; ++b) { A.in[b] = alm64[b]; A.out[b] = alm64[b]; }
    const int grid = L.nm * L.nchunks;
    if (direction == PIXSHT_ALM2MAP) {
        const size_t need = (size_t)P->nalm * BatchRec<NB>::ND;
        if (P->d_rec0.n < need && P->d_rec0.alloc(need)) return fail(PIXSHT_ERR_NOMEM, "record buffer allocation failed");
        L.rec = P->d_rec0.p;
        PIXSHT_LAUNCH((k_prep_synth_b<NB>), prep_grid, 256, 0, st, 0LL, (long long)P->nalm, P->lmax, P->d_ad0.p, P->d_gamma0.p, A, P->d_rec0.p);
        PIXSHT_LAUNCH((leg_synth_b<RS, NB>), grid, LEG_NT, 0, st, L);
        P->launches += 2;
        CU(cudaGetLastError());
        return stage_fft(P, PIXSHT_ALM2MAP, NB, 0, NB, P->d_phase.p, 0, P->nrings, dmap, st, nullptr, false);
    }
    rc = stage_fft(P, PIXSHT_MAP2ALM, NB, 0, NB, P->d_phase.p, 0, P->nrings, dmap, st, nullptr, false); if (rc) return rc;
    for (int b = 0; b < NB; ++b) CU(cudaMemsetAsync(alm64[b], 0, (size_t)P->nalm * sizeof(double2), st));
    PIXSHT_LAUNCH((leg_anal_b<RA, NB>), grid, LEG_NT, 0, st, L, A);
    P->launches++;
    CU(cudaGetLastError());
    return PIXSHT_OK;
}

static int execute_batch_locked(pixsht_plan* P, int direction, int nbatch, void* const* alms, void* const* maps, int location);

extern "C" int pixsht_execute_batch(pixsht_plan* P, int direction, int nbatch, void* const* alms, void* const* maps, int location)
{
    if (!P || !alms || !maps) return fail(PIXSHT_ERR_ARG, "null argument");
    if (direction != PIXSHT_MAP2ALM && direction != PIXSHT_ALM2MAP) return fail(PIXSHT_ERR_ARG, "bad direction");
    if (nbatch < 1) return fail(PIXSHT_ERR_ARG, "need nbatch >= 1");
    if (location != PIXSHT_HOST && location != PIXSHT_DEVICE) return fail(PIXSHT_ERR_ARG, "bad location");
    for (int b = 0; b < nbatch; ++b) if (!alms[b] || !maps[b]) return fail(PIXSHT_ERR_ARG, "null map or alm pointer");
    std::lock_guard<std::mutex> lock(P->mu);
    if (P->multi) return execute_batch_multi(P, direction, nbatch, alms, maps, location);
    const int rc = execute_batch_locked(P, direction, nbatch, alms, maps, location);
    if (rc) quiesce(P);   // nothing may still reference the caller's buffers when a failed call returns
    return rc;
}

static int execute_batch_locked(pixsht_plan* P, int direction, int nbatch, void* const* alms, void* const* maps, int location)
{
    int rc = check_device(P->device); if (rc) return rc;
    const auto t_begin = std::chrono::steady_clock::now();
    P->launches = 0;
    // the phase rows of a group hold NB "components"; make room for the largest group
    rc = ensure_phase(P, LEG_MAXBATCH); if (rc) return rc;
    cudaStream_t st = P->stream;
    const size_t esz = P->dtype == PIXSHT_F32 ? 4 : 8;
    const size_t map_bytes = (size_t)P->nx * P->ny * esz, alm_bytes = (size_t)P->nalm * 2 * esz;
    // Host pointers: one group of maps is staged, transformed and copied back at a time.  With batch_overlap the staging is double
    // buffered and the copies run on the copy streams, so that group g + 1 arrives and group g - 1 leaves while group g computes.
    const bool ovl = location == PIXSHT_HOST && P->batch_overlap;
    cudaStream_t sh = ovl ? P->s_h2d : st, sd = ovl ? P->s_d2h : st;
    int nev = 0;
    auto next_ev = [&]() { return P->dep[nev++ % PIXSHT_NDEP]; };
    cudaEvent_t e_free[2] = {nullptr, nullptr};   // the last copy-out that used the staging set
    if (ovl) {
        cudaEvent_t e = next_ev();
        CU(cudaEventRecord(e, st));
        CU(cudaStreamWaitEvent(sh, e, 0));
        CU(cudaStreamWaitEvent(sd, e, 0));
    }
    int group = 0;
    for (int b0 = 0; b0 < nbatch; ++group) {
        const int left = nbatch - b0, nb = left >= 4 ? 4 : (left >= 2 ? 2 : 1);
        const int set = ovl ? (group & 1) : 0, base = 4 * set;
        void* dmap[4] = {nullptr, nullptr, nullptr, nullptr};
        void* dalm[4] = {nullptr, nullptr, nullptr, nullptr};
        double2* alm64[4] = {nullptr, nullptr, nullptr, nullptr};
        if (ovl && e_free[set]) CU(cudaStreamWaitEvent(sh, e_free[set], 0));   // the set's previous group has been computed and copied out
        for (int b = 0; b < nb; ++b) {
            const int k = base + b;
            if (location == PIXSHT_HOST) {
                if (P->d_map[k].n < map_bytes && P->d_map[k].alloc(map_bytes)) return fail(PIXSHT_ERR_NOMEM, "map staging allocation failed");
                if (P->d_alm[k].n < alm_bytes && P->d_alm[k].alloc(alm_bytes)) return fail(PIXSHT_ERR_NOMEM, "alm staging allocation failed");
                dmap[b] = P->d_map[k].p; dalm[b] = P->d_alm[k].p;
                if (direction == PIXSHT_ALM2MAP) CU(host_copy_in(P, host_is_pageable(alms[b0 + b]), dalm[b], alms[b0 + b], alm_bytes, sh));
                else CU(host_copy_in(P, host_is_pageable(maps[b0 + b]), dmap[b], maps[b0 + b], map_bytes, sh));
            } else { dmap[b] = maps[b0 + b]; dalm[b] = alms[b0 + b]; }
            rc = work_alm(P, k, dalm[b], &alm64[b]); if (rc) return rc;
        }
        if (ovl) { cudaEvent_t e = next_ev(); CU(cudaEventRecord(e, sh)); CU(cudaStreamWaitEvent(st, e, 0)); }
        if (direction == PIXSHT_ALM2MAP)
            for (int b = 0; b < nb; ++b) convert_alm(P, true, dalm[b], alm64[b], 0, P->nalm, st);
        if (nb == 4) rc = batch_group<4>(P, direction, alm64, dmap, st);
        else if (nb == 2) rc = batch_group<2>(P, direction, alm64, dmap, st);
        else {
            // a single map: the ordinary spin-0 kernels
            if (direction == PIXSHT_ALM2MAP) {
                const double2* a1[3] = {alm64[0], nullptr, nullptr};
                rc = stage_alm2phase(P, 1, a1, P->mmax + 1, nullptr, {P->d_phase.p, 0, 0}, st);
                if (!rc) rc = stage_fft(P, PIXSHT_ALM2MAP, 1, 0, 1, P->d_phase.p, 0, P->nrings, dmap, st, nullptr, false);
            } else {
                rc = stage_fft(P, PIXSHT_MAP2ALM, 1, 0, 1, P->d_phase.p, 0, P->nrings, dmap, st, nullptr, false);
                if (!rc) rc = cudaMemsetAsync(alm64[0], 0, (size_t)P->nalm * sizeof(double2), st) == cudaSuccess ? PIXSHT_OK : PIXSHT_ERR_CUDA;
                double2* a1[3] = {alm64[0], nullptr, nullptr};
                if (!rc) rc = stage_phase2alm(P, 1, {P->d_phase.p, 0, 0}, P->mmax + 1, nullptr, a1, st);
            }
        }
        if (rc) return rc;
        if (direction == PIXSHT_MAP2ALM)
            for (int b = 0; b < nb; ++b) convert_alm(P, false, dalm[b], alm64[b], 0, P->nalm, st);
        if (ovl) { cudaEvent_t e = next_ev(); CU(cudaEventRecord(e, st)); CU(cudaStreamWaitEvent(sd, e, 0)); }
        if (location == PIXSHT_HOST) {
            for (int b = 0; b < nb; ++b) {
                if (direction == PIXSHT_ALM2MAP) CU(host_copy_out(P, host_is_pageable(maps[b0 + b]), maps[b0 + b], dmap[b], map_bytes, sd));
                else CU(host_copy_out(P, host_is_pageable(alms[b0 + b]), alms[b0 + b], dalm[b], alm_bytes, sd));
            }
            if (ovl) { e_free[set] = next_ev(); CU(cudaEventRecord(e_free[set], sd)); }
            else CU(cudaStreamSynchronize(st));   // the single staging set is reused by the next group
        }
        b0 += nb;
    }
    if (ovl) { CU(cudaStreamSynchronize(sh)); CU(cudaStreamSynchronize(sd)); }
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    host_copies_done(P);
    for (auto& t : P->timings) t = 0;
    P->timings[4] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    return PIXSHT_OK;
}

extern "C" int pixsht_plan_set_stream(pixsht_plan* P, void* stream, int use_caller_stream)
{
    if (!P) return fail(PIXSHT_ERR_ARG, "null plan");
    if (P->multi) return fail(PIXSHT_ERR_UNSUPPORTED, "a multi-GPU plan runs on its own streams");
    std::lock_guard<std::mutex> lock(P->mu);
    P->stream = use_caller_stream ? (cudaStream_t)stream : P->own_stream;
    return PIXSHT_OK;
}

extern "C" int pixsht_get_timings(const pixsht_plan* P, double ms[8])
{
    if (!P || !ms) return fail(PIXSHT_ERR_ARG, "null argument");
    for (int i = 0; i < 8; ++i) ms[i] = P->timings[i];
    return PIXSHT_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// stage API (multi-GPU pipeline)
// ---------------------------------------------------------------------------------------------------------------
static int stage_common(pixsht_plan* P, int ncomp)
{
    if (!P) return fail(PIXSHT_ERR_ARG, "null plan");
    if (P->multi) return fail(PIXSHT_ERR_ARG, "the stage API works on single-GPU plans (a multi-GPU plan runs its own stages inside pixsht_execute)");
    if (ncomp < 1 || ncomp > 3) return fail(PIXSHT_ERR_ARG, "SHTs require 1 <= ncomp <= 3, for I, QU, and IQU.");
    return check_device(P->device);
}

extern "C" int64_t pixsht_phase_row_len(const pixsht_plan* P) { return P ? (int64_t)P->MP : 0; }

// components [cb, cb + cn) of an ncomp-component set that the selected spin families cover
static void stage_components(const pixsht_plan* P, int ncomp, int& cb, int& cn)
{
    const bool h0 = ncomp != 2 && P->stage_fam0, h2 = ncomp >= 2 && P->stage_fam2;
    const int c0 = ncomp == 3 ? 1 : 0;
    if (h0 && h2) { cb = 0; cn = ncomp; }
    else if (h0) { cb = 0; cn = 1; }
    else if (h2) { cb = c0; cn = 2; }
    else { cb = 0; cn = 0; }
}

// Stokes-U sign convention of the caller's maps (src/enmap.jl:178-196, 209-215 of the reference: read_map flips U of an IAU file
// on the host): here a flag of the plan, applied inside the FFT kernels' row I/O in both directions (fft.cuh: neg_mask).
extern "C" int pixsht_plan_set_polconv(pixsht_plan* P, int polconv)
{
    if (!P) return fail(PIXSHT_ERR_ARG, "null plan");
    if (polconv != PIXSHT_POLCONV_COSMO && polconv != PIXSHT_POLCONV_IAU) return fail(PIXSHT_ERR_ARG, "polconv must be PIXSHT_POLCONV_COSMO or PIXSHT_POLCONV_IAU");
    std::lock_guard<std::mutex> lock(P->mu);
    P->polconv_iau = polconv == PIXSHT_POLCONV_IAU;
    if (P->multi) multi_set_polconv(P->multi, P->polconv_iau);
    return PIXSHT_OK;
}

// Pixel areas of the band's rows (steradians), map row order: (sin(dec_hi) - sin(dec_lo)) * |d alpha| with the row edges half a
// pixel either side of the ring and clipped at the poles -- pixareamap! of the reference (src/enmap_ops.jl:124-138), one value per
// row because CAR pixel areas do not depend on RA.  O(nrings) host arithmetic, no device needed.
extern "C" int pixsht_ring_pixarea(const pixsht_geom* g, double* area)
{
    if (!g || !area) return fail(PIXSHT_ERR_ARG, "null argument");
    if (g->nphi < 1 || g->nrings_total < 1 || g->nrings < 0 || g->ring_first < 0 || g->ring_first + g->nrings > g->nrings_total)
        return fail(PIXSHT_ERR_ARG, "inconsistent geometry");
    const long double pi = 3.14159265358979323846264338327950288L;
    const bool fejer = g->ring_scheme == PIXSHT_RINGS_FEJER1;
    if (!fejer && g->nrings_total < 2) return fail(PIXSHT_ERR_ARG, "a Clenshaw-Curtis grid has at least two rings");
    const long double dth = fejer ? pi / g->nrings_total : pi / (g->nrings_total - 1);
    const long double dal = 2 * pi / g->nphi;
    for (int r = 0; r < g->nrings; ++r) {
        const int k = g->ring_first + r;
        const long double th = fejer ? dth * (k + 0.5L) : dth * k;
        long double d2 = pi / 2 - (th - dth / 2), d1 = pi / 2 - (th + dth / 2);
        if (d2 > pi / 2) d2 = pi / 2;
        if (d1 < -pi / 2) d1 = -pi / 2;
        area[g->flipy ? (g->nrings - 1 - r) : r] = (double)((sinl(d2) - sinl(d1)) * dal);
    }
    return PIXSHT_OK;
}

extern "C" int pixsht_plan_set_stage_families(pixsht_plan* P, int spin0, int spin2)
{
    if (!P) return fail(PIXSHT_ERR_ARG, "null plan");
    std::lock_guard<std::mutex> lock(P->mu);
    P->stage_fam0 = spin0 != 0; P->stage_fam2 = spin2 != 0;
    return PIXSHT_OK;
}

extern "C" int pixsht_stage_alm2phase(pixsht_plan* P, int ncomp, const void* const* d_alms, int nm, const int32_t* d_m_list,
                                      void* d_phase, int64_t row_len, void* stream)
{
    int rc = stage_common(P, ncomp); if (rc) return rc;
    std::lock_guard<std::mutex> lock(P->mu);   // the stages build the activation tables lazily and count launches
    if (!d_alms || !d_phase || nm < 0 || nm > P->mmax + 1 || row_len < nm) return fail(PIXSHT_ERR_ARG, "bad argument");
    if (nm == 0) return PIXSHT_OK;
    const double2* alm[3] = {nullptr, nullptr, nullptr};
    for (int c = 0; c < ncomp; ++c) alm[c] = (const double2*)d_alms[c];
    const PhaseRef ph = {(double2*)d_phase, (long long)row_len, 1};
    return stage_alm2phase(P, ncomp, alm, nm, d_m_list, ph, (cudaStream_t)stream, P->stage_fam0, P->stage_fam2);
}

extern "C" int pixsht_stage_phase2alm(pixsht_plan* P, int ncomp, const void* d_phase, int64_t row_len, int nm, const int32_t* d_m_list,
                                      void* const* d_alms, void* stream)
{
    int rc = stage_common(P, ncomp); if (rc) return rc;
    std::lock_guard<std::mutex> lock(P->mu);   // the stages build the activation tables lazily and count launches
    if (!d_alms || !d_phase || nm < 0 || nm > P->mmax + 1 || row_len < nm) return fail(PIXSHT_ERR_ARG, "bad argument");
    if (nm == 0) return PIXSHT_OK;
    double2* alm[3] = {nullptr, nullptr, nullptr};
    for (int c = 0; c < ncomp; ++c) alm[c] = (double2*)d_alms[c];
    const PhaseRef ph = {(double2*)d_phase, (long long)row_len, 1};
    return stage_phase2alm(P, ncomp, ph, nm, d_m_list, alm, (cudaStream_t)stream, P->stage_fam0, P->stage_fam2);
}

extern "C" int pixsht_stage_phase2map(pixsht_plan* P, int ncomp, const int64_t* d_mtab, int ring_begin, int ring_count,
                                      void* const* d_maps, void* stream)
{
    int rc = stage_common(P, ncomp); if (rc) return rc;
    std::lock_guard<std::mutex> lock(P->mu);   // the stages build the activation tables lazily and count launches
    if (!d_maps || !d_mtab || ring_begin < 0 || ring_count < 0 || ring_begin + ring_count > P->nrings) return fail(PIXSHT_ERR_ARG, "bad argument");
    int cb, cn; stage_components(P, ncomp, cb, cn);
    return stage_fft(P, PIXSHT_ALM2MAP, ncomp, cb, cn, nullptr, ring_begin, ring_count, d_maps, (cudaStream_t)stream, (const long long*)d_mtab);
}

extern "C" int pixsht_stage_map2phase(pixsht_plan* P, int ncomp, const void* const* d_maps, int ring_begin, int ring_count,
                                      const int64_t* d_mtab, void* stream)
{
    int rc = stage_common(P, ncomp); if (rc) return rc;
    std::lock_guard<std::mutex> lock(P->mu);   // the stages build the activation tables lazily and count launches
    if (!d_maps || !d_mtab || ring_begin < 0 || ring_count < 0 || ring_begin + ring_count > P->nrings) return fail(PIXSHT_ERR_ARG, "bad argument");
    int cb, cn; stage_components(P, ncomp, cb, cn);
    return stage_fft(P, PIXSHT_MAP2ALM, ncomp, cb, cn, nullptr, ring_begin, ring_count, (void* const*)d_maps, (cudaStream_t)stream, (const long long*)d_mtab);
}

// ---------------------------------------------------------------------------------------------------------------
// peer-visible device memory (multi-GPU phase buffers): CUDA IPC between the one-process-per-GPU ranks of a node
// ---------------------------------------------------------------------------------------------------------------
#ifndef PIXSHT_EMU
extern "C" int pixsht_shared_alloc(int device, size_t bytes, void** dptr, unsigned char handle[64])
{
    if (!dptr || !handle || bytes == 0) return fail(PIXSHT_ERR_ARG, "bad argument");
    int rc = check_device(device); if (rc) return rc;
    void* p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) { (void)cudaGetLastError(); return fail(PIXSHT_ERR_NOMEM, "shared phase buffer allocation failed"); }
    static_assert(sizeof(cudaIpcMemHandle_t) <= 64, "IPC handle does not fit");
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return fail(PIXSHT_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e)); }
    memset(handle, 0, 64);
    memcpy(handle, &h, sizeof(h));
    *dptr = p;
    return PIXSHT_OK;
}
extern "C" int pixsht_shared_open(int device, const unsigned char handle[64], void** dptr)
{
    if (!dptr || !handle) return fail(PIXSHT_ERR_ARG, "bad argument");
    int rc = check_device(device); if (rc) return rc;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return fail(PIXSHT_ERR_CUDA, std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e));
    *dptr = p;
    return PIXSHT_OK;
}
extern "C" int pixsht_shared_close(void* dptr)
{
    if (dptr && cudaIpcCloseMemHandle(dptr) != cudaSuccess) { (void)cudaGetLastError(); return fail(PIXSHT_ERR_CUDA, "cudaIpcCloseMemHandle failed"); }
    return PIXSHT_OK;
}
extern "C" int pixsht_shared_free(void* dptr)
{
    if (dptr && cudaFree(dptr) != cudaSuccess) { (void)cudaGetLastError(); return fail(PIXSHT_ERR_CUDA, "cudaFree failed"); }
    return PIXSHT_OK;
}
#else
// host emulation (tests only): POSIX shared memory stands in for CUDA IPC so that the world-size-2 gloo test runs the
// same peer-pointer pipeline.  handle = { name[48], size }.
#include <fcntl.h>
#include <sys/mman.h>
#include <unistd.h>
#include <map>
static std::map<void*, std::pair<size_t, std::string>> g_shm;
extern "C" int pixsht_shared_alloc(int, size_t bytes, void** dptr, unsigned char handle[64])
{
    static int counter = 0;
    char name[48];
    snprintf(name, sizeof(name), "/pixsht_%d_%d", (int)getpid(), counter++);
    int fd = shm_open(name, O_CREAT | O_RDWR | O_EXCL, 0600);
    if (fd < 0 || ftruncate(fd, (off_t)bytes) != 0) return fail(PIXSHT_ERR_NOMEM, "shm_open failed");
    void* p = mmap(nullptr, bytes, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    close(fd);
    if (p == MAP_FAILED) return fail(PIXSHT_ERR_NOMEM, "mmap failed");
    memset(handle, 0, 64);
    memcpy(handle, name, strlen(name) + 1);
    unsigned long long sz = bytes; memcpy(handle + 48, &sz, 8);
    g_shm[p] = {bytes, std::string(name)};
    *dptr = p;
    return PIXSHT_OK;
}
extern "C" int pixsht_shared_open(int, const unsigned char handle[64], void** dptr)
{
    unsigned long long sz; memcpy(&sz, handle + 48, 8);
    int fd = shm_open((const char*)handle, O_RDWR, 0600);
    if (fd < 0) return fail(PIXSHT_ERR_CUDA, "shm_open of a peer segment failed");
    void* p = mmap(nullptr, (size_t)sz, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    close(fd);
    if (p == MAP_FAILED) return fail(PIXSHT_ERR_NOMEM, "mmap failed");
    g_shm[p] = {(size_t)sz, std::string()};
    *dptr = p;
    return PIXSHT_OK;
}
extern "C" int pixsht_shared_close(void* dptr)
{
    auto it = g_shm.find(dptr);
    if (it != g_shm.end()) { munmap(dptr, it->second.first); g_shm.erase(it); }
    return PIXSHT_OK;
}
extern "C" int pixsht_shared_free(void* dptr)
{
    auto it = g_shm.find(dptr);
    if (it != g_shm.end()) { munmap(dptr, it->second.first); if (!it->second.second.empty()) shm_unlink(it->second.second.c_str()); g_shm.erase(it); }
    return PIXSHT_OK;
}
#endif

// ---------------------------------------------------------------------------------------------------------------
// page-locked host memory for the caller's arrays
// ---------------------------------------------------------------------------------------------------------------
// On a multi-socket host the pages of an allocation are interleaved over the NUMA nodes (mmap + mbind(MPOL_INTERLEAVE) +
// cudaHostRegister): the GPUs of a multi-GPU plan hang off different sockets and each pulls its own alm columns / map rows, so a
// buffer that lives on one node sends half of the traffic over the inter-socket link.  PIXSHT_HOST_NUMA=local keeps the
// allocating thread's node (plain cudaHostAlloc); single-node hosts always take that path.
#ifndef PIXSHT_EMU
static std::mutex g_hostmu;
static std::unordered_map<void*, size_t> g_host_mmaps;   // allocations made by mmap + register: address -> length
static int numa_node_count()
{
    int n = 0;
    for (int i = 0; i < 64; ++i) {
        char path[64];
        snprintf(path, sizeof(path), "/sys/devices/system/node/node%d", i);
        if (access(path, F_OK) == 0) n = i + 1;
    }
    return n;
}
#endif
extern "C" int pixsht_host_alloc(void** ptr, size_t bytes)
{
    if (!ptr || bytes == 0) return fail(PIXSHT_ERR_ARG, "bad argument");
    *ptr = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) { (void)cudaGetLastError(); return fail(PIXSHT_ERR_NODEVICE, "no CUDA device available"); }
#ifdef PIXSHT_EMU
    if (cudaMallocHost(ptr, bytes) != cudaSuccess) return fail(PIXSHT_ERR_NOMEM, "host allocation failed");
#else
    const char* mode = getenv("PIXSHT_HOST_NUMA");
    const int nodes = numa_node_count();
    if (nodes > 1 && !(mode && strcmp(mode, "local") == 0)) {
        const size_t page = 2u << 20, len = (bytes + page - 1) / page * page;
        void* p = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
        if (p != MAP_FAILED) {
            unsigned long mask[2] = {nodes >= 64 ? ~0ul : ((1ul << nodes) - 1), 0};
            (void)syscall(SYS_mbind, p, len, 3 /* MPOL_INTERLEAVE */, mask, (unsigned long)(nodes + 1), 0u);   // best effort: a refused policy leaves the default
            if (cudaHostRegister(p, len, cudaHostRegisterPortable) == cudaSuccess) {
                std::lock_guard<std::mutex> lock(g_hostmu);
                g_host_mmaps[p] = len;
                *ptr = p;
                return PIXSHT_OK;
            }
            (void)cudaGetLastError();
            munmap(p, len);
        }
    }
    if (cudaHostAlloc(ptr, bytes, cudaHostAllocPortable) != cudaSuccess) { (void)cudaGetLastError(); return fail(PIXSHT_ERR_NOMEM, "page-locked host allocation failed"); }
#endif
    return PIXSHT_OK;
}
extern "C" int pixsht_host_free(void* ptr)
{
#ifndef PIXSHT_EMU
    if (ptr) {
        size_t len = 0;
        {
            std::lock_guard<std::mutex> lock(g_hostmu);
            auto it = g_host_mmaps.find(ptr);
            if (it != g_host_mmaps.end()) { len = it->second; g_host_mmaps.erase(it); }
        }
        if (len) {
            if (cudaHostUnregister(ptr) != cudaSuccess) (void)cudaGetLastError();
            munmap(ptr, len);
            return PIXSHT_OK;
        }
    }
#endif
    if (ptr && cudaFreeHost(ptr) != cudaSuccess) { (void)cudaGetLastError(); return fail(PIXSHT_ERR_CUDA, "cudaFreeHost failed"); }
    return PIXSHT_OK;
}
extern "C" int pixsht_host_register(void* ptr, size_t bytes)
{
    if (!ptr || bytes == 0) return fail(PIXSHT_ERR_ARG, "bad argument");
#ifndef PIXSHT_EMU
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) { (void)cudaGetLastError(); return fail(PIXSHT_ERR_NODEVICE, "no CUDA device available"); }
    const cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable);
    if (e == cudaErrorHostMemoryAlreadyRegistered) { (void)cudaGetLastError(); return PIXSHT_OK; }
    if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(PIXSHT_ERR_CUDA, std::string("cudaHostRegister: ") + cudaGetErrorString(e)); }
#endif
    return PIXSHT_OK;
}
extern "C" int pixsht_host_unregister(void* ptr)
{
    if (!ptr) return PIXSHT_OK;
#ifndef PIXSHT_EMU
    const cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess && e != cudaErrorHostMemoryNotRegistered) { (void)cudaGetLastError(); return fail(PIXSHT_ERR_CUDA, std::string("cudaHostUnregister: ") + cudaGetErrorString(e)); }
    (void)cudaGetLastError();
#endif
    return PIXSHT_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// introspection
// ---------------------------------------------------------------------------------------------------------------
extern "C" int pixsht_plan_info(const pixsht_plan* P, int32_t info[16])
{
    if (!P || !info) return fail(PIXSHT_ERR_ARG, "null argument");
    for (int i = 0; i < 16; ++i) info[i] = 0;
    info[0] = P->nphi; info[1] = P->nrings; info[2] = P->lmax; info[3] = P->mmax; info[4] = P->dtype; info[5] = P->device;
    info[6] = P->npairs; info[7] = P->sm_count; info[8] = P->nfft; info[9] = P->launches; info[10] = P->R0; info[11] = P->R2; info[12] = P->R0a; info[13] = P->R2a;
    info[14] = P->multi ? multi_ndev(P->multi) : 1;
    info[15] = P->fft_threads | (P->fft_edge ? (1 << 16) : 0) | (P->fft_rows ? (1 << 17) : 0) | ((P->fft_edge ? P->nsp : P->nsp_plain) << 20);
    return PIXSHT_OK;
}

// executed vs nominal (l, m, ring pair) steps of one spin family: the activation table decides what runs
// pairs [p1, p2) run the two-step spin-0 kernels (table lact2s, steps of two degrees): their steps are counted in out[2]
__global__ void k_count_work(int lmax, int mmax, int npairs, int s, const int* __restrict__ lact, unsigned long long* out, int p1 = 0, int p2 = 0,
                             const int* __restrict__ lact2s = nullptr)
{
    const long long n = (long long)(mmax + 1) * npairs;
    unsigned long long exec = 0, nominal = 0, exec2 = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int m = (int)(i / npairs);
        const int l0 = m > s ? m : s;
        if (l0 <= lmax) nominal += (unsigned long long)(lmax - l0 + 1);
        const int pr = (int)(i - (long long)m * npairs);
        if (pr >= p1 && pr < p2) {
            const int la = lact2s[i], lmaxp = twostep_lmax(lmax, m);
            if (la <= lmaxp) exec2 += (unsigned long long)(lmaxp - la + 1);
        } else {
            const int la = lact[i];
            if (la <= lmax) exec += (unsigned long long)(lmax - la + 1);
        }
    }
    atomicAdd(&out[0], exec); atomicAdd(&out[1], nominal); atomicAdd(&out[2], exec2);
}

// executed steps per m (one CTA per m): the load-balancing weight of the m-sharded multi-GPU partition
__global__ void k_count_work_m(int lmax, int npairs, const int* __restrict__ lact, double* out)
{
    __shared__ double red[128];
    const int m = blockIdx.x;
    double acc = 0.0;
    for (int p = threadIdx.x; p < npairs; p += blockDim.x) {
        const int la = lact[(size_t)m * npairs + p];
        if (la <= lmax) acc += (double)(lmax - la + 1);
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 64; o > 0; o >>= 1) { if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) out[m] = red[0];
}

// executed steps per m of one spin family (host vector of mmax+1); the caller holds the plan's lock or owns the plan
static int work_per_m(pixsht_plan* P, int spin, std::vector<double>& out)
{
    int rc = check_device(P->device); if (rc) return rc;
    rc = ensure_seek(P, spin, P->stream); if (rc) return rc;
    DevBuf<double> d;
    if (d.alloc(P->mmax + 1)) return fail(PIXSHT_ERR_NOMEM, "allocation failed");
    PIXSHT_LAUNCH(k_count_work_m, P->mmax + 1, 128, 0, P->stream, P->lmax, P->npairs, spin == 0 ? P->d_lact0.p : P->d_lact2.p, d.p);
    CU(cudaGetLastError());
    out.resize(P->mmax + 1);
    CU(cudaMemcpyAsync(out.data(), d.p, sizeof(double) * (P->mmax + 1), cudaMemcpyDeviceToHost, P->stream));
    CU(cudaStreamSynchronize(P->stream));
    return PIXSHT_OK;
}

extern "C" int pixsht_plan_work_per_m(pixsht_plan* P, int spin, double* out)
{
    if (!P || !out || (spin != 0 && spin != 2)) return fail(PIXSHT_ERR_ARG, "bad argument");
    std::lock_guard<std::mutex> lock(P->mu);
    pixsht_plan* Q = P->multi ? multi_first_sub(P->multi) : P;
    std::vector<double> w;
    int rc = work_per_m(Q, spin, w); if (rc) return rc;
    memcpy(out, w.data(), sizeof(double) * w.size());
    return PIXSHT_OK;
}

extern "C" int pixsht_plan_work(pixsht_plan* P, int spin, double out[2])
{
    if (!P || !out || (spin != 0 && spin != 2)) return fail(PIXSHT_ERR_ARG, "bad argument");
    std::lock_guard<std::mutex> lock(P->mu);
    if (P->multi) P = multi_first_sub(P->multi);   // tables are replicated: every shard's plan reports the same counts
    int rc = check_device(P->device); if (rc) return rc;
    rc = ensure_seek(P, spin, P->stream); if (rc) return rc;
    DevBuf<unsigned long long> d;
    if (d.alloc(3)) return fail(PIXSHT_ERR_NOMEM, "allocation failed");
    CU(cudaMemsetAsync(d.p, 0, 24, P->stream));
    // spin 0: the pairs of the two-step chunks execute steps of two degrees at 6 FP64 ops each = 1.5 steps of the 4-op count
    int p1 = 0, p2 = 0;
    if (spin == 0) { int lo, hi; twostep_range(P, P->R0, lo, hi); p1 = std::min(P->npairs, lo * 32 * P->R0); p2 = std::min(P->npairs, hi * 32 * P->R0); }
    if (p2 > p1) { rc = ensure_twostep(P, P->stream); if (rc) return rc; }
    PIXSHT_LAUNCH(k_count_work, 1024, 256, 0, P->stream, P->lmax, P->mmax, P->npairs, spin, spin == 0 ? P->d_lact0.p : P->d_lact2.p, d.p, p1, p2,
                  p2 > p1 ? P->d_lact1.p : (const int*)nullptr);
    unsigned long long h[3] = {0, 0, 0};
    CU(cudaMemcpyAsync(h, d.p, 24, cudaMemcpyDeviceToHost, P->stream));
    CU(cudaStreamSynchronize(P->stream));
    d.release();
    out[0] = (double)h[0] + 1.5 * (double)h[2]; out[1] = (double)h[1];
    return PIXSHT_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// alm2cl: the first consumer of the alm (Healpix.alm2cl as used at test/test_transforms.jl:104-107 of the reference)
// ---------------------------------------------------------------------------------------------------------------
// C_l = (a_l0 b_l0* + 2 sum_{m=1..min(l,mmax)} Re(a_lm b_lm*)) / (2l+1); one thread per l, coalesced in l for every m
template <class C>
__global__ void k_alm2cl(int lmax, int mmax, const C* __restrict__ a, const C* __restrict__ b, double* __restrict__ cl)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l > lmax) return;
    double acc = 0.0;
    const int mtop = l < mmax ? l : mmax;
    for (int m = 0; m <= mtop; ++m) {
        const long long k = alm_index(lmax, l, m);
        const C x = a[k], y = b[k];
        const double t = (double)x.x * (double)y.x + (double)x.y * (double)y.y;
        acc += (m == 0) ? t : 2.0 * t;
    }
    cl[l] = acc / (2.0 * l + 1.0);
}

extern "C" int pixsht_alm2cl(int lmax, int mmax, const void* alm1, const void* alm2, double* cl, int dtype, int location, int device)
{
    if (!alm1 || !cl || lmax < 0 || mmax < 0 || mmax > lmax) return fail(PIXSHT_ERR_ARG, "bad argument");
    if (dtype != PIXSHT_F64 && dtype != PIXSHT_F32) return fail(PIXSHT_ERR_ARG, "dtype must be PIXSHT_F64 or PIXSHT_F32");
    if (location != PIXSHT_HOST && location != PIXSHT_DEVICE) return fail(PIXSHT_ERR_ARG, "bad location");
    if (!alm2) alm2 = alm1;
    int rc = check_device(device); if (rc) return rc;
    const size_t n = (size_t)pixsht_nalm(lmax, mmax), bytes = n * (dtype == PIXSHT_F64 ? 16 : 8);
    DevBuf<unsigned char> da, db; DevBuf<double> dcl;
    const void *pa = alm1, *pb = alm2; double* pc = cl;
    if (location == PIXSHT_HOST) {
        if (da.alloc(bytes) || dcl.alloc(lmax + 1) || (alm2 != alm1 && db.alloc(bytes))) { da.release(); db.release(); dcl.release(); return fail(PIXSHT_ERR_NOMEM, "allocation failed"); }
        CU(cudaMemcpy(da.p, alm1, bytes, cudaMemcpyHostToDevice));
        if (alm2 != alm1) CU(cudaMemcpy(db.p, alm2, bytes, cudaMemcpyHostToDevice));
        pa = da.p; pb = (alm2 != alm1) ? (const void*)db.p : (const void*)da.p; pc = dcl.p;
    }
    const int grid = (lmax + 128) / 128;
    if (dtype == PIXSHT_F64) PIXSHT_LAUNCH(k_alm2cl<double2>, grid, 128, 0, 0, lmax, mmax, (const double2*)pa, (const double2*)pb, pc);
    else PIXSHT_LAUNCH(k_alm2cl<float2>, grid, 128, 0, 0, lmax, mmax, (const float2*)pa, (const float2*)pb, pc);
    CU(cudaGetLastError());
    if (location == PIXSHT_HOST) CU(cudaMemcpy(cl, dcl.p, sizeof(double) * (lmax + 1), cudaMemcpyDeviceToHost));
    else CU(cudaStreamSynchronize(0));
    da.release(); db.release(); dcl.release();
    return PIXSHT_OK;
}

extern "C" int pixsht_plan_weights(const pixsht_plan* P, double* weights, double* theta)
{
    if (!P) return fail(PIXSHT_ERR_ARG, "null argument");
    if (weights) memcpy(weights, P->h_wgt.data(), sizeof(double) * P->nrings);
    if (theta) memcpy(theta, P->h_theta.data(), sizeof(double) * P->nrings);
    return PIXSHT_OK;
}

extern "C" const char* pixsht_last_error(void) { return g_err.c_str(); }
extern "C" const char* pixsht_version(void)
{
#ifdef PIXSHT_EMU
    return "pixsht 0.1 (HOST EMULATION BUILD - tests only)";
#else
    return "pixsht 0.1 (sm_100a)";
#endif
}
extern "C" int pixsht_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
    return n;
}

extern "C" int pixsht_measure_fma_peak(int device, double* fp64_tflops, double* fp32_tflops)
{
#ifdef PIXSHT_EMU
    (void)device; (void)fp64_tflops; (void)fp32_tflops;
    return fail(PIXSHT_ERR_UNSUPPORTED, "not available in the host emulation build");
#else
    int rc = check_device(device); if (rc) return rc;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    void* buf = nullptr; void* din = nullptr;
    CU(cudaMalloc(&buf, (size_t)blocks * threads * sizeof(double)));
    CU(cudaMalloc(&din, 16 * sizeof(double)));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    for (int pass = 0; pass < 2; ++pass) {
        const int iters = pass == 0 ? 4096 : 16384;   // fp64, fp32
        double hd[16]; float hf[16];
        for (int i = 0; i < 16; ++i) { hd[i] = 1e-3 * (i + 1); hf[i] = (float)hd[i]; }
        if (pass == 0) CU(cudaMemcpy(din, hd, sizeof(hd), cudaMemcpyHostToDevice));
        else CU(cudaMemcpy(din, hf, sizeof(hf), cudaMemcpyHostToDevice));
        float best = 1e30f;
        for (int rep = 0; rep < 4; ++rep) {
            CU(cudaEventRecord(e0, 0));
            if (pass == 0) k_fma_peak<double><<<blocks, threads>>>((double*)buf, iters, (const double*)din);
            else k_fma_peak<float><<<blocks, threads>>>((float*)buf, iters, (const float*)din);
            CU(cudaEventRecord(e1, 0));
            CU(cudaEventSynchronize(e1));
            float ms; CU(cudaEventElapsedTime(&ms, e0, e1));
            if (rep > 0 && ms < best) best = ms;
        }
        const double flops = 2.0 * 64.0 * (double)iters * (double)blocks * (double)threads;
        const double tf = flops / ((double)best * 1e-3) / 1e12;
        if (pass == 0) { if (fp64_tflops) *fp64_tflops = tf; }
        else { if (fp32_tflops) *fp32_tflops = tf; }
    }
    cudaFree(din);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(buf);
    CU(cudaGetLastError());
    return PIXSHT_OK;
#endif
}

#ifdef PIXSHT_FFT_PROF
// profiling builds only (not declared in include/pixsht.h): per-phase cycle sums of the FFT kernels since the last call
extern "C" int pixsht_debug_fft_prof(unsigned long long* out32)
{
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpyFromSymbol(out32, g_fft_prof, 32 * sizeof(unsigned long long)));
    unsigned long long z[32] = {0};
    CU(cudaMemcpyToSymbol(g_fft_prof, z, sizeof(z)));
    return PIXSHT_OK;
}
#endif

#include "multi.inl"
