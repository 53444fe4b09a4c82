/*
 * pixsht.h -- C ABI of libpixsht.so, the B200-native (sm_100a) spherical-harmonic-transform engine that replaces the
 * libsharp2 calls on Pixell.jl's map2alm / alm2map hot path.
 *
 * What each entry point replaces in the reference (simonsobs/Pixell.jl v0.2.9, file:line under /root/reference):
 *
 *   pixsht_plan_create     <- the per-call setup of src/transforms.jl:33-63 (make_cc_geom_info: ring grid, CC weights
 *                             x 2pi/nphi, phi0, offsets, ccall sharp_make_geom_info) and :94 (make_triangular_alm_info)
 *                             and the band bookkeeping of :66-82 (create_sht_band: flips + zero padding, done here as
 *                             index arithmetic inside the FFT kernels instead of a host copy).
 *   pixsht_execute         <- sharp_execute!(SHARP_MAP2ALM|SHARP_ALM2MAP, spin, alms, maps, geom, alm_info, SHARP_DP)
 *                             at src/transforms.jl:101-106, 128-132, 185-194, 214-218, 240-244.  ncomp = 1 is the
 *                             spin-0 job, 2 the spin-2 (Q,U)<->(E,B) job, 3 runs both (the IQU path of :138-165,254).
 *   pixsht_plan_destroy    <- Libsharp.jl finalizers (sharp_destroy_geom_info / sharp_destroy_alm_info).
 *   pixsht_stage_*         <- no reference counterpart (the reference is single-process); the m-sharded multi-GPU
 *                             pipeline of SURVEY.md 8(e) drives these around an NCCL all-to-all.
 *
 * A libsharp2-symbol-compatible shim over this API is declared in include/pixsht_sharp_shim.h.
 *
 * Conventions (identical to the reference's):  alm = complex (re,im interleaved), triangular m-major,
 * idx0(l,m) = m(2 lmax+1-m)/2 + l, m >= 0 only;  maps = caller's column-major (nx, ny) arrays (RA index fastest), in
 * the caller's own orientation -- the flips of get_flip_slices (src/transforms.jl:25-30) are described by pixsht_geom,
 * not applied by the caller.  All functions return PIXSHT_OK (0) or an error code; pixsht_last_error() gives the text.
 * Nothing aborts.  There is no CPU fallback: without a CUDA device every compute entry point returns PIXSHT_ERR_NODEVICE.
 */
#ifndef PIXSHT_H
#define PIXSHT_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct pixsht_plan pixsht_plan;

enum { PIXSHT_OK = 0, PIXSHT_ERR_ARG = 1, PIXSHT_ERR_CUDA = 2, PIXSHT_ERR_UNSUPPORTED = 3, PIXSHT_ERR_NOMEM = 4, PIXSHT_ERR_NODEVICE = 5 };
enum { PIXSHT_F64 = 0, PIXSHT_F32 = 1 };             /* element type of maps and alm at the boundary */
enum { PIXSHT_MAP2ALM = 0, PIXSHT_ALM2MAP = 1 };     /* numerically equal to libsharp2's SHARP_MAP2ALM / SHARP_ALM2MAP */
enum { PIXSHT_HOST = 0, PIXSHT_DEVICE = 1 };
enum { PIXSHT_POLCONV_COSMO = 0, PIXSHT_POLCONV_IAU = 1 };   /* Stokes-U sign convention of the caller's maps (pixsht_plan_set_polconv) */
enum { PIXSHT_RINGS_CC = 0, PIXSHT_RINGS_FEJER1 = 1 };  /* ring scheme of pixsht_geom */         /* where the alm / map pointers passed to pixsht_execute live */

/* How the caller's (nx, ny) map sits on the full-sky ring grid (SURVEY.md A.1). */
typedef struct pixsht_geom {
    int32_t nphi;          /* pixels of a full ring           = fullringsize(wcs)   (src/transforms.jl:3-4)   */
                           /* any length libsharp2 takes: even or odd, any prime factors (2/3/5-smooth even lengths whose
                              nphi/2 complex samples fit 227 KB of shared memory take the fast path; the rest use global
                              work buffers); limit nphi <= 131070 (even) / 65535 (odd) -> PIXSHT_ERR_UNSUPPORTED      */
    int32_t nrings_total;  /* rings of the full-sky grid      = fullringnum(wcs)    (src/transforms.jl:7-8)   */
    int32_t ring_first;    /* 0-based full-sky index of the band's first ring, rings ascending in theta (:11-22) */
    int32_t nrings;        /* rings in the map (= ny)                                                            */
    int32_t nx;            /* columns in the map (<= nphi); band columns nx..nphi-1 are zeros (:70-75)          */
    int32_t flipx;         /* 1: band column i is map column nx-1-i  (cdelt1 < 0, :25-30)                       */
    int32_t flipy;         /* 1: band ring r is map row ny-1-r       (cdelt2 > 0, :25-30)                       */
    int32_t ring_scheme;   /* PIXSHT_RINGS_CC: theta_k = pi k/(N-1), Clenshaw-Curtis weights (the reference's only SHT grid,
                              src/transforms.jl:44-46); PIXSHT_RINGS_FEJER1: theta_k = pi (k+1/2)/N, Fejer-1 weights (the
                              CarFejer1 grid of src/projections/car_proj.jl:14-19, which has no SHT path upstream)   */
    double phi0;           /* RA (radians) of band column 0 (:41)                                                */
} pixsht_geom;

/* ---- plans ---------------------------------------------------------------------------------------------- */
int pixsht_plan_create(pixsht_plan **out, const pixsht_geom *geom, int lmax, int mmax, int dtype, int device);
/* generic iso-latitude ring set with explicit colatitudes and quadrature weights (all rings nphi samples, first
 * sample at phi0, rings ascending in theta, maps stored ring-major without flips: nx = nphi).  Used by the shim. */
int pixsht_plan_create_rings(pixsht_plan **out, int nrings, const double *theta, const double *weight, int nphi,
                             double phi0, int lmax, int mmax, int dtype, int device);
/* Multi-GPU plan: ONE process drives `ndev` GPUs of a node behind the same blocking pixsht_execute call -- the shape of the
 * reference's transform (sharp_execute! on caller-owned host arrays, src/transforms.jl:88-108, 185-194), no second process,
 * no torch, no NCCL.  m is sharded (contiguous segments of equal measured Legendre work, dealt to the GPUs), rings are split
 * into contiguous slabs, the phase transpose between the two stages happens inside the FFT kernels' row loads / stores over
 * peer memory (cudaDeviceEnablePeerAccess: the GPUs must be NVLink / NVSwitch peers -> PIXSHT_ERR_UNSUPPORTED otherwise).
 * Each GPU copies its alm columns / map rows straight from / to the caller's arrays.  A device index may appear more than
 * once in `devices` (each entry is its own shard; that is how a single-GPU box exercises this path).
 * On such a plan: pixsht_execute takes whole arrays in host memory (or any memory the GPUs can copy from; `location` is
 * ignored); pixsht_execute_batch deals whole transforms to the GPUs; the stage API and pixsht_plan_set_stream do not apply. */
int pixsht_plan_create_multi(pixsht_plan **out, const pixsht_geom *geom, int lmax, int mmax, int dtype, int ndev, const int *devices);
/* shard `shard` of a multi-GPU plan: info = { device, first band ring, ring count, number of m values }; m_list (may be NULL)
 * receives the shard's m values, ascending */
int pixsht_multi_shard(const pixsht_plan *plan, int shard, int32_t info[4], int32_t *m_list);
/* The same transform with the data already distributed over the GPUs (nothing is copied): alms[d*ncomp + c] = device pointer
 * on shard d's GPU to a FULL-LENGTH alm array of which only the shard's m columns are read / written;  maps[d*ncomp + c] =
 * device pointer on shard d's GPU to the shard's slab of map rows (ring count * nx elements, the caller's row order). */
int pixsht_execute_sharded(pixsht_plan *plan, int direction, int ncomp, void *const *alms, void *const *maps);
void pixsht_plan_destroy(pixsht_plan *plan);

/* ---- host memory ------------------------------------------------------------------------------------------ */
/* Page-locked host memory for the caller's maps and alm: pixsht_execute(..., PIXSHT_HOST) overlaps its copies with the
 * kernels only from / to page-locked memory (copies from pageable memory are staged by the driver and serialise the
 * pipeline).  pixsht_host_alloc / pixsht_host_free own an allocation; pixsht_host_register / pixsht_host_unregister
 * page-lock an array the caller already owns (e.g. a Julia Array) for the lifetime of the registration. */
int pixsht_host_alloc(void **ptr, size_t bytes);
int pixsht_host_free(void *ptr);
int pixsht_host_register(void *ptr, size_t bytes);
int pixsht_host_unregister(void *ptr);

/* ---- transforms ----------------------------------------------------------------------------------------- */
/* direction: PIXSHT_MAP2ALM | PIXSHT_ALM2MAP.  ncomp: 1 = T (spin 0), 2 = Q,U <-> E,B (spin 2), 3 = T,Q,U <-> T,E,B.
 * alms[c]: nalm complex numbers of the plan's dtype; maps[c]: nx*ny reals of the plan's dtype.
 * location: PIXSHT_HOST (pageable or pinned host memory; copies are inside the call) or PIXSHT_DEVICE (pointers on the
 * plan's device; the call is enqueued on the plan's stream and synchronised before returning).
 * Outputs are overwritten (SHARP_ADD is never used by the reference). */
int pixsht_execute(pixsht_plan *plan, int direction, int ncomp, void *const *alms, void *const *maps, int location);

/* map2alm refined by niter Jacobi iterations, a <- a + A(m - Y a), on one GPU.  niter = 0 is pixsht_execute(MAP2ALM)
 * exactly.  maps are inputs only and are not modified.  Between iterations the maps, the residual and the alm stay on the
 * device; with host pointers the maps are copied in once and the alm out once.
 * (healpy's map2alm(iter=...), python-pixell's map2alm(niter=...).)  The plain analysis is exact on the Clenshaw-Curtis grid
 * only for lmax <= (nrings-1)/2; above that each iteration removes most of the remaining error, except near the ring's Nyquist
 * lmax (the columns m << lmax converge slowly there) and on cut-sky bands, which barely improve (DESIGN.md section 10).
 * ncomp, alms, maps and location as in pixsht_execute; niter < 0 -> PIXSHT_ERR_ARG; a multi-GPU plan with niter > 0 ->
 * PIXSHT_ERR_UNSUPPORTED.  Device pointers use the plan's stream (or the caller's, pixsht_plan_set_stream) and the call
 * synchronises it; pixsht_plan_set_polconv applies to the maps and to the residual alike.  The plan keeps ncomp residual
 * maps of nx*ny elements of its dtype, allocated by the first call with niter > 0. */
int pixsht_map2alm_iter(pixsht_plan *plan, int ncomp, void *const *alms, void *const *maps, int niter, int location);

/* Batch of nbatch independent spin-0 transforms on one geometry (simulation sweeps; no counterpart in the reference, which
 * transforms one map per libsharp job).  alms[b] / maps[b] as for ncomp = 1.  Up to four maps share one recurrence per
 * (m, ring pair): 2 + 2 NB FP64 ops per (l, m, ring pair) instead of 4 NB. */
int pixsht_execute_batch(pixsht_plan *plan, int direction, int nbatch, void *const *alms, void *const *maps, int location);

/* Run pixsht_execute on the caller's CUDA stream (cudaStream_t passed as void*; NULL is the legacy default stream) when
 * use_caller_stream != 0, or go back to the plan's own stream.  The call still synchronises that stream before returning. */
int pixsht_plan_set_stream(pixsht_plan *plan, void *stream, int use_caller_stream);

/* Stokes-U sign convention of the maps passed to this plan.  The transforms use the COSMO / HEALPix convention (libsharp2's, the
 * one the reference computes in).  The reference converts an IAU file at read time by negating U on the host
 * (read_map -> resolve_polcconv!, src/enmap.jl:178-196, 209-215); with PIXSHT_POLCONV_IAU the caller keeps the file's values and
 * the sign is applied inside the ring-FFT kernels' row loads (map2alm) and stores (alm2map): no pass over the map.  Applies to
 * the U component of ncomp = 2 and ncomp = 3 calls, on single- and multi-GPU plans; default PIXSHT_POLCONV_COSMO. */
int pixsht_plan_set_polconv(pixsht_plan *plan, int polconv);

/* Pixel areas (steradians) of the rows of the map described by `geom`, one value per map row (CAR pixel areas do not depend
 * on RA), in the caller's row order: (sin dec_hi - sin dec_lo) |d alpha| with the row edges clipped at the poles.  Replaces
 * pixareamap / pixareamap! of the reference (src/projections/car_proj.jl:265-273, src/enmap_ops.jl:124-138); used as ring
 * weights through pixsht_plan_create_rings it gives the pixel-area-weighted analysis.  Host arithmetic, no device needed. */
int pixsht_ring_pixarea(const pixsht_geom *geom, double *area /* geom->nrings */);

/* per-stage device time (ms, CUDA events) of the last pixsht_execute on this plan:
 * device pointers: [1] Legendre stage, [2] FFT stage, [4] whole call (host wall clock), [6] the spin-0 Legendre kernel
 * alone (leg_synth<0,R> or leg_anal<0,R>), [7] the spin-2 Legendre kernel alone;
 * host pointers (copies, Legendre and FFT are pipelined over three streams, so stages overlap): [4] whole call,
 * [5] span of the compute stream; the rest 0;
 * pixsht_map2alm_iter with niter > 0 (either location): [4] whole call, [5] span of the compute stream; the rest 0 */
int pixsht_get_timings(const pixsht_plan *plan, double ms[8]);

/* ---- stage API for the m-sharded multi-GPU pipeline (device pointers, asynchronous on `stream`) ------------
 * m-sharded phase layout: a rank's phase buffer holds ITS m values for ALL band rings, element (ring, c, i) at
 * ((ring*ncomp + c)*row_len + i) with i the position of m in the rank's m_list and row_len >= nm.  The Legendre stages work
 * on that local buffer.  The FFT stages, which run on a rank's slab of rings over all m, reach every m through a device
 * table d_mtab of 2*(mmax+1) int64: [2m] = address of element (ring 0, comp 0, m) in the buffer of the rank that owns m
 * (pixsht_shared_open for peers), [2m+1] = that buffer's row_len.  With m dealt to ranks in runs of 16 the remote
 * accesses are 256-byte runs, so the phase transpose of SURVEY.md 8(e) happens inside the FFT kernels' own row loads /
 * stores over NVLink and there is no separate exchange pass.
 * Element types: phase rows and the alm of the Legendre stages are always complex double (a Float32 plan converts at the
 * pixsht_execute boundary only); the maps of the FFT stages are of the plan's dtype. */
int64_t pixsht_phase_row_len(const pixsht_plan *plan);   /* row length of the single-GPU layout (mmax+1 rounded up to 8) */
/* Which spin families the following pixsht_stage_* calls on this plan process: the T component (spin0), the Q/U <-> E/B pair
 * (spin2), or both (the default).  Component arrays and the phase layout stay those of the full ncomp set; a caller uses this
 * to pipeline an IQU transform per family (T on the device while Q/U are still on the wire: pixsht/distributed.py). */
int pixsht_plan_set_stage_families(pixsht_plan *plan, int spin0, int spin2);
/* Legendre stage over the m values m_list[0..nm) (device array of int32, or NULL for m = 0..nm-1). */
int pixsht_stage_alm2phase(pixsht_plan *plan, int ncomp, const void *const *d_alms, int nm, const int32_t *d_m_list,
                           void *d_phase, int64_t row_len, void *stream);
int pixsht_stage_phase2alm(pixsht_plan *plan, int ncomp, const void *d_phase, int64_t row_len, int nm, const int32_t *d_m_list,
                           void *const *d_alms, void *stream);
/* FFT stage over band rings [ring_begin, ring_begin+ring_count); d_maps are the full caller-layout maps (only the rows of
 * those rings are touched). */
int pixsht_stage_phase2map(pixsht_plan *plan, int ncomp, const int64_t *d_mtab, int ring_begin, int ring_count,
                           void *const *d_maps, void *stream);
int pixsht_stage_map2phase(pixsht_plan *plan, int ncomp, const void *const *d_maps, int ring_begin, int ring_count,
                           const int64_t *d_mtab, void *stream);
/* Peer-visible device memory for the phase buffers (CUDA IPC between the one-process-per-GPU ranks of a node):
 * alloc on the owner and export a 64-byte handle; open maps a peer's buffer into this process (peer access over
 * NVLink is enabled lazily); close unmaps an opened buffer; free releases an owned one. */
int pixsht_shared_alloc(int device, size_t bytes, void **dptr, unsigned char handle[64]);
int pixsht_shared_open(int device, const unsigned char handle[64], void **dptr);
int pixsht_shared_close(void *dptr);
int pixsht_shared_free(void *dptr);

/* ---- alm2cl ---------------------------------------------------------------------------------------------- */
/* Healpix.alm2cl as the reference's tests use it (test/test_transforms.jl:104-107): cross (or auto, alm2 = NULL) spectrum
 * C_l = (a_l0 b_l0* + 2 sum_{m>=1} Re(a_lm b_lm*)) / (2l+1), l = 0..lmax, of two alm in the triangular m-major layout.
 * dtype: element type of the alm (complex double / complex float); cl: lmax+1 doubles; location as in pixsht_execute. */
int pixsht_alm2cl(int lmax, int mmax, const void *alm1, const void *alm2, double *cl, int dtype, int location, int device);

/* ---- introspection -------------------------------------------------------------------------------------- */
int64_t pixsht_nalm(int lmax, int mmax);
int pixsht_plan_info(const pixsht_plan *plan, int32_t info[16]);
/* info: [0] nphi [1] nrings [2] lmax [3] mmax [4] dtype [5] device [6] npairs (north/south folded ring pairs)
 *       [7] SM count [8] FFT length [9] kernels launched by the last execute [10..13] ring pairs per thread of the
 *       spin-0 / spin-2 synthesis and spin-0 / spin-2 analysis kernels [14] number of GPUs (shards) of the plan
 *       [15] ring-FFT plan: threads per CTA | bit 16: outer passes fused into the row I/O (fft_edge.cuh) | bit 17: work buffers in
 *            global memory | bits 20+: number of super-passes */
/* (l, m, ring pair) steps of one spin family (0 or 2): out[0] = executed by the kernels (the plan-time activation table
 * skips what stays below 2^-90), out[1] = nominal count of SURVEY.md 8(d) (every l >= max(m,|s|) for every pair) */
int pixsht_plan_work(pixsht_plan *plan, int spin, double out[2]);
/* executed steps per m (mmax+1 doubles, host): the load-balancing weight of the m-sharded multi-GPU partition */
int pixsht_plan_work_per_m(pixsht_plan *plan, int spin, double *out);
int pixsht_plan_weights(const pixsht_plan *plan, double *weights /* nrings */, double *theta /* nrings */);
const char *pixsht_last_error(void);
const char *pixsht_version(void);
int pixsht_device_count(void);
/* register-resident DFMA / FFMA chain micro-benchmark on `device`: measured peak in TFLOP/s (1 FMA = 2 flop) */
int pixsht_measure_fma_peak(int device, double *fp64_tflops, double *fp32_tflops);

#ifdef __cplusplus
}
#endif
#endif /* PIXSHT_H */
