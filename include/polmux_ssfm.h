/*
 * polmux_ssfm.h -- C ABI of the B200-native split-step Fourier fiber channel.
 *
 * Drop-in boundary for ONE path of the Optilux/Polmux reference: the SSFM
 * propagation loop inside fiber.m.  Every entry point names the reference
 * interface it replaces (file:line under the reference tree).  Plain C, POD
 * only, no exceptions cross the boundary, no torch / MATLAB types.
 *
 * Conventions
 *   - all lengths in [m], times [ns], powers [mW]  (fiber.m units)
 *   - complex samples are IEEE double (the reference's arithmetic); the
 *     "field" is two polarizations x nfc columns x nfft samples, column-major
 *     like GSTATE.FIELDX / GSTATE.FIELDY (reset_all.m:158-159)
 *   - every function returns PMX_OK (0) or a negative pmx_status; the text of
 *     the last error is available through pmx_last_error()
 *   - a pmx_ctx owns one CUDA device, one stream and its cached tables; it is
 *     thread-compatible (one ctx per host thread), not thread-safe
 *   - there is NO CPU fallback: without a usable CUDA device pmx_ctx_create
 *     fails with PMX_ERR_CUDA
 */
#ifndef POLMUX_SSFM_H
#define POLMUX_SSFM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PMX_VERSION 100 /* 0.1.0 */

typedef enum pmx_status {
    PMX_OK = 0,
    PMX_ERR_INVALID = -1,      /* bad argument (message says which)                    */
    PMX_ERR_UNSUPPORTED = -2,  /* valid in the reference, not built here (message)     */
    PMX_ERR_CUDA = -3,         /* CUDA runtime / driver error                          */
    PMX_ERR_PLATE_INDEX = -4,  /* trunk counter ran past nplates: the reference fails  */
                               /* with an index error at fiber.m:910 (SURVEY A.8.1)    */
    PMX_ERR_NUMERIC = -5,      /* NaN/Inf met in step control                          */
    PMX_ERR_XPM_VECTOR = -6    /* fiber.m:854 'The CNLSE with separate fields is not   */
                               /* yet implemented'                                     */
} pmx_status;

typedef enum pmx_precision { PMX_F64 = 0, PMX_F32 = 1 } pmx_precision;

/* Host-side layouts of a field handed across the boundary. */
typedef enum pmx_layout {
    PMX_PLANAR = 0,  /* four real arrays xr, xi, yr, yi -- the split storage the    */
                     /* reference's MEX files use (mxGetPr/mxGetPi, fastexp.c:61-63)*/
    PMX_COMPLEX = 1  /* two interleaved complex arrays x, y (re,im,re,im,...)       */
} pmx_layout;

typedef enum pmx_disp_mode { PMX_DISP_VECTOR = 0, PMX_DISP_SCALAR = 1 } pmx_disp_mode;

typedef struct pmx_ctx pmx_ctx;
typedef struct pmx_plan pmx_plan;         /* one fiber() worth of device constants */
typedef struct pmx_devfield pmx_devfield; /* a field resident in HBM               */

/* ---- context -------------------------------------------------------------- */
int pmx_version(void);
int pmx_device_count(void);
int pmx_ctx_create(pmx_ctx** ctx, int device_id);
void pmx_ctx_destroy(pmx_ctx* ctx);
/* ctx may be NULL: returns the calling thread's last error text. */
const char* pmx_last_error(const pmx_ctx* ctx);
/* Blocks until all work queued on the ctx stream is done. */
int pmx_ctx_sync(pmx_ctx* ctx);
/* Raw cudaStream_t of the ctx, so a caller can record its own events on it. */
void* pmx_ctx_stream(pmx_ctx* ctx);

/* ---- the fiber --------------------------------------------------------------
 * pmx_fiber_desc is the argument list of
 *   [firstdz,ncycle,ux,uy,brf] = matrix_ssfm(ux,uy,betat,db1,dzmaxt,dphimaxt,
 *        gam,alphalin,nfc,Lf,nplates,manakov,fls,brf)          fiber.m:459-460
 * (the seam inside fiber.m:381-383), plus a batch axis over independent
 * realizations.  Everything above that seam in fiber.m:126-369 is host scalar
 * set-up and stays on the caller's side.
 */
typedef struct pmx_fiber_desc {
    int64_t nfft;        /* rows of FIELDX = NSYMB*NT (fiber.m:133); power of two, 2^6..2^24 */
    int32_t nfc;         /* columns of FIELDX (fiber.m:132): <= 64; <= 8 for nfft < 2^12 (on-chip: one cluster) */
    int32_t batch;       /* independent realizations propagated by one call (>=1); batch*nfc <= 65535 */
    int32_t precision;   /* pmx_precision                                                     */
    int32_t manakov;     /* strcmp(manakov,'yes')   fiber.m:499                               */
    double length;       /* Lf        fiber.m:459 */
    double alphalin;     /* [1/m]     fiber.m:302 */
    double dzmaxt;       /* fiber.m:157-251       */
    double dphimaxt;     /* may be +Inf (linear flags -> exactly one step) */
    const double* gam;   /* [nfc] 1/mW/m, BEFORE the Manakov 8/9 (applied inside, fiber.m:500) */
    int32_t fls[4];      /* [g p s x]  fiber.m:157 */
    int32_t nplates;     /* fiber.m:297 / 265 / 272 */
    int32_t plate_sets;  /* 1: all realizations share the plates; batch: one draw each */
    const double* db0;     /* [plate_sets][nplates]  brf.db0      fiber.m:266,274 */
    const double* theta;   /* [plate_sets][nplates]  brf.theta    fiber.m:267,275 */
    const double* epsilon; /* [plate_sets][nplates]  brf.epsilon  fiber.m:268,276 */
    const double* betat;   /* [nfc][nfft] host, fiber.m:350-356 (FFT order)        */
    const double* db1;     /* [nfc][nfft] host, fiber.m:358; NULL means zeros      */
    /* Optional scalar dispersion mode.  With disp_mode == PMX_DISP_SCALAR the library rebuilds
     * the two vectors per bin from the scalars fiber.m:350-362 builds them from --
     *   omega = 2*pi*symbolrate*FN,  FN = signed FFT bin / nsymb            (reset_all.m:153)
     *   betat = omega*beta1 + 0.5*omega^2*beta2 + omega^3*b30/6,  db1 = dgdrms*omega
     * -- and betat / db1 may be NULL: nothing but the field crosses PCIe.  omega, db1 and the
     * first two betat terms are bit-identical to the host vectors; the cubic term may differ by
     * one ulp (omega^3 is formed by two multiplications, b30/6 is pre-divided). */
    int32_t disp_mode;     /* pmx_disp_mode */
    int32_t nsymb;         /* GSTATE.NSYMB */
    int32_t nt;            /* GSTATE.NT    */
    int32_t scalar_field;  /* 1: the scalar path of fiber.m:372-380 (FIELDY empty, no 'p' flag): Y is absent and the
                            * 'x' flag couples the columns (nl_step, fiber.m:793-799); 0: matrix_ssfm            */
    double symbolrate;     /* GSTATE.SYMBOLRATE [GBaud] */
    double b30;            /* fiber.m:309-311 [ns^3/m] */
    double dgdrms;         /* fiber.m:269/277/284 [ns]; 0 without the 'p' flag */
    const double* beta1;   /* [nfc] fiber.m:323/327 */
    const double* beta2;   /* [nfc] fiber.m:330-332 */
    /* Resuming a propagation part-way (scalar_ssfm with x.dphiadapt, fiber.m:588-611: the first step is taken by the
     * local-error method on the host side of the boundary, the loop then starts at zprop = zdone + dz with the step the
     * adaptive method proposed).  Both zero: a fresh fiber, first step from nextstep (fiber.m:512 / :585). */
    double z_start;        /* [m] length already propagated when the loop starts */
    double dz_first;       /* [m] first step of the loop; 0 = nextstep on the incoming field */
} pmx_fiber_desc;

typedef struct pmx_field {
    int32_t layout;   /* pmx_layout */
    int32_t reserved;
    /* PMX_PLANAR : xr,xi,yr,yi each [batch][nfc][nfft] doubles; xi / yi may be
     *              NULL on input (purely real array, as mxGetPi returns NULL);
     *              yr may be NULL on input (FIELDY empty -> zeros, fiber.m:286).
     * PMX_COMPLEX: xr -> complex X array, yr -> complex Y array; xi, yi unused. */
    double* xr;
    double* xi;
    double* yr;
    double* yi;
} pmx_field;

/* Per-realization outputs of matrix_ssfm that the caller prints or checks. */
typedef struct pmx_fiber_result {
    double* firstdz;   /* [batch]  fiber.m:516 */
    int32_t* ncycle;   /* [batch]  fiber.m:506,536 */
    int32_t* ntot;     /* [batch]  trunk counter after the run (== nplates when 'p') */
    int32_t* status;   /* [batch]  0 or a pmx_status (e.g. PMX_ERR_PLATE_INDEX)      */
    /* optional trace of the step schedule, for tests (may be NULL):
     * trace_dz[b*trace_cap + i] = length of step i, trace_ntrunk likewise.    */
    double* trace_dz;
    int32_t* trace_ntrunk;
    int32_t trace_cap;
} pmx_fiber_result;

/* One call == one fiber(x,flag) on host buffers, in place: H2D, the whole SSFM
 * loop on the device, D2H.  Replaces the dispatch at fiber.m:381-383. */
int pmx_fiber_run(pmx_ctx* ctx, const pmx_fiber_desc* desc, pmx_field* io, pmx_fiber_result* out);

/* ---- HBM-resident API (span loops, Monte-Carlo batches, benchmarks) --------- */
/* batch*nfc <= 65535 (the kernels put a field's realization-columns in one grid dimension); larger fields return
 * PMX_ERR_UNSUPPORTED, as does a plan (pmx_plan_create, pmx_filter_create, pmx_dbp_create) with batch*nfc above it. */
int pmx_field_create(pmx_ctx* ctx, int64_t nfft, int32_t nfc, int32_t batch, int32_t precision,
                     pmx_devfield** f);
void pmx_field_destroy(pmx_devfield* f);
/* b0..b0+nb-1: realizations to transfer; host arrays hold nb realizations. */
int pmx_field_upload(pmx_devfield* f, const pmx_field* host, int32_t b0, int32_t nb);
int pmx_field_download(pmx_devfield* f, pmx_field* host, int32_t b0, int32_t nb);
/* 1 when `p` points into page-locked (CUDA-registered) host memory, 0 when not (or when no device is usable).  The
 * host mirror uses it to decide whether a received field may be written back into the caller's own arrays: pinned
 * buffers are reused in place (no staging copy), ordinary arrays are never overwritten behind the caller's back. */
int pmx_host_is_pinned(const void* p);
/* dst[b] = src[0] for all b (same Tx field for every realization). */
int pmx_field_broadcast(pmx_devfield* dst, const pmx_devfield* src);
/* Raw device pointer of the interleaved (xr,xi,yr,yi) sample array (doubles, or floats for PMX_F32 fields).
 * Layout inside a column: for nfft = 2^m in [2^12, 2^24] the samples are stored TRANSPOSED with respect to the
 * four-step split N1 = 2^floor(m/2), N2 = nfft/N1 -- time sample n1*N2 + n2 at position n2*N1 + n1 -- so that the
 * time-domain passes of the SSFM stream contiguous rows; other sizes are in natural order.  pmx_field_upload /
 * pmx_field_download convert from / to time order. */
void* pmx_field_device_ptr(pmx_devfield* f);

/* Uploads betat/db1/plates, builds twiddle tables (cached in ctx by nfft). */
int pmx_plan_create(pmx_ctx* ctx, const pmx_fiber_desc* desc, pmx_plan** plan);
void pmx_plan_destroy(pmx_plan* plan);
/* Replace the plate angles of an existing plan (new Monte-Carlo draw). */
int pmx_plan_set_plates(pmx_plan* plan, int32_t plate_sets, const double* db0, const double* theta,
                        const double* epsilon);
/* The SSFM loop on a resident field (asynchronous wrt. the host except for the
 * step-control polling; returns after the fiber is complete).  The field may belong to another context of the same
 * device (contexts are streams: a receive chain can work on one batch beside the propagation of the next); the caller
 * orders the two. */
int pmx_fiber_exec(pmx_plan* plan, pmx_devfield* f, pmx_fiber_result* out);
/* Total kernel launches issued by this ctx so far (bench `gpu_launches`). */
int64_t pmx_ctx_launch_count(const pmx_ctx* ctx);

/* Per-pass device timing for benchmarks: when enabled, every pass launch is bracketed by CUDA
 * events on the ctx stream.  ms[k] / n[k]: accumulated milliseconds and launch count of
 * k = 0 pass A (NL + column FFT), 1 pass B (row FFT + Jones + row IFFT), 2 pass C (column IFFT +
 * attenuation + max + step control), 3 initial max reduction.  Early-exit launches of finished
 * realizations are included (they are launches).  Enabling resets the counters. */
int pmx_ctx_profile(pmx_ctx* ctx, int enable);
int pmx_ctx_profile_read(pmx_ctx* ctx, double* ms, int64_t* n);

/* ---- span boundary: flat-gain amplifier with ASE --------------------------------
 * ampliflat(x,'gain',options)  ampliflat.m:61-148.
 *   field <- field*sqrt(gain) + sigma[c]*noise
 * gain   : linear power gain 10^(x/10)                       ampliflat.m:62
 * sigma  : [nfc] sqrt(mW) per column, 0 disables ASE           ampliflat.m:91-106
 * noise  : NULL -> complex standard normals from the counter-based generator
 *          (Philox4x32-10 + Box-Muller) keyed by (seed, realization), else a
 *          HOST array [batch][2*nfc][nfft] complex (options.noise, :123-129,
 *          X columns first then Y columns).
 */
int pmx_ampliflat_exec(pmx_ctx* ctx, pmx_devfield* f, double gain, const double* sigma,
                       const double* noise_host, uint64_t seed);
/* The same with the ASE on one polarization only (options.onepol = 'asex' / 'asey', ampliflat.m:107-118):
 * asepol = 1 (X), 2 (Y), 3 (both = pmx_ampliflat_exec). */
int pmx_ampliflat_exec_pol(pmx_ctx* ctx, pmx_devfield* f, double gain, const double* sigma,
                           const double* noise_host, uint64_t seed, int32_t asepol);
/* ... for a batch whose first realization has the global index realization0: the generator is keyed by
 * (seed, realization0 + b, column, sample), so the noise of a realization does not depend on how a Monte-Carlo run
 * groups or shards its realizations. */
int pmx_ampliflat_exec_at(pmx_ctx* ctx, pmx_devfield* f, double gain, const double* sigma, const double* noise_host,
                          uint64_t seed, int32_t asepol, uint64_t realization0);

/* ---- span loop: nspan x [ fiber ; ampliflat ] without returning to the host ---------------
 * The loop every multi-span script of the reference writes around its in-line devices
 *   for k=1:Nspan, fiber(x,flag); ampliflat(Gerbio,'gain',opt); end        ex06_ber.m:110-115
 * as one call: the field stays in HBM between the fibers and the amplifiers.  The fiber of every span is the one
 * the plan / pmx_fiber_desc describes; the waveplates may change from span to span (fiber.m:274-276 draws new
 * ones at every call). */
typedef struct pmx_link_desc {
    int32_t nspan;
    int32_t plate_sets;      /* 1 or batch: plate draws per span handed in below                                  */
    const double* db0;       /* [nspan][plate_sets][nplates], or NULL: every span keeps the plates of the plan    */
    const double* theta;     /* same shape */
    const double* epsilon;   /* same shape */
    double gain;             /* linear power gain of the amplifier after every span (ampliflat.m:62); 0: none     */
    const double* sigma;     /* [nfc] ASE sigma per column (ampliflat.m:91-106); NULL or zeros: no ASE            */
    const double* noise;     /* NULL: device generator keyed by seeds[k]; else HOST [nspan][batch][2*nfc][nfft]   */
                             /* complex standard normals, options.noise of span k (ampliflat.m:123-129)            */
    const uint64_t* seeds;   /* [nspan] ASE seed of every span, or NULL: seed k                                   */
    uint64_t realization0;   /* global index of the batch's first realization (device generator key, see          */
                             /* pmx_ampliflat_exec_at); 0 for a stand-alone link                                   */
    int32_t asepol;          /* 0 or 3: ASE on both polarizations; 1: X only, 2: Y only (options.onepol,           */
    int32_t reserved;        /* ampliflat.m:107-118)                                                               */
} pmx_link_desc;
/* Resident form.  out (may be NULL): arrays of nspan*batch entries, span-major ([k*batch + b]); no trace. */
int pmx_link_exec(pmx_plan* plan, pmx_devfield* f, const pmx_link_desc* link, pmx_fiber_result* out);
/* Host-buffer form: H2D of the transmitted field, the whole link on the device, D2H of the received field. */
int pmx_link_run(pmx_ctx* ctx, const pmx_fiber_desc* desc, const pmx_link_desc* link, pmx_field* io,
                 pmx_fiber_result* out);

/* ---- digital backpropagation: the link run backwards on the receive side ----------------------------------------------
 * An extension (the reference has no DBP).  The field is propagated through a virtual copy of the link with dispersion,
 * nonlinearity and loss negated, spans last first.  With u the field of one realization, for span k = nspan..1:
 *   u <- u / sqrt(gain)                                          (when a gain is given: the amplifier after the span)
 *   for the span's steps h = h_M .. h_1 (reverse of their forward order):
 *     u <- exp(+alpha*h/2) * u
 *     u <- ifft( fft(u) .* exp(+i*betat*h) )                     per column
 *     u <- N(-xi*gam, h) u                                       matrix_nl_step (fiber.m:827-851) with gam -> -xi*gam and
 *                                                                the forward leff(h) = (1 - exp(-alpha*h))/alpha
 *     (scalar path, scalar_field = 1: nl_step (fiber.m:786-803) with gam -> -xi*gam; with the 'x' flag its power is
 *      that of the cross-phase modulation over the sum of |u_j|^2 of all backpropagated columns j, taken after the scale)
 * With xi = 1 and the forward run's own steps (pmx_fiber_result.trace_dz), DBP inverts a noise-free fiber without PMD up
 * to rounding, on the scalar path with the 'x' flag as well.  With pmd = 0, DBP ignores the 'p' flag, the plates and
 * dgdrms; the 'x' flag on a two-polarization field fails with PMX_ERR_XPM_VECTOR as in fiber.
 * PMD-aware DBP (pmd = 1, the fiber's 'p' flag, plates from pmx_dbp_set_plates): the linear operator of a step is the
 * inverse of the forward step's trunk product (matrix_step, fiber.m:904-935): the same trunk pieces in reverse order,
 * the plates last to first, db0, db1 (dgdrms) and betat negated, from and back to the laboratory basis.  The trunk
 * pieces of every step are the forward run's: checkstep (fiber.m:739-758) replayed on the span's forward steps, with
 * zprop accumulated step by step and the last step ending at the fiber length, so that trace_dz reproduces the forward
 * run's partition exactly.  Steps that would index past the last plate fail with PMX_ERR_PLATE_INDEX as fiber would.
 * With xi = 1 and trace_dz, PMD-aware DBP inverts a noise-free 'gps-' link up to rounding.
 * Sizes, FP64 or FP32 (PMX_ERR_UNSUPPORTED otherwise, checked before a context is needed):
 *   two-polarization fields, nfft from 2^12 to 2^24, nfc <= 64: every step is the three HBM passes of a forward step;
 *   two-polarization fields, nfft from 2^6 to 2^11, and the scalar path, nfft from 2^6 to 2^12 (flags 's' and / or 'x'),
 *   nfc <= 8: the whole link in one launch of the single-launch kernel of small fields, one CTA per column and the
 *   columns of a realization in one thread-block cluster (PMX_NO_ONCHIP does not apply: these fields have no other route).
 * The step packages of the whole schedule are built when the plan is created, so pmx_dbp_exec runs every step without
 * reading anything back. */
typedef struct pmx_dbp_desc {
    int32_t nspan;
    int32_t steps_per_span;    /* > 0: uniform steps of length/steps_per_span; 0: the explicit schedule below           */
    const int32_t* span_steps; /* [nspan] steps of each span (explicit schedule), or NULL (uniform steps)               */
    const double* step_len;    /* all spans' steps concatenated, each span in FORWARD order (e.g. trace_dz)             */
    double xi;                 /* fraction of gamma backpropagated; 1 = all                                              */
    double gain;               /* linear amplifier gain after every span, undone first; 0 = none                         */
    int32_t pmd;               /* 1: PMD-aware (the fiber's 'p' flag, plates from pmx_dbp_set_plates); 0: PMD ignored    */
    int32_t reserved;
} pmx_dbp_desc;
/* fiber: the link's fiber (length, alphalin, gam, manakov, fls, dispersion as for pmx_plan_create; batch and precision of
 * the fields the plan will run on; with pmd, nplates, dgdrms or db1 as well).  Validates dbp: PMX_ERR_INVALID for
 * nspan < 1, a non-finite xi, gain < 0, a negative or non-finite step, or a span whose steps do not sum to fiber->length
 * within 1e-9 relative.  The explicit schedule (steps_per_span = 0) needs span_steps and step_len, span_steps[k] >= 1.
 * pmd = 1 needs the 'p' flag and nplates >= 1 (PMX_ERR_INVALID) and a step package table of at most 1 GiB
 * (steps * batch * 2800 bytes, PMX_ERR_INVALID); a schedule that indexes past the last plate fails with
 * PMX_ERR_PLATE_INDEX. */
int pmx_dbp_create(pmx_ctx* ctx, const pmx_fiber_desc* fiber, const pmx_dbp_desc* dbp, pmx_plan** plan);
/* The waveplates of a PMD-aware plan: db0, theta, epsilon [nspan][plate_sets][nplates] in FORWARD span and plate order
 * and sign, as pmx_link_desc takes them; plate_sets is 1 (shared by the batch) or batch.  The library reverses and
 * negates them and rebuilds the step packages on the device; calling it again swaps in a new draw. */
int pmx_dbp_set_plates(pmx_plan* plan, int32_t plate_sets, const double* db0, const double* theta, const double* epsilon);
/* Filtered DBP (Du & Lowery 2010): a Gaussian low-pass with a one-sided -3 dB bandwidth bw, in DFT bins of the plan's grid,
 *   H[k] = exp(-(ln 2 / 2) * (k_s / bw)^2),  k_s the signed bin in [-N/2, N/2)
 * (H(0) = 1, |H(bw)|^2 = 1/2, real, even, a real and positive impulse response), on the intensity of every backward
 * nonlinear step N(-xi*gam, h): each quantity the step computes from |u|^2 is replaced by ifft(fft(q) .* H), the rest of
 * the step is unchanged.  Two polarizations: the phase uses the filtered |ux|^2+|uy|^2 and, CNLSE, the s3 rotation the
 * filtered s3 (P + i*s3 is filtered as one complex signal).  Scalar path: every |u_j|^2 of nl_step is the filtered one;
 * with the 'x' flag the sum over the columns is taken over the filtered powers.  bw = 0: no filter (the plan runs as it
 * did before any call).  Calling it again swaps the bandwidth.  On a single-channel plan (pmx_dbp_channel_create) it applies
 * to the M-sample plan: the bins are equally spaced on both grids, so the same bw is the same frequency.
 * On the three passes a filtered step adds pass C' without its nonlinear epilogue, two pointwise kernels and a filter
 * plan (pmx_filter_create) on a work field of ceil(batch*nfc/2) columns.  PMX_ERR_INVALID for a negative or non-finite
 * bw, for a plan that is not a DBP plan, and for bw > 0 on a plan that has taps (pmx_dbp_set_taps). */
int pmx_dbp_set_filter(pmx_plan* plan, double bw);
/* Enhanced split-step DBP (ESSFM; Secondini, Marsella, Forestieri, ECOC 2014): a real circular FIR on the intensity of
 * every backward nonlinear step N(-xi*gam, h).  taps c[0..2K], ntaps = 2K+1 odd, 1 <= ntaps <= 65 (K <= 32) and at most
 * the number of samples of the plan's grid; c[K] is lag 0.  At time index n of the grid (indices mod N, the sum taken
 * left to right in m)
 *   q~[n] = sum_{m=-K..K} c[m+K] * q[(n - m) mod N],
 * and every quantity the step computes from |u|^2 is replaced by its q~; the rest of the step is unchanged.  Two
 * polarizations: q = P + i*s3 (s3 = 0 for Manakov), as filtered DBP filters it; scalar path: every |u_j|^2, with the
 * 'x' flag the column sum taken over the filtered powers.  This is filtered DBP with H = fft(c placed circularly), but
 * it costs a time-domain FIR, not a transform: on the three passes a step adds pass C' without its nonlinear epilogue,
 * the intensity into a work field of ceil(batch*nfc/2) columns and one kernel that applies the FIR and the nonlinear
 * step.  The same taps serve every step.  ntaps = 0 (taps may then be NULL): no taps, the plan runs as it did before any
 * call.  Calling it again swaps the taps.  On a single-channel plan (pmx_dbp_channel_create) the taps act on the
 * M-sample grid: one tap there spans r = N/M samples of the full field.  PMX_ERR_INVALID for an even ntaps or more than
 * 65, a non-finite tap, more taps than samples, a plan that is not a DBP plan, and taps on a plan that has a filter
 * bandwidth (pmx_dbp_set_filter). */
int pmx_dbp_set_taps(pmx_plan* plan, int32_t ntaps, const double* taps);
/* In place on a resident field; returns when the field is backpropagated.  The field may belong to another context of
 * the same device (as for pmx_fiber_exec).  A PMD-aware plan needs its plates first (PMX_ERR_INVALID).  Destroy the
 * plan with pmx_plan_destroy. */
int pmx_dbp_exec(pmx_plan* plan, pmx_devfield* f);

/* (Perturbation-based nonlinearity compensation, a symbol-rate alternative to DBP: pmx_pb_create below.) */

/* ---- single-channel digital backpropagation: one channel of a 'unique' multiplex at a reduced sample rate ------------
 * A coherent receiver sees its own channel only.  For a field of N = fiber->nfft samples in one column (nfc = 1, every
 * channel in it) and band = {m, r}, M = N/r, the plan runs per realization, in place:
 *   down : u <- ifft(fft(u) .* H), H = 1 on the M bins (k - m) mod N of the signed k in [-M/2, M/2), 0 elsewhere (a filter
 *          plan, pmx_filter_create); v[n] = u[n*r] * exp(+2*pi*i*m*n*r/N), n < M: the channel at baseband, decimated
 *   DBP  : pmx_dbp_exec on v, a plan of pmx_dbp_create at M samples (same schedule, xi, gain, model, precision and
 *          PMD-aware variant) whose dispersion is the channel's own: betat_M[k] = betat_N[(k - m) mod N], db1 likewise
 *   up   : u[n] = r * v[n/r] * exp(-2*pi*i*m*n/N) where r divides n, 0 elsewhere; u <- ifft(fft(u) .* H)
 * Afterwards the field holds the backpropagated channel on its own bins and zeros elsewhere, so a receiver downstream
 * (pmx_field_modulate by m, its filters) is unchanged.  The phase indices are reduced modulo N in integers, as in
 * pmx_field_modulate.  With PMX_DISP_VECTOR the channel's betat / db1 are cropped from fiber's tables; with PMX_DISP_SCALAR
 * the host evaluates them at the channel's signed bins k - m (betat = omega*beta1 + 0.5*omega^2*beta2 + omega^3*b30/6,
 * db1 = dgdrms*omega, omega = 2*pi*symbolrate*FN).  The M-sample plan takes the route pmx_dbp_create gives M samples. */
typedef struct pmx_dbp_band {
    int64_t shift;    /* bins that bring the channel to baseband (as pmx_field_modulate's m; the receiver's ndfn) */
    int32_t decim;    /* r: power of two >= 2; the channel is backpropagated on nfft/r samples                    */
    int32_t reserved;
} pmx_dbp_band;
/* fiber describes the link at N samples.  Checked before a context is needed: PMX_ERR_INVALID for decim not a power of
 * two >= 2 or nfft/decim < 2^6; PMX_ERR_UNSUPPORTED for nfc != 1 and for the scalar path with nfft/decim > 2^12; and
 * everything pmx_dbp_create rejects.  pmx_dbp_set_plates, pmx_dbp_exec (fields of nfft samples, one column) and
 * pmx_plan_destroy take the returned plan; it owns the M-sample DBP plan, the band filter and an M x batch work field. */
int pmx_dbp_channel_create(pmx_ctx* ctx, const pmx_fiber_desc* fiber, const pmx_dbp_desc* dbp, const pmx_dbp_band* band,
                           pmx_plan** plan);

/* ---- perturbation-based nonlinearity compensation (PB-NLC): a first-order triplet correction at the symbol rate -----
 * An extension (the reference has none; Mecozzi, Clausen & Shtaif, IEEE PTL 12(4), 2000; Tao et al., JLT 29(17), 2011).
 * For a resident one-column two-polarization FP64 field of nfft = nsymb*nt samples holding one channel whose dispersion
 * is already compensated (the all-pass step of the link), per realization, in place, with p the pulse table:
 *   project : A^x_k = sum_j p[j] * ux[(k*nt - npulse/2 + j) mod nfft] / sum_j p[j]^2  (A^y likewise), k < nsymb: the
 *             matched filter of the pulse of symbol k, centred at time index k*nt
 *   triplets: Delta^x_k = sum_i C'_i * ( a*A^x_{k+m} A^x_{k+n} conj(A^x_{k+m+n}) + b*A^x_{k+m} A^y_{k+n} conj(A^y_{k+m+n})
 *                                      + c*A^y_{k+m} A^y_{k+n} conj(A^x_{k+m+n}) ),     (x <-> y for Delta^y)
 *             symbol indices mod nsymb, the sum over the list i = (m_i, n_i, C_i) in list order, C'_i = -j*gamma*s^2*C_i
 *   apply   : u[t] -= xi * sum_k Delta_k * p[t - k*nt + npulse/2] over the k whose pulse covers t (k descending)
 * The triplets are formed on s*A and subtracted in the field's units, which is gamma -> gamma*s^2: s brings the received
 * field to launch scale, the field keeps its own.  (a, b, c) = (1, 1, 0) is Manakov (gamma then carries the 8/9), (1, 2/3,
 * 1/3) the CNLSE.  xi = 0 runs no kernel and leaves the field bit for bit as it was.  The sum has a fixed order and no
 * atomics: two executions give the same bits. */
#define PMX_PB_MAX_K 128           /* |m|, |n| <= PMX_PB_MAX_K                                                           */
#define PMX_PB_MAX_COEF 1000000    /* at most this many (m, n, C) entries                                                */
typedef struct pmx_pb_desc {
    int64_t nfft;           /* samples per column: nsymb*nt, a power of two from 2^6 to 2^24                          */
    int32_t nsymb, nt;      /* symbols per block and samples per symbol                                                */
    int32_t batch;          /* realizations of the fields the plan runs on                                             */
    int32_t nfc;            /* columns of those fields: 1 (one channel)                                               */
    int32_t precision;      /* PMX_F64                                                                                 */
    int32_t npulse;         /* pulse samples: even, 2 .. min(16*nt, nfft)                                             */
    const double* pulse;    /* [npulse] real pulse table (electricsource's 2*nt samples: symbol k from (k-1)*nt)        */
    double weights[3];      /* (a, b, c)                                                                                */
    double gamma;           /* [1/W/m] of the triplet sum (Manakov: with the 8/9)                                       */
    double xi;              /* fraction of the perturbation subtracted                                                  */
    double scale;           /* s: received field -> launch scale                                                        */
    int32_t ncoef;          /* entries of the coefficient list, 1 .. PMX_PB_MAX_COEF                                    */
    int32_t reserved;
    const int32_t* m;       /* [ncoef] */
    const int32_t* n;       /* [ncoef] */
    const double* coef;     /* [ncoef][2] C = (re, im), finite                                                         */
} pmx_pb_desc;
typedef struct pmx_pb_plan pmx_pb_plan;
/* Checked before a context is needed: PMX_ERR_UNSUPPORTED for nfc != 1 and for FP32; PMX_ERR_INVALID for nsymb*nt !=
 * nfft, nfft not a power of two from 2^6 to 2^24, batch < 1, a bad pulse (odd or out-of-range npulse, NULL, non-finite,
 * zero energy), non-finite weights, gamma, xi or scale, ncoef out of range, |m| or |n| > PMX_PB_MAX_K, and a non-finite
 * coefficient.  The plan copies the pulse and the list to the device; it holds two [batch][2][nsymb] complex buffers. */
int pmx_pb_create(pmx_ctx* ctx, const pmx_pb_desc* desc, pmx_pb_plan** plan);
/* In place on a resident field of the same device: PMX_ERR_UNSUPPORTED for nfc != 1 or FP32, PMX_ERR_INVALID for a field
 * whose nfft or batch differs from the plan's. */
int pmx_pb_exec(pmx_pb_plan* plan, pmx_devfield* f);
/* The projected symbols A and the perturbation Delta of the last pmx_pb_exec (with xi != 0), each [batch][2][nsymb] complex
 * (re, im interleaved) into host buffers; either may be NULL.  Returns when the copies are done. */
int pmx_pb_symbols(pmx_pb_plan* plan, double* A, double* delta);
void pmx_pb_destroy(pmx_pb_plan* plan);

/* ---- single-channel PB-NLC: one channel of a 'unique' multiplex compensated at a reduced sample rate ------------------
 * As single-channel DBP (pmx_dbp_channel_create) with the stage in place of the backpropagation.  desc describes the
 * channel at M = desc->nfft samples (nt and the pulse at that rate, nsymb unchanged); band = {m, r}; the plan runs on
 * resident one-column FP64 fields of N = M*r samples, per realization, in place:
 *   down : the band filter at N (H = 1 on the M bins (k - m) mod N of the signed k in [-M/2, M/2)), then the channel at
 *          baseband, decimated to M samples (pmx_dbp_channel_create's down)
 *   stage: pmx_pb_exec at M samples (project, triplets, apply)
 *   up   : stuffed back onto the channel's bins, the band filter at N
 * Afterwards the field holds channel m alone on its own bins, exactly as single-channel DBP leaves it.  With xi = 0 only
 * down and up run.  The table is the channel's: its dispersion betat_M[k] = betat_N[(k - m) mod N] less the channel's
 * phase and group delay, which cancel in the triplets; it differs from the centre channel's only through the dispersion
 * slope (polmux_b200/pbnlc.py, channel_setup).
 * Checked before a context is needed: PMX_ERR_INVALID for decim not a power of two >= 2 or M < 2^6; PMX_ERR_UNSUPPORTED
 * for N > 2^24, nfc != 1 and FP32; and everything pmx_pb_create rejects.  pmx_pb_exec (PMX_ERR_INVALID for a field whose
 * nfft is not N or whose batch differs), pmx_pb_symbols ([batch][2][nsymb] of the M-sample stage) and pmx_pb_destroy take
 * the returned plan; it owns the M-sample stage, the band filter and an M x batch work field. */
int pmx_pb_channel_create(pmx_ctx* ctx, const pmx_pb_desc* desc, const pmx_dbp_band* band, pmx_pb_plan** plan);

/* ---- XPM-aware single-channel PB-NLC: the neighbours' symbols compensate the channel's cross-phase modulation ---------
 * Single-channel PB-NLC (pmx_pb_channel_create: the channel of interest, COI, at shift m0) plus the first-order
 * inter-channel triplets of nint interferers, the channels that shift[c] bins bring to baseband (a joint multi-channel
 * receiver has their symbols).  Per realization, in place, with xi != 0:
 *   interferers: for c = 0 .. nint-1 in list order, a copy of the field, the band filter of channel c at N, the channel at
 *                baseband decimated to M (as down), projected as the COI is (the COI's pulse, nt and norm): B_c [2][nsymb]
 *   COI        : down, project (A), the SPM triplets (Delta), as pmx_pb_channel_create
 *   XPM        : Delta^x_k += sum_c sum_i C'_ci * ( w1*A^x_{k+m} B^x_{k+n} conj(B^x_{k+m+n}) + w2*A^x_{k+m} B^y_{k+n}
 *                conj(B^y_{k+m+n}) + w3*A^y_{k+m} B^x_{k+n} conj(B^y_{k+m+n}) + w4*A^y_{k+m} B^y_{k+n} conj(B^x_{k+m+n}) ),
 *                x <-> y for Delta^y, B = B_c, (m, n, C) = entry i of interferer c's table, C' = -j*gamma*s^2*C with the
 *                COI's gamma and s; interferers in list order, each table in list order, no atomics
 *   apply, up  : as pmx_pb_channel_create
 * (w1, w2, w3, w4) = (2, 1, 1, 0) is Manakov (gamma with the 8/9), (2, 2/3, 2/3, 2/3) the CNLSE: the first-order terms of
 * the nonlinear step at the COI's frequency linear in A and in B*conj(B).  Four-wave mixing between two interferers and
 * the triplets whose indices do not satisfy i + j - l = k are left out.  The tables come from polmux_b200/pbnlc.py,
 * xpm_coefficients: the overlap conj(g_0) g_m h_n conj(h_{m+n}) of the COI's pulse g and the interferer's h, each dispersed
 * with its own dispersion in the COI's frame (the walk-off kept).  With xi = 0 only the COI's down and up run, as for
 * pmx_pb_channel_create; no interferer is extracted.
 * Checked before a context is needed: PMX_ERR_INVALID for nint outside 1 .. PMX_PB_XPM_MAX_INT, an interferer shift equal
 * (mod N) to the COI's or to another interferer's, an ncoef below 1 or a total above PMX_PB_MAX_COEF, |m| >
 * PMX_PB_MAX_K, |n| > PMX_PB_XPM_MAX_N, NULL lists and non-finite weights or coefficients; and everything
 * pmx_pb_channel_create refuses (PMX_ERR_UNSUPPORTED for FP32 and nfc != 1).  pmx_pb_exec, pmx_pb_symbols (the COI's A
 * and the total Delta) and pmx_pb_destroy take the plan; pmx_pb_xpm_symbols reads an interferer's B.  Besides the channel
 * plan it owns a band filter per interferer, an N x batch copy of the field and the B buffers. */
#define PMX_PB_XPM_MAX_INT 8       /* interferers per plan                                                               */
#define PMX_PB_XPM_MAX_N 1024      /* |n| <= PMX_PB_XPM_MAX_N in an interferer's table (the walk-off of the link)          */
typedef struct pmx_pb_xpm_desc {
    int32_t nint;           /* interferers, 1 .. PMX_PB_XPM_MAX_INT                                                     */
    int32_t reserved;
    const int64_t* shift;   /* [nint] bins that bring interferer c to baseband (the receiver's ndfn)                    */
    const int32_t* ncoef;   /* [nint] entries of each interferer's table, >= 1, PMX_PB_MAX_COEF in all                  */
    const int32_t* m;       /* [sum ncoef] the tables concatenated in interferer order                                  */
    const int32_t* n;       /* [sum ncoef] */
    const double* coef;     /* [sum ncoef][2] C = (re, im), finite                                                      */
    double weights[4];      /* (w1, w2, w3, w4)                                                                          */
} pmx_pb_xpm_desc;
int pmx_pb_xpm_create(pmx_ctx* ctx, const pmx_pb_desc* desc, const pmx_dbp_band* band, const pmx_pb_xpm_desc* xpm,
                      pmx_pb_plan** plan);
/* The projected symbols B of interferer c (list order) of the last pmx_pb_exec with xi != 0, [batch][2][nsymb] complex
 * (re, im interleaved) into a host buffer.  PMX_ERR_INVALID for a plan without interferers or c out of range. */
int pmx_pb_xpm_symbols(pmx_pb_plan* plan, int32_t c, double* B);

/* ---- the PB-NLC triplet table on the device: what polmux_b200/pbnlc.py, pb_coefficients, computes on the host ----------
 * For a link of nspan spans of `length` [m], loss alphalin [1/m] and dispersion betat (per metre, FFT order, on the grid
 * of nfft = nsymb*nt samples the stage runs on; for single-channel PB-NLC the channel's M samples, pbnlc.channel_setup):
 *   window : W symbols; 0 takes the default rule: the pulse placed on nfft samples and dispersed over nspan*length, the
 *            samples holding all but 1e-9 of its energy (centred, 0.5e-9 cut from either end), plus 2K+8 symbols, rounded
 *            up to a power of two, at most nsymb.  W must divide nsymb; Ws = W*nt samples.  The rule is evaluated on the
 *            device's transform and a sequential host sum where pbnlc.default_window uses numpy's FFT and pairwise sum:
 *            when a 1e-9 energy boundary falls within rounding of a sample, or the count lands within rounding of a
 *            power of two, the two may pick neighbouring windows (window_used tells which was taken).
 *   nodes  : nquad Gauss-Legendre nodes (x, w) per span s: zeta = s*length + length/2*(x+1), weight length/2*w*exp(-alphalin*
 *            length/2*(x+1))
 *   pulses : g_q = ifft(fft(p0) .* exp(-i*bt*zeta_q)) on Ws samples, p0[(j - npulse/2) mod Ws] = pulse[j], bt[k] =
 *            betat[k*nfft/Ws] (the link's bins on the window's grid)
 *   rows   : R[m][n] = sum_q w_q sum_t b(t) conj(b(t - n*nt)) / sum p^2, b(t) = conj(g_q(t)) g_q(t - m*nt), indices mod Ws,
 *            0 <= m, n <= K (R[m][-n] = conj(R[m][n]))
 *   table  : C[m][n] = R[m][n] for m >= 0, conj(R[-m][n]) for m < 0, then C <- (C + C^T)/2 (exactly symmetric); the entries
 *            with |C| >= prune*|C[0][0]| (every entry for prune = 0), m-major with n ascending, -K <= m, n <= K.
 * The outputs hold (2K+1)^2 entries; coef is (re, im) interleaved, so (m, n, coef, ncoef) go into pmx_pb_desc as they are.
 * window_used (may be NULL) receives W.  The lag sums run on the device in a fixed order without atomics: two calls give
 * the same bits.  Checked before a context is needed: PMX_ERR_INVALID for nfft not a power of two from 2^6 to 2^24, nt < 1
 * or not dividing nfft, a bad pulse (as pmx_pb_create), K outside 0..PMX_PB_MAX_K, nquad < 1, nspan < 1, more than 2^20
 * nodes, a non-finite or non-positive length, a negative or non-finite alphalin, a NULL or non-finite betat, a non-finite
 * prune, a window that is negative or does not divide nsymb, and NULL outputs; PMX_ERR_UNSUPPORTED for a window of fewer
 * than 2^6 samples, given or by the default rule. */
typedef struct pmx_pb_table_desc {
    int64_t nfft;           /* samples of the grid the stage runs on                                                    */
    int32_t nt;             /* samples per symbol                                                                       */
    int32_t npulse;         /* pulse samples, as in pmx_pb_desc                                                         */
    const double* betat;    /* [nfft] phase per metre, FFT order                                                         */
    const double* pulse;    /* [npulse] real pulse table, as in pmx_pb_desc                                              */
    int32_t nspan;          /* spans                                                                                    */
    int32_t K;              /* |m|, |n| <= K, 0 .. PMX_PB_MAX_K                                                          */
    double length;          /* span length [m]                                                                          */
    double alphalin;        /* loss [1/m]                                                                               */
    int32_t nquad;          /* Gauss-Legendre nodes per span                                                            */
    int32_t window;         /* symbols of the window; 0: the default rule                                               */
    double prune;           /* keep |C| >= prune*|C[0][0]|                                                              */
} pmx_pb_table_desc;
int pmx_pb_table(pmx_ctx* ctx, const pmx_pb_table_desc* desc, int32_t* m, int32_t* n, double* coef, int32_t* ncoef,
                 int32_t* window_used);

/* ---- create_field('unique'): the WDM multiplex on the device (create_field.m:113-149,180-199) ----------------
 * The reference builds the single field as
 *   FIELDX = ifft( sum_ch fastshift( fft(sigx(:,ch)), -ndfn(ch) ) ),   ndfn = round(deltafn/SYMBOLRATE/minfreq)
 * A circular shift of the spectrum by -ndfn bins is the modulation exp(-2*pi*i*ndfn*n/nfft) in time, so the same
 * field is  sum_ch scale(ch) * sig(mod(n - delay(ch), nfft), ch) * exp(-2*pi*i*ndfn(ch)*n/nfft)  -- one pointwise
 * pass, no transform (the phase index ndfn*n is reduced modulo nfft in integers, the argument of sincospi is exact).
 *   f      : batch 1, nfc 1 field to fill (either precision)
 *   sig    : HOST arrays [nch][nfft] per polarization (PMX_COMPLEX: xr -> X, yr -> Y or NULL; PMX_PLANAR likewise)
 *   ndfn   : [nch] frequency offsets in bins (create_field.m:183)
 *   scale  : [nch] amplitude factors (options.power = 'average', :113-124) or NULL (ones)
 *   delayx, delayy : [nch] integer sample delays per polarization (options.delay, :127-146) or NULL (zeros) */
int pmx_field_mux(pmx_devfield* f, const pmx_field* sig, int32_t nch, const int64_t* ndfn, const double* scale,
                  const int64_t* delayx, const int64_t* delayy);

/* ---- integer error counting (ber_estimate.m:118) --------------------------------
 * counts[b] = #{ i : pat_hat[b][i] != pat[i] } over n symbols-bits, on the device. */
int pmx_count_errors(pmx_ctx* ctx, const uint8_t* pat_hat_dev, const uint8_t* pat_dev, int64_t n,
                     int32_t batch, int64_t* counts_dev);

/* ---- minimal coherent decision + error count for Monte-Carlo runs -------------------------
 * Not the reference's dsp4cohdec.m (its blind DSP core is pmx_dsp_count below): a data-aided stand-in used only to turn a propagated (and
 * linearly equalised, see polmux_b200/mc.py) PDM-QPSK field into the INTEGER error count that
 * ber_estimate.m:118 feeds its recursion with.  Per realization and polarization:
 *   r_k = field[k*nt]                                 symbol-centre sample (samp2pat.m:60-67)
 *   phi = angle(sum_k r_k conj(s_k))                  data-aided carrier phase
 *   bits = (Re(r_k e^{-i phi}) > 0, Im(...) > 0)      Gray QPSK decision (pat_decoder.m:68-82)
 *   counts[b] = #bits != transmitted bits, over both polarizations
 * sym: HOST array [2][nsymb] of transmitted symbol indices 0..3 (bit0 -> sign Re, bit1 -> sign Im).
 * counts_dev: DEVICE pointer to [batch] int64 (e.g. the NCCL send buffer), overwritten. */
int pmx_qpsk_count(pmx_ctx* ctx, pmx_devfield* f, const uint8_t* sym, int32_t nsymb, int32_t nt,
                   int64_t* counts_dev);

/* ---- blind DSP core of the coherent receiver + error count ------------------------------------------------------
 * What dsp4cohdec.m does between its decimator and its outputs, for a dual-polarization QPSK field already compensated
 * for chromatic dispersion, on one complex sample per symbol (the sample at time index k*nt of symbol k) normalised to
 * unit mean power:
 *   easipolardemux  (optional, before or instead of the CMA) EASI source separation with one 2x2 tap
 *   cmapolardemux   constant-modulus 2x2 FIR polarization demultiplexer: cmaadaptivefilter.m:33-55 (C twin
 *                   cmaadaptivefilter.c:57-91) passed over the block until the taps move by less than 5e-5
 *                   (dsp4cohdec.m:353-427), taps initialised to the rotation by phizero
 *   carrier         frequency from (s.*conj(shift(s))).^4 averaged over 2*freqavg+1 symbols, cumulated and cleaned to
 *                   the block's circularity; phase by Viterbi & Viterbi with 2*phasavg+1 symbols (vitvit,
 *                   dsp4cohdec.m:241-283, 320-345)
 *   decision        samp2pat 'coherent' (samp2pat.m:60-67), differential decoding pat_decoder 'dqpsk'
 *                   (pat_decoder.m:68-82), X/Y swap test and error count (ex20_coherent_polmux.m:168-176,
 *                   ber_estimate.m:118)
 * Neither the waveplates nor the transmitted symbols enter the processing; ref_patmat is only counted against.
 * The front-end of receiver_cohmix.m is pmx_filter_create / pmx_field_modulate / pmx_cohmix_exec below.  Not built:
 * mygeteyeinfo's pattern-correlation timing search (the 'theory' delay of dsp4cohdec.m:490-503 enters as sample_shift) and
 * a pinned decimator (dsp4cohdec.m:176-184) -- `decimate` is a Signal Processing Toolbox function that is not in the
 * reference tree; the currents are sampled at the symbol centres, optionally behind an anti-alias FIR the caller designs
 * (decim_taps).  p.applyadc is
 * pmx_field_quantize on the currents, p.applynlr the desc's nlr_alpha, p.applydcf (one sample per symbol) its dcf_h. */
typedef struct pmx_dsp_desc {
    int32_t nsymb, nt;        /* symbols per block, samples per symbol                                   */
    int32_t apply_cma;        /* p.applypol with p.polmethod = 'cma'                                      */
    int32_t taps;             /* p.cmaparams.taps (odd, <= 15)                                            */
    double mu;                /* p.cmaparams.mu                                                           */
    double R[2];              /* p.cmaparams.R                                                            */
    double phizero;           /* p.cmaparams.phizero                                                      */
    int32_t max_passes;       /* 0: the reference's bound 50*ceil(1/(L*mu)) - 1                           */
    int32_t modorder;         /* p.modorder (2 = QPSK)                                                    */
    int32_t freqavg, phasavg; /* p.freqavg, p.phasavg                                                     */
    int32_t poworder;         /* p.poworder                                                               */
    int32_t sample_shift;     /* symbol k is sampled at time index k*nt + sample_shift (circular): 0 for a field; for the
                               * receiver's currents round(delay*NT), the shift dsp4cohdec.m:167-169 undoes            */
    double peak;              /* samples are divided by peak = 4*sqrt(GSTATE.POWER(ich)) (dsp4cohdec.m:226-227);
                               * 0: normalise the block to unit mean power instead                                     */
    /* p.polmethod = 'easi' (apply_easi = 1, apply_cma = 0) or 'combo' (both: EASI first, dsp4cohdec.m:236-241):
     * easipolardemux / easiadaptivefilter (dsp4cohdec.m:428-482, easiadaptivefilter.m:28-61), one 2x2 tap */
    int32_t apply_easi;
    int32_t easi_max_passes;  /* 0: the reference's bound 20*ceil(1/(L*mu)) - 1                                        */
    double easi_mu;           /* p.easiparams.mu                                                                       */
    double easi_phizero;      /* p.easiparams.phizero                                                                  */
    int32_t* easi_passes;     /* HOST [batch] output: passes the EASI stage ran; may be NULL                           */
    double nlr_alpha;         /* p.applynlr ? p.nlralpha : 0 -- NLRotation (dsp4cohdec.m:219-221,308-315), applied to the
                               * sampled signals before the division by peak                                            */
    const double* dcf_h;      /* p.applydcf: HOST [nsymb] complex Hfilt of DispCompFilter (dsp4cohdec.m:289-297) applied to the
                               * sampled signals, ifft(fft(Signals).*Hfilt) (:198-210), before the rotation above; or NULL;
                               * nsymb must then be a power of two >= 64                                                  */
    /* The decimator's anti-alias FIR in front of the sampling (dsp4cohdec.m:176-184: decimate(I, r, 16, 'fir')).  `decimate`
     * and `fir1` belong to the Signal Processing Toolbox, not to the reference tree: the caller designs the taps (the host
     * mirror restates the toolbox's PUBLISHED algorithm -- Hamming-windowed sinc, unit DC gain, group delay compensated;
     * parity unpinned) and the sampler evaluates filter(b,1,I) at the sampling instants only, circularly. */
    int32_t decim_ntaps;      /* 0 / 1: plain sampling; else odd, <= 65                                                  */
    int32_t reserved2;
    const double* decim_taps; /* HOST [decim_ntaps]                                                                      */
} pmx_dsp_desc;
/* ref_patmat: HOST [nsymb][4] bytes, the differentially decoded transmitted pattern [x1 x2 y1 y2] (pat_decoder of the
 * transmitted bits); counts_dev: DEVICE [batch] int64 (e.g. the NCCL send buffer); passes_host (may be NULL): [batch]
 * passes the demultiplexer ran. */
int pmx_dsp_count(pmx_ctx* ctx, pmx_devfield* f, const pmx_dsp_desc* dsp, const uint8_t* ref_patmat, int64_t* counts_dev,
                  int32_t* passes_host);
/* The same processing up to the outputs of dsp4cohdec itself (dsp4cohdec.m:284-287): Phases = angle(Signals .* Carrier)
 * and Amplitudes = abs(Signals) per symbol, HOST [batch][2][nsymb] each (amps may be NULL) -- what samp2pat / pat_decoder
 * of a script take next (ex20_coherent_polmux.m:151-161). */
int pmx_dsp_phases(pmx_ctx* ctx, pmx_devfield* f, const pmx_dsp_desc* dsp, double* phases, double* amps, int32_t* passes_host);

/* ---- Monte-Carlo over independent realizations on the GPUs of one node (BASELINE config C5) ------------------------
 * The `while cond` loop of ex20_coherent_polmux.m:131-181 with its realizations sharded over several GPUs from ONE
 * process: contiguous realization groups per GPU (rank g owns [g*nreal/ndev, (g+1)*nreal/ndev)), one host thread and
 * one context per GPU, every realization = nspan x [fiber ; ampliflat] on the resident batch, optionally the ideal
 * linear equaliser (GVD and PMD of every span undone with the known plates, cf. inverse_pmd.m:100-124), then the
 * error counter (pmx_qpsk_count) writing into the rank's slice of a zero-initialised [nreal] int64 vector and ONE
 * ncclAllReduce(sum) over NVLink.  NCCL is bound at run time (libnccl.so.2); with a single GPU it is optional.
 * The caller replays ber_estimate's recursion (ber_estimate.m:121-127) over counts[] in realization order. */
/* The reference's receive chain behind the link of a Monte-Carlo job (ex20_coherent_polmux.m:151-176): receiver_cohmix's
 * front-end, the sampler and the DSP core, per resident batch.  hf_opt already carries whatever all-pass compensation the
 * receiver applies (x.dpost, receiver_cohmix.m:139-166, or p.applydcf), unless dbp is set.  Single-column ('unique') FP64 fields.  The chain of
 * a group runs on a context (stream) and host thread of its own beside the propagation of the next group. */
typedef struct pmx_mc_receiver {
    const double* hf_opt;      /* [nfft] complex: post fiber .* optical filter                              */
    const double* hf_el;       /* [nfft] complex: low-pass filter as myfilter returns it                    */
    double lo_ecw, lo_detune;  /* local oscillator (pmx_cohmix_exec)                                        */
    const double* lo_phase;    /* [nfft] or NULL                                                            */
    int32_t balanced;
    int32_t reserved;
    pmx_dsp_desc dsp;          /* sampler (sample_shift, peak), demultiplexer, carrier recovery             */
    const uint8_t* ref_patmat; /* [nsymb][4] decoded transmitted pattern (pmx_dsp_count)                    */
    const pmx_dbp_desc* dbp;   /* NULL: hf_opt carries the all-pass compensation; else digital backpropagation of the  */
                               /* link (pmx_dbp_exec) on every received batch before the front-end, hf_opt then     */
                               /* carrying the optical filter only                                                  */
} pmx_mc_receiver;

typedef struct pmx_mc_desc {
    int32_t ndev;                /* GPUs of this node to shard over                                          */
    const int32_t* device_ids;   /* [ndev]                                                                   */
    int32_t nreal;               /* realizations in total                                                     */
    int32_t batch;               /* realizations resident per GPU at a time                                   */
    int32_t nspan;
    int32_t equalize;            /* 1: ideal linear equaliser before the decision                             */
    const double* db0;           /* [nspan][nreal][nplates] plate draws (fiber.m:274-276), host; NULL without 'p' */
    const double* theta;
    const double* epsilon;
    double gain;                 /* linear power gain of the amplifier after every span; 0: none              */
    const double* sigma;         /* [nfc] ASE sigma per column or NULL                                        */
    uint64_t ase_seed;           /* span k uses the seed ((ase_seed & 0xffffff) << 40) + (k << 32), keyed by the     */
                                 /* global realization index (pmx_ampliflat_exec_at)                          */
    const uint8_t* sym;          /* [2][nsymb] transmitted QPSK symbol indices (pmx_qpsk_count)               */
    int32_t nsymb, nt;
    const pmx_mc_receiver* rx;   /* NULL: the data-aided counter above; else the reference's receive chain     */
    const pmx_dbp_desc* dbp;     /* without rx: NULL, or PMD-aware DBP (pmd = 1) with every group's own plates in place */
                                 /* of the equaliser ahead of the data-aided counter; pmd = 0 is PMX_ERR_INVALID       */
                                 /* there.  With rx, rx->dbp with pmd = 1 gets the group's plates the same way.       */
} pmx_mc_desc;
/* fiber: the span's fiber (batch / plate_sets / plates are taken from mc); tx: HOST Tx field of one realization;
 * counts: [nreal] bit errors per realization; sa_steps (may be NULL): sum over all realizations of nfft*nfc*ncycle;
 * errbuf (may be NULL): message of the first failure. */
int pmx_mc_run(const pmx_fiber_desc* fiber, const pmx_mc_desc* mc, const pmx_field* tx, int64_t* counts,
               int64_t* sa_steps, char* errbuf, int32_t errlen);
int pmx_mc_nccl_available(void);

/* ---- building blocks of the local-error adaptive step (scalar path only) -------------------------
 * scalar_a_ssfm / adaptssfm, fiber.m:639-679,938-1010: one symmetric step against two half steps, local error
 * max|u - uh|/dz, Richardson extrapolation 4/3*uh - 1/3*u, step proposal safety*sqrt(err/est_err)*dz.  The loop itself
 * is host logic (polmux_b200/fiber.py, as it is interpreter code in the reference); the field never leaves the
 * device.  FP64 fields, X polarization (the scalar path has no Y).
 *   pmx_scalar_nl_exec : u_k <- u_k .* fastexp(-gam_k .* pow * leff) * atten   nl_step (:786-803, pow with the
 *                        SPM / XPM rules of :792-799) followed by u*exp(-halfalpha*dz) (:971,976,...)
 *   pmx_plan_set_length: a plan of a linear flag ('g---': one step) then applies lin_step(betat*length, u) (:762-773)
 *   pmx_field_max_power: umax[b*nfc+c] = max_n |ux|^2 + |uy|^2 (nextstep's Umax, :693-698)
 *   pmx_field_maxdiff2 : *out = max over samples and columns of |a - b|^2 of the X polarization (:996)
 *   pmx_field_lincomb  : dst <- ca*a - cb*b (X and Y), products rounded separately as the interpreter does (:1003) */
int pmx_scalar_nl_exec(pmx_ctx* ctx, pmx_devfield* f, const double* gam, double leff, double atten, int32_t spm,
                       int32_t xpm);
/* The whole adaptive dispatch on host buffers, for callers that are not the Python mirror (the MEX gateway):
 *   first_only = 0: scalar_a_ssfm (fiber.m:639-679) -- every step from the local error (x.ltol);
 *   first_only = 1: scalar_ssfm with x.dphiadapt (fiber.m:588-611) -- first step from the local error, dphimax
 *                   recalibrated from it (:607), the rest of the fiber by the device loop.
 * desc: scalar_field = 1, batch 1, FP64; io: X planes only (Y absent); out: firstdz[1], ncycle[1]. */
int pmx_scalar_adaptive_run(pmx_ctx* ctx, const pmx_fiber_desc* desc, double ltol, double safety, int32_t first_only,
                            pmx_field* io, pmx_fiber_result* out);
int pmx_plan_set_length(pmx_plan* plan, double length);
int pmx_field_max_power(pmx_ctx* ctx, pmx_devfield* f, double* umax);
/* pavg[b*nfc+c] = mean_n |ux|^2 + |uy|^2: the average power avg_power.m:63-76 returns for a separate-channel field
 * (ampliflat's 'fixpower' gain, ampliflat.m:65-72). */
int pmx_field_mean_power(pmx_ctx* ctx, pmx_devfield* f, double* pavg);
/* the two polarizations apart: px, py [batch*nfc] (x.avgebx / x.avgeby of receiver_cohmix.m:174-175,233-234) */
int pmx_field_mean_power_xy(pmx_ctx* ctx, pmx_devfield* f, double* px, double* py);
int pmx_field_maxdiff2(pmx_ctx* ctx, pmx_devfield* a, pmx_devfield* b, double* out);
int pmx_field_lincomb(pmx_ctx* ctx, pmx_devfield* dst, double ca, pmx_devfield* a, double cb, pmx_devfield* b);

/* ---- linear filters: ifft(fft(u) .* H) -----------------------------------------------------------------------------
 * The building block of the toolbox's filter devices and receivers (receiver_cohmix.m:169,180,231,302: optical band-pass
 * and electrical low-pass filters given by myfilter.m as a vector over GSTATE.FN).  The plan runs the same three passes
 * as a linear fiber step with H(k) as the per-bin factor; pmx_fiber_exec(plan, f, NULL) filters both polarizations of
 * every column and realization of f in place.  H: [hcols][nfft] complex128 (re, im interleaved), in the order of
 * GSTATE.FN (FFT order); hcols = 1 (one filter for every column) or nfc.  Destroy with pmx_plan_destroy. */
int pmx_filter_create(pmx_ctx* ctx, int64_t nfft, int32_t nfc, int32_t batch, int32_t precision, const double* H,
                      int32_t hcols, pmx_plan** out);

/* ---- front-end of the coherent receiver: receiver_cohmix.m -----------------------------------------------------------
 *   x.sigx = GSTATE.FIELDX(:,nch) (a copy, :133-137)            pmx_field_copy_cols
 *   x.sigx = fft(x.sigx); x.sigx = x.sigx(nind)  (:171-172)     pmx_field_modulate (the shift by ndfn bins, in time)
 *   x.sigx = x.sigx .* Hf; ifft  (:169,176,240-241)             filter plan with Hf = fastexp(-betat_post) .* myfilter(...)
 *   LO, four mixer outputs, photodiodes  (:178-290)             pmx_cohmix_exec
 *   Iric = real(ifft(fft(Iric) .* Hf))  (:293-302)              filter plan with the Hermitian part of the low-pass Hf
 * pmx_field_copy_cols: count realization-columns of src, starting at src_bc, to dst starting at dst_bc (device to device).
 * pmx_field_modulate : u(n) <- u(n)*exp(+i*2*pi*m*n/nfft), both polarizations of every column.
 * pmx_cohmix_exec    : in place, per polarization s -> I_a + i*I_b with (I_a, I_b) = (I1 - I2, I3 - I4) (balanced) or
 *                      (I1, I3); Elo(n) = lo_ecw * fastexp(lo_detune*(n+1) + lo_phase[n]); lo_phase: HOST [nfft] or NULL. */
int pmx_field_copy_cols(pmx_devfield* dst, int32_t dst_bc, const pmx_devfield* src, int32_t src_bc, int32_t count);
int pmx_field_modulate(pmx_ctx* ctx, pmx_devfield* f, int64_t m);
int pmx_cohmix_exec(pmx_ctx* ctx, pmx_devfield* f, double lo_ecw, double lo_detune, const double* lo_phase, int32_t balanced);
/* p.applyadc (dsp4cohdec.m:157-162) on the currents a front-end left in f: per realization M = max |I| over its samples and
 * currents, I <- round((I + M)/2/M*2^bits)*2*M/2^bits - M.  FP64 fields. */
int pmx_field_quantize(pmx_ctx* ctx, pmx_devfield* f, int32_t bits);
/* The same on host buffers in one call (what the MEX gateway binds for matlab/receiver_cohmix.m): sig = the channel's
 * column(s) x.sigx / x.sigy in time, one realization; iric: [nfft][2 or 4] column-major, as receiver_cohmix returns it;
 * avgeb (may be NULL): [2] = sum |X(band)|^2 / Nfft^2 of the two polarizations (x.avgebx, x.avgeby before the division by
 * GSTATE.POWER).  hf_el is myfilter(x.eftype, ...) as the reference builds it (its Hermitian part is taken inside). */
typedef struct pmx_cohmix_desc {
    int64_t nfft;
    int32_t precision;       /* pmx_precision of the device arithmetic */
    int32_t two_pol;         /* ~isempty(GSTATE.FIELDY) */
    int32_t balanced;        /* ~strcmp(x.pdtype,'normal') (:264-268) */
    int32_t reserved;
    int64_t ndfn;            /* spectrum shift in bins (:87-89); 0 for separate channels */
    int64_t ndfnl, ndfnr;    /* the channel's band for avgeb (:90-110) */
    const double* hf_opt;    /* [nfft] complex: fastexp(-betat) .* myfilter(x.oftype,...) (:166-169) */
    const double* hf_el;     /* [nfft] complex: myfilter(x.eftype,...) (:293) */
    double lo_ecw;           /* LO_Ecw (:215-219) */
    double lo_detune;        /* 2*pi*kdet/Nfft (:187-200) */
    const double* lo_phase;  /* [nfft] LO_PhaseNoise or NULL (:201-214) */
} pmx_cohmix_desc;
int pmx_cohmix_run(pmx_ctx* ctx, const pmx_cohmix_desc* d, const pmx_field* sig, double* iric, double* avgeb);

/* ---- inverse_pmd.m: the PMD matrix of a chain of fibers, and a constant Jones matrix on the field -------------------
 * One fiber of the chain as fiber() returns it in its brf struct (inverse_pmd.m:9-17). */
typedef struct pmx_brf {
    int32_t ntrunk;        /* length(brf.theta) */
    int32_t reserved;
    double lcorr;          /* trunk length [m] */
    const double* db0;     /* [ntrunk] */
    const double* theta;   /* [ntrunk] */
    const double* epsilon; /* [ntrunk] */
    const double* betat;   /* [nfft]  scalar phase per metre (brf.betat) */
    const double* db1;     /* [nfft]  differential phase per trunk (brf.db1) */
} pmx_brf;
/* U(:,:,n) and Uinv(:,:,n) of inverse_pmd.m:73-131 evaluated on the device, one thread per frequency, in the
 * interpreter's order of operations (update_U keeps the first row and completes it to [a b; -b* a*], :152-161).
 * mat: options.mat as 8 doubles (m11 re, im, m12, m21, m22), or NULL; gvd = 0 is options.gvd = 'no'.
 * U, Uinv: [nfft][2][2] complex128 in the interpreter's column-major order (element (i,j,n) at i + 2j + 4n); either
 * may be NULL. */
int pmx_pmd_matrix(pmx_ctx* ctx, int64_t nfft, int32_t nfiber, const pmx_brf* brf, const double* mat, int32_t gvd,
                   double* U, double* Uinv);
/* [ux; uy] <- J [ux; uy] for every sample of every column; j = 8 doubles, row-major (j11 re, im, j12, j21, j22).  The
 * change of reference system options.mat of inverse_pmd.m:87-89 commutes with the transforms, so it is applied in time. */
int pmx_field_jones(pmx_ctx* ctx, pmx_devfield* f, const double* j);
/* inverse_pmd(brf, options) on host buffers in one call (the gateway's 'invpmd', matlab/inverse_pmd.m): the chain's inverse as
 * reversed / negated single-step runs of the SSFM passes on the device (inverse_pmd.m:91-141), options.mat as a constant
 * Jones matrix (:87-89), gvd = 0 for options.gvd = 'no', apply = 0 to leave the field alone (:135); U / Uinv as
 * pmx_pmd_matrix returns them, or NULL.  io: one realization, one column, both polarizations. */
int pmx_inverse_pmd_run(pmx_ctx* ctx, int64_t nfft, int32_t nfiber, const pmx_brf* brf, const double* mat, int32_t gvd,
                        int32_t apply, pmx_field* io, double* U, double* Uinv);

#ifdef __cplusplus
}
#endif
#endif /* POLMUX_SSFM_H */
