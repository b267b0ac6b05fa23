// Shared device-side types of the SSFM kernels (sm_100a).
//
// Field layout in HBM: one "Sa" = (xr, xi, yr, yi) = 4 reals (32 B in FP64, 16 B in FP32), stored as
// two consecutive complex numbers (X then Y).  field[((b*nfc + c)*N + n)*2 + pol].
// Four-step index split: time n = n1*N2 + n2, frequency k = k1 + N1*k2.
//
// Precision: the kernel translation units are compiled twice, without and with -DPMX_F32.  `real`/`cpx` are
// the field's arithmetic type in that translation unit; step control, plate constants and every phase
// ARGUMENT stay in double in both builds (phases reach 1e3..1e5 rad: their reduction needs the 53 bits).
// The structs shared with the host (StepCtl, StepPkg, PlateConst, FiberConst, PassParams) are the same in
// both builds; the kernels carry the real type as a template parameter so that the two builds do not collide.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#ifdef PMX_F32
typedef float real;
typedef float2 cpx;
#define PMX_PRECISION 1
__host__ __device__ __forceinline__ cpx mkc(real a, real b) { return make_float2(a, b); }
#define R_MUL(a, b) __fmul_rn(a, b)
#define R_ADD(a, b) __fadd_rn(a, b)
#else
typedef double real;
typedef double2 cpx;
#define PMX_PRECISION 0
__host__ __device__ __forceinline__ cpx mkc(real a, real b) { return make_double2(a, b); }
#define R_MUL(a, b) __dmul_rn(a, b)
#define R_ADD(a, b) __dadd_rn(a, b)
#endif
#define PMX_SA_BYTES (4 * (int)sizeof(real))

#define PMX_MAX_NFC 64

// Debug builds (make EXTRA=-DPMX_DEBUG, `make debug`): index checks in the tile walks and the bin arithmetic; the
// compute-sanitizer is not available on the pool, these traps stand in for its bounds checks.
#ifdef PMX_DEBUG
#include <cstdio>
#define PMX_ASSERT(cond)                                                                                  \
    do {                                                                                                  \
        if (!(cond)) {                                                                                    \
            printf("PMX_ASSERT failed: %s (%s:%d) block %d thread %d\n", #cond, __FILE__, __LINE__, (int)blockIdx.x, \
                   (int)threadIdx.x);                                                                     \
            __trap();                                                                                     \
        }                                                                                                 \
    } while (0)
#else
#define PMX_ASSERT(cond) ((void)0)
#endif

enum { PMX_ST_RUN = 0, PMX_ST_LAST = 1, PMX_ST_DONE = 2, PMX_ST_ERROR = 3 };
// Basis bookkeeping of the PMD product.  The reference goes laboratory -> PSP basis of the first trunk at the
// start of every linear step and back at its end (fiber.m:920-921,931-932).  When the nonlinear step is a
// scalar phase (Manakov) or absent, those constant unitary matrices commute with everything between two
// linear steps (phase rotation, FFTs, attenuation; |ux|^2+|uy|^2 is invariant), so the field can stay in
// the PSP basis of the trunk it is in: R(last)*...*R(first)^H of consecutive steps collapses to nothing
// (same trunk) or to the boundary matrix of the plate just left.
enum { PMX_BM_ENTRY_R = 1, PMX_BM_ENTRY_C = 2, PMX_BM_EXIT_R = 4,
       // pass A: every nonlinear phase of this step is below 2^-6 rad (gam*leff*max|u|^2 bounds it): short Taylor kernels
       PMX_BM_NL_SMALL = 256 };

// Per-realization propagation state + the schedule of the step about to run.
// Written by the last CTA of pass C (or by the init kernel), read by passes A/B/C.
struct __align__(16) StepCtl {
    // running state of matrix_ssfm (fiber.m:506-517)
    double zprop;      // end coordinate of the step about to be taken (SURVEY A.4)
    double dz;         // dz returned by the last nextstep
    double dz_miss;    // fiber.m:508
    double firstdz;    // fiber.m:516
    int ntot;          // fiber.m:515
    int ncycle;        // fiber.m:506
    int state;         // PMX_ST_*
    int err;           // pmx_status when state == PMX_ST_ERROR
    // schedule of the current step
    double dz_cur;     // dz (or last_step) used by NL, linear and attenuation
    double leff;       // fiber.m:827-831
    double scale;      // exp(-alpha/2*dz_cur) / N   (attenuation fused with the ifft 1/N)
    double dzb_first;  // dzb(1)
    double dzb_last;   // dzb(ntrunk)
    int ntrunk;        // fiber.m:743,749
    int nmem;          // fiber.m:742,748
    int n_first;       // 0-based plate index of trunk k=1:  ntot + 1 - nmem - 1
    int bmode;         // PMX_BM_* : which constant basis changes pass B applies around the trunk product
    // reduction scratch for nextstep
    unsigned long long umax_bits[PMX_MAX_NFC];  // max over n of |ux|^2+|uy|^2, per column
    unsigned int pad_ticket;
    unsigned int pad1;
};

// Per-plate constants, precomputed on the host in IEEE double.
struct __align__(16) PlateConst {
    // matR = Rtheta*Repsilon (fiber.m:910-912), row-major complex
    double r11r, r11i, r12r, r12i, r21r, r21i, r22r, r22i;
    // C = matR(next)^H * matR(this): change of PSP basis at the boundary to the next plate
    double c11r, c11i, c12r, c12i, c21r, c21i, c22r, c22i;
    double db0;       // brf.db0(n)
    double h0r, h0i;  // exp(-i*db0/2): interior-plate phase factor
    // the same boundary matrix factored as C = diag(p, conj(p)) * [ka kb; -conj(kb) ka] with ka = |c11| real: the
    // product with a vector costs 12 instead of 16 FMAs per bin, and the diagonal phase p joins the next trunk's
    // (bin-independent) base phasor
    double ka, kbr, kbi, pr, pi;
};

// What the pass kernels need to know about the step in flight, per realization: written by the step-control
// kernel (pmx_k_ctl) once per step, fetched by every tile with ONE bulk copy (cp.async.bulk, same mbarrier as the
// tile itself), so no pass thread ever waits on a dependent global load of step state.
#define PMX_PKG_PLATES 12
struct __align__(16) StepPkg {
    double dz_cur, leff, scale, dzb_first, dzb_last, gpf_r, gpf_i, gpl_r, gpl_i, db0_last;
    int ntrunk, n_first, bmode, state;  // -- 96 bytes: what passes A and C copy
    double gd3_r, gd3_i;
    double gpf2[2], gpf4[2], gpl2[2], gpl4[2];   // -- 176-byte header (PMX_PKG_HEAD)
    double E[8];   // pass B entry matrix (row-major re,im): R(first)^H, or the boundary matrix of the plate before
    double X[8];   // pass B exit matrix R(last)
    PlateConst plates[PMX_PKG_PLATES];  // the first trunks of the step (more are read from the plate array)
};
#define PMX_PKG_HEAD 176
#define PMX_PKG_HEAD_AC 96

// Constants of one fiber() call (kernel parameter, by value).
struct FiberConst {
    double Lf, alphalin, halfalpha, dzmax, phimax, lcorr, invN;
    double gam[PMX_MAX_NFC];  // after the Manakov 8/9 (fiber.m:500)
    int nplates, nfc, spm, manakov, pmd, gvd_any, plate_sets, trace_cap;
    int keep_basis;        // pmd && (manakov || !spm), see PMX_BM_*
    int scalar_field;      // scalar_ssfm dispatch (fiber.m:372-380): Y absent; nl_step's operation order
    int xpm;               // scalar path with the 'x' flag: cross-phase modulation between the columns (:793-799)
    // scalar dispersion mode (fiber.m:350-362 regenerated per bin instead of read from HBM):
    //   omega = w0*fn, fn = kk/NSYMB (kk = signed FFT bin), betat = omega*beta1 + 0.5*omega^2*beta2
    //   + omega^3*b30/6, db1 = dgdrms*omega
    int disp_scalar;
    unsigned nfc_magic;   // ceil(2^32/nfc): bc / nfc = umulhi(bc, nfc_magic) for nfc > 1
    double w0, inv_nsymb, b30_6, dgdrms, domega;  // domega = w0*NT/8: spacing of a thread's bins
    double g1r, g1i;                              // exp(-i*0.5*dgdrms*domega)
    double g2r, g2i, g4r, g4i;                    // its square and fourth power
    double beta1[PMX_MAX_NFC], beta2[PMX_MAX_NFC];
    double z_start, dz_first;  // loop resumed at zprop = z_start + dz_first (pmx_fiber_desc); 0/0 = fresh fiber
};

struct PassParams {
    void* field;            // cpx [batch*nfc][N][2] in the precision of the launch
    StepCtl* ctl;           // [batch]
    StepCtl* ctl_out;       // fused step control (pass A, a batch of one): the control block the step writes; ctl is read
    int first;              // fused step control: this launch runs the first step of the fiber
    const void* tw_stage;   // cpx: in-CTA FFT stage twiddles for this L
    const double* betat_p;  // [nfc][N1][N2] permuted so that bin k1 + N1*k2 sits at k1*N2 + k2
    const double* db1_p;    // same layout
    const double2* hfilt;   // linear-filter plans (pmx_filter_create): the per-bin factor H, same layout; else null
    long long hfilt_stride; // N when every column has its own H, 0 when they share one
    const PlateConst* plates;  // [plate_sets][nplates]
    StepPkg* pkg;           // [batch]
    const void* tw4;        // cpx: four-step twiddle rows for this pass: [rows][PmxTw4<L>::PER], see pmx_kernels.cuh
    double* trace_dz;       // [batch][trace_cap] or null
    int* trace_ntrunk;
    int N1, N2, log2N1, log2N2;
    int batch;
    int bc0;                // first realization-column of this launch inside the field (tensor-map coordinate offset)
    int pdl;                // launched with programmatic stream serialization: the prologue overlaps the tail of the
                            // previous kernel of the stream, griddepcontrol.wait orders the dependent accesses
    int reverse;            // walk the tile list backwards (alternates from pass to pass: the tiles the previous
                            // pass wrote last are still in L2 when this pass reads them first)
    long long* dbg;         // optional per-CTA phase cycle counters (PMX_TIMING builds only)
};

// The fixed schedule of a digital-backpropagation plan for the single-launch kernel of small fields (pmx_k_onchip with
// DBP = true, its third argument): step s runs package pkg[idx[s]][b]; a PMD-aware plan reads the plates of span span[s],
// at plates + span[s] * plate_stride.
struct DbpSteps {
    const StepPkg* pkg;     // [npkg][batch]
    const int* idx;         // [nstep]
    const int* span;        // [nstep], or null without PMD
    int nstep;
    int pkg_bytes;          // bytes of a package the steps read: the header alone without PMD, all of it with
    long long plate_stride; // PlateConst per span: plate_sets * nplates
};
// Filtered DBP on the single-launch kernel (pmx_dbp_set_filter): the step table and the Gaussian response over the
// transform length, hn[k] = H(k)/N at the unsigned bin k.  Its own type, so that its instances are new ones.
struct DbpFiltSteps {
    DbpSteps s;
    const double* hn;       // [L]
};
// Enhanced split-step DBP (pmx_dbp_set_taps): the real FIR c[0..2k] on the intensity of every nonlinear step, c[k] at
// lag 0.  A kernel parameter, by value: every thread reads the same tap at the same time.
#define PMX_MAX_TAPS 65
struct DbpTaps {
    int k;                  // half-length: 2k+1 taps, 0 <= k <= 32
    double c[PMX_MAX_TAPS];
};
struct DbpTapSteps {
    DbpSteps s;
    DbpTaps taps;
};
__host__ __device__ __forceinline__ DbpSteps pmx_dbp_steps(const DbpSteps& s) { return s; }
__host__ __device__ __forceinline__ DbpSteps pmx_dbp_steps(const DbpFiltSteps& s) { return s.s; }
__host__ __device__ __forceinline__ DbpSteps pmx_dbp_steps(const DbpTapSteps& s) { return s.s; }

__device__ __forceinline__ cpx cmul(cpx a, cpx b) { return mkc(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ cpx cmulc(cpx a, cpx b) {  // a * conj(b)
    return mkc(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y);
}
__device__ __forceinline__ cpx cadd(cpx a, cpx b) { return mkc(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ cpx csub(cpx a, cpx b) { return mkc(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ cpx cscale(cpx a, real s) { return mkc(a.x * s, a.y * s); }
__device__ __forceinline__ cpx cconj(cpx a) { return mkc(a.x, -a.y); }

// One Sa (both polarizations) per vector global access: 256-bit in FP64 (LDG.E.256 / STG.E.256 on sm_100a),
// 128-bit in FP32.
#ifdef PMX_F32
__device__ __forceinline__ void ld_sa(const cpx* p, cpx& x, cpx& y) {
    const float4 v = *reinterpret_cast<const float4*>(p);
    x = make_float2(v.x, v.y);
    y = make_float2(v.z, v.w);
}
__device__ __forceinline__ void st_sa(cpx* p, cpx x, cpx y) { *reinterpret_cast<float4*>(p) = make_float4(x.x, x.y, y.x, y.y); }
#else
__device__ __forceinline__ void ld_sa(const cpx* p, cpx& x, cpx& y) {
    asm("ld.global.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(x.x), "=d"(x.y), "=d"(y.x), "=d"(y.y) : "l"(p));
}
__device__ __forceinline__ void st_sa(cpx* p, cpx x, cpx y) {
    asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(x.x), "d"(x.y), "d"(y.x), "d"(y.y) : "memory");
}
#endif
// One Sa of a landed / staged tile in shared memory at (swizzled) byte offset `off`.  FP64: X at off, Y at
// off ^ 16 (two 128-bit accesses); FP32: both in one 128-bit access.
__device__ __forceinline__ void lds_sa(const unsigned char* base, uint32_t off, cpx& x, cpx& y) {
#ifdef PMX_F32
    const float4 v = *reinterpret_cast<const float4*>(base + off);
    x = make_float2(v.x, v.y);
    y = make_float2(v.z, v.w);
#else
    x = *reinterpret_cast<const cpx*>(base + off);
    y = *reinterpret_cast<const cpx*>(base + (off ^ 16u));
#endif
}
__device__ __forceinline__ void sts_sa(unsigned char* base, uint32_t off, cpx x, cpx y) {
#ifdef PMX_F32
    *reinterpret_cast<float4*>(base + off) = make_float4(x.x, x.y, y.x, y.y);
#else
    *reinterpret_cast<cpx*>(base + off) = x;
    *reinterpret_cast<cpx*>(base + (off ^ 16u)) = y;
#endif
}

// Branch-free sin/cos: three-term Cody-Waite reduction by pi/2 carried out with FMAs (each product q*c is
// exact inside the FMA, so the reduction stays accurate far beyond the |x| < 105615 range of the library's own
// fast path: the absolute error of the reduced argument is about 2^-53 * |x| * 6e-17, i.e. below one ulp of
// the result for |x| up to ~1e9 rad and never worse than the spacing of the doubles around x), then the fdlibm
// kernel polynomials on [-pi/4, pi/4]; <= ~1 ulp like the libm calls the reference makes in fastexp.c:41-42.
// No slow path and no branch: the compiler interleaves the evaluations a thread needs.
__device__ __forceinline__ void pmx_sincos_fast(double x, double* sp, double* cp) {
    const double q = rint(x * 6.3661977236758138e-01);
    double r = fma(q, -1.5707963267948966e+00, x);
    r = fma(q, -6.1232339957367574e-17, r);
    r = fma(q, -1.4973849048591698e-33, r);
    const int n = (int)(long long)q;
    const double z = r * r;
    double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
    ps = fma(z, ps, 2.75573137070700676789e-06);
    ps = fma(z, ps, -1.98412698298579493134e-04);
    ps = fma(z, ps, 8.33333333332248946124e-03);
    ps = fma(z, ps, -1.66666666666666324348e-01);
    const double sn = fma(z * r, ps, r);
    double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
    pc = fma(z, pc, -2.75573143513906633035e-07);
    pc = fma(z, pc, 2.48015872894767294178e-05);
    pc = fma(z, pc, -1.38888888888741095749e-03);
    pc = fma(z, pc, 4.16666666666666019037e-02);
    const double cs = fma(z * z, pc, fma(z, -0.5, 1.0));
    const double a = (n & 1) ? cs : sn, b = (n & 1) ? sn : cs;
    *sp = (n & 2) ? -a : a;
    *cp = ((n + 1) & 2) ? -b : b;
}
__device__ __forceinline__ void pmx_sincos(double x, double* sp, double* cp) { pmx_sincos_fast(x, sp, cp); }
__device__ __forceinline__ void pmx_sincos8(const double (&x)[8], double (&s)[8], double (&c)[8]) {
#pragma unroll
    for (int q = 0; q < 8; ++q) pmx_sincos_fast(x[q], &s[q], &c[q]);
}

// exp(i*a) in the field's precision for a phase argument given in double
#ifdef PMX_F32
__device__ __forceinline__ cpx pmx_cis(double a) {
    const double q = rint(a * 6.3661977236758138e-01);  // the reduction needs the double: |a| reaches 1e5 rad
    double r = fma(q, -1.5707963267948966e+00, a);
    r = fma(q, -6.1232339957367574e-17, r);
    const int n = (int)(long long)q;
    const float rf = (float)r, z = rf * rf;
    float ps = fmaf(z, -1.9515295891e-4f, 8.3321608736e-3f);
    ps = fmaf(z, ps, -1.6666654611e-1f);
    const float sn = fmaf(z * rf, ps, rf);
    float pc = fmaf(z, 2.443315711809948e-5f, -1.388731625493765e-3f);
    pc = fmaf(z, pc, 4.166664568298827e-2f);
    const float cs = fmaf(z * z, pc, fmaf(z, -0.5f, 1.0f));
    const float u = (n & 1) ? cs : sn, v = (n & 1) ? sn : cs;
    return make_float2(((n + 1) & 2) ? -v : v, (n & 2) ? -u : u);
}
// ... and for an argument already in the field's precision (nonlinear phase rotation: small angles)
__device__ __forceinline__ cpx pmx_cis_r(float a) {
    const float q = rintf(a * 6.3661977e-01f);
    float rf = fmaf(q, -1.5707963705062866e+00f, a);
    rf = fmaf(q, 4.3711388286737929e-08f, rf);
    const int n = (int)q;
    const float z = rf * rf;
    float ps = fmaf(z, -1.9515295891e-4f, 8.3321608736e-3f);
    ps = fmaf(z, ps, -1.6666654611e-1f);
    const float sn = fmaf(z * rf, ps, rf);
    float pc = fmaf(z, 2.443315711809948e-5f, -1.388731625493765e-3f);
    pc = fmaf(z, pc, 4.166664568298827e-2f);
    const float cs = fmaf(z * z, pc, fmaf(z, -0.5f, 1.0f));
    const float u = (n & 1) ? cs : sn, v = (n & 1) ? sn : cs;
    return make_float2(((n + 1) & 2) ? -v : v, (n & 2) ? -u : u);
}
#else
__device__ __forceinline__ cpx pmx_cis(double a) {
    cpx e;
    pmx_sincos_fast(a, &e.y, &e.x);
    return e;
}
__device__ __forceinline__ cpx pmx_cis_r(double a) { return pmx_cis(a); }
#endif

// exp(i*a) for |a| < 2^-6: no reduction, sin to a^7 (truncation a^9/9! < 2e-22), cos to a^6 (a^8/8! < 1e-19): 9 FP64
// instructions and nothing else, against ~24 + 15 for the general evaluation.  The step control guarantees the bound
// for every sample of a step (the nonlinear phase is at most gam*leff*max|u|^2, which it knows) and flags it.
__device__ __forceinline__ cpx pmx_cis_small(real a) {
    const real z = a * a;
#ifdef PMX_F32
    const real sn = fmaf(a * z, fmaf(z, 8.3333333e-03f, -1.6666667e-01f), a);
    const real cs = fmaf(z, fmaf(z, 4.1666668e-02f, -0.5f), 1.0f);
#else
    const real sn = fma(a * z, fma(z, fma(z, -1.984126984126984e-04, 8.333333333333333e-03), -1.6666666666666666e-01), a);
    const real cs = fma(z, fma(z, fma(z, -1.388888888888889e-03, 4.1666666666666664e-02), -0.5), 1.0);
#endif
    return mkc(cs, sn);
}

// |ux|^2+|uy|^2 in the reference's order, no FMA contraction (fiber.m:694, SURVEY A.3)
__device__ __forceinline__ real power_ref(cpx x, cpx y) {
    real p = R_ADD(R_MUL(x.x, x.x), R_MUL(x.y, x.y));
    p = R_ADD(p, R_MUL(y.x, y.x));
    p = R_ADD(p, R_MUL(y.y, y.y));
    return p;
}
