// Small fields (Nfft = L <= 4096 samples per column): the whole fiber in ONE kernel launch, the field never
// leaves the SM.  One CTA per realization-column keeps its column in registers (8 Sa per thread, L/8 threads), runs
// the complete matrix_ssfm / scalar_ssfm loop (fiber.m:459-555, 557-636) -- nextstep + checkstep, nonlinear step,
// in-CTA Stockham FFT of the full length, the step's trunks, inverse FFT, attenuation, max |u|^2 -- until the fiber is
// done, and writes the column back once.  HBM traffic: 64 B per Sa and fiber() call instead of 192 B per Sa and step.
//
// Columns of one realization ('sepfields', nfc > 1) couple through the step control (Pmax = max over the columns,
// fiber.m:694-698) and, on the scalar path with the 'x' flag, through sum_j |u_j|^2 of every sample (nl_step,
// fiber.m:793-799): the nfc CTAs of a realization form a THREAD-BLOCK CLUSTER and read each other's maxima / powers
// through distributed shared memory; every CTA runs the (deterministic) scalar step control redundantly, so no
// broadcast is needed and all CTAs leave the loop in the same iteration.
//
// Digital backpropagation (DBP = true, pmx_dbp_exec on fields of up to 4096 samples): the same kernel walks the plan's
// fixed step table (DbpSteps) instead of running the step control.  A step is the forward transform, the linear step of
// the package (dispersion negated; for a PMD-aware plan the inverse trunk product), the inverse transform, the scale
// exp(+alpha*h/2)/N (times 1/sqrt(G) on the first step of a span), on the scalar path with 'x' the cluster-wide
// sum_j |u_j|^2, and the nonlinear step with gam -> -xi*gam: pass A, B and C' of a DBP step on the three-pass route.
// No max reduction, no step control, no StepCtl write-back; the next step's package is fetched while this step runs.
// Filtered DBP (the step table is a DbpFiltSteps: pmx_dbp_set_filter): after the scale the field is parked in registers,
// the intensity it drives the nonlinear step with (P + i*s3, on the scalar path |u|^2) is transformed in the CTA,
// multiplied by H/N at the thread's bins and transformed back, and the nonlinear step runs from the filtered quantities.
// Enhanced split-step DBP (a DbpTapSteps: pmx_dbp_set_taps): after the scale the intensity goes to shared memory in time
// order and every thread takes the circular FIR of the taps at its own samples; the nonlinear step runs from that.
#pragma once
#include <type_traits>
#include <cooperative_groups.h>
#include "pmx_kernels.cuh"

namespace cg = cooperative_groups;

#define PMX_ONCHIP_MAX_L 4096
#define PMX_ONCHIP_MAX_NFC 8    // portable cluster size

template <int L>
struct OnchipSmem {
    static constexpr int T = L / 8;
    static constexpr int R16(int v) { return (v + 15) / 16 * 16; }
    static constexpr int WORK_BYTES = 2 * L * (int)sizeof(cpx);   // exchange buffer (and, before a step, XPM powers)
    static constexpr int TW_OFF = WORK_BYTES;
    static constexpr int SCR_OFF = TW_OFF + R16(pmx_tw_total(L) * (int)sizeof(cpx));
    static constexpr int PKG_OFF = SCR_OFF + PMX_B_SCR * T * (int)sizeof(double2);
    static constexpr int PLATE_OFF = PKG_OFF + (int)sizeof(StepPkg);
    static constexpr int CTL_OFF = PLATE_OFF + PMX_PKG_PLATES * (int)sizeof(PlateConst);
    static constexpr int RED_OFF = CTL_OFF + R16((int)sizeof(StepCtl));
    static constexpr int XCH_OFF = RED_OFF + 32 * 8;              // [2] column maxima, by step parity (read by the cluster)
    static constexpr int GO_OFF = XCH_OFF + 16;
    static constexpr int TOTAL = GO_OFF + 16;
};

// block-wide max of an order-preserving key; the result is valid in thread 0
__device__ __forceinline__ unsigned long long pmx_block_max_t0(unsigned long long key, void* scratch) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
        key = other > key ? other : key;
    }
    unsigned long long* red = reinterpret_cast<unsigned long long*>(scratch);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarp = (blockDim.x + 31) >> 5;
    if (lane == 0) red[warp] = key;
    __syncthreads();
    unsigned long long m = 0ull;
    if (threadIdx.x == 0)
        for (int w = 0; w < nwarp; ++w) m = red[w] > m ? red[w] : m;
    return m;
}

// The DBP instances take the step table as a third argument (Steps = DbpSteps); the forward instances keep their two.
template <typename R, int L, bool SC, bool DBP = false, typename... Steps>
__global__ void __launch_bounds__((L / 8) < 32 ? 32 : (L / 8), 1) pmx_k_onchip(PassParams p, FiberConst f, Steps... steps) {
    static_assert(sizeof...(Steps) == (DBP ? 1 : 0), "the DBP instances take one DbpSteps, the forward ones nothing");
    constexpr bool FILT = (std::is_same<Steps, DbpFiltSteps>::value || ... || false);
    constexpr bool TAPS = (std::is_same<Steps, DbpTapSteps>::value || ... || false);
    using S = OnchipSmem<L>;
    constexpr int T = L / 8;
    constexpr bool PRE = SC;
    extern __shared__ __align__(16) unsigned char smo[];
    cpx* work = reinterpret_cast<cpx*>(smo);
    cpx* stw = reinterpret_cast<cpx*>(smo + S::TW_OFF);
    StepPkg* st = reinterpret_cast<StepPkg*>(smo + S::PKG_OFF);
    PlateConst* schunk = reinterpret_cast<PlateConst*>(smo + S::PLATE_OFF);
    StepCtl* c = reinterpret_cast<StepCtl*>(smo + S::CTL_OFF);
    void* sred = smo + S::RED_OFF;
    unsigned long long* xch = reinterpret_cast<unsigned long long*>(smo + S::XCH_OFF);
    int* s_go = reinterpret_cast<int*>(smo + S::GO_OFF);
    const int col = blockIdx.x, b = blockIdx.y, t = threadIdx.x;
    const bool live = t < T;   // (L = 64, 128: the CTA is padded to one warp)
    const int tt = live ? t : 0;   // (padding threads shadow thread 0: same loads, same values, same stores)
    dcpx* scr = reinterpret_cast<dcpx*>(smo + S::SCR_OFF) + tt;
    cg::cluster_group cluster = cg::this_cluster();
    const size_t N = L;
    cpx* fld = reinterpret_cast<cpx*>(p.field) + (size_t)(b * f.nfc + col) * N * 2;
    // position of time sample n in the resident column (transposed four-step layout for 2^12, natural order below)
    auto mem = [&](int n) { return (size_t)(((n & ((1 << p.log2N2) - 1)) << p.log2N1) + (n >> p.log2N2)); };
    PMX_ASSERT(col < f.nfc && b < p.batch && mem(L - 1) < N && (int)blockDim.x >= T && (int)gridDim.x == f.nfc);

    pmx_load_stage_tw<L>(stw, p.tw_stage);
    cpx x[8], y[8];
    // ---- scalar path with the 'x' flag: sum over the columns of |u|^2 per sample, left to right (fiber.m:793-799), into y
    auto xpm_sum = [&]() {
        real* pw = reinterpret_cast<real*>(work);
        if (live) {
#pragma unroll
            for (int q = 0; q < 8; ++q) pw[t + q * T] = R_ADD(R_MUL(x[q].x, x[q].x), R_MUL(x[q].y, x[q].y));
        }
        cluster.sync();
        real sum[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) sum[q] = (real)0;
        for (int k = 0; k < f.nfc; ++k) {
            const real* rp = cluster.map_shared_rank(pw, k);
#pragma unroll
            for (int q = 0; q < 8; ++q) sum[q] = R_ADD(sum[q], rp[tt + q * T]);
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) y[q] = mkc(sum[q], (real)0);
        cluster.sync();   // everybody has read this CTA's powers: the buffer goes back to the transforms
    };
    // ---- linear step: full-length transform, the step's trunks, inverse transform (= conj o forward o conj)
    auto linear_step = [&](const PassParams& pp, int ntrunk, bool any_full, double fn0, double fn4, double dfn) {
#pragma unroll 1
        for (int dir = 0; dir < 2; ++dir) {
            CtaFFT<R, L>::run(x, y, work, work + L, tt, stw);
            if (dir == 1) break;
            if (ntrunk > 0)
                pmx_linear_bins<SC, PRE>(x, y, st, f, pp, scr, T, schunk, b, col, 0, tt, T, N, fn0, fn4, dfn, any_full);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                x[q] = cconj(x[q]);
                y[q] = cconj(y[q]);
            }
        }
    };
    if constexpr (DBP) {
        const DbpSteps ds = pmx_dbp_steps(steps...);
        // a thread's bins after the full-length transform: k = t + q*T, q < 4 positive frequencies, q >= 4 negative
        const double dfn = (double)T * f.inv_nsymb;
        const double fn0 = (double)tt * f.inv_nsymb;
        const double fn4 = (double)(tt + 4 * T - L) * f.inv_nsymb;
        // the package of step s: every thread fetches its 16-byte words into registers (issued a step ahead, landed in
        // shared memory between two steps)
        constexpr int NTH = (L / 8) < 32 ? 32 : (L / 8);
        constexpr int PW = ((int)(sizeof(StepPkg) / 16) + NTH - 1) / NTH;
        const int nw = ds.pkg_bytes / 16;
        uint4 nxt[PW];
        const PlateConst* nxt_pl = p.plates;
        auto fetch = [&](int s) {
            const uint4* src = reinterpret_cast<const uint4*>(ds.pkg + (size_t)__ldg(&ds.idx[s]) * p.batch + b);
#pragma unroll
            for (int i = 0; i < PW; ++i)
                if (t + i * NTH < nw) nxt[i] = __ldg(&src[t + i * NTH]);
            if (ds.span) nxt_pl = p.plates + (size_t)__ldg(&ds.span[s]) * ds.plate_stride;
        };
        auto land = [&]() {
#pragma unroll
            for (int i = 0; i < PW; ++i)
                if (t + i * NTH < nw) reinterpret_cast<uint4*>(st)[t + i * NTH] = nxt[i];
        };
        PMX_ASSERT(ds.nstep >= 1 && (ds.pkg_bytes == PMX_PKG_HEAD || ds.pkg_bytes == (int)sizeof(StepPkg)));
#pragma unroll
        for (int q = 0; q < 8; ++q) ld_sa(fld + 2 * mem(tt + q * T), x[q], y[q]);
        fetch(0);
        land();
        __syncthreads();
        PassParams ps = p;   // the step's plate table: its span's (PMD-aware plans)
        for (int s = 0; s < ds.nstep; ++s) {
            ps.plates = nxt_pl;
            if (s + 1 < ds.nstep) fetch(s + 1);
            const int ntrunk = st->ntrunk;
            const bool any_full = (ntrunk > 2) || (st->dzb_first == f.lcorr) || (st->dzb_last == f.lcorr);
            if constexpr (PRE) {
                if (ntrunk > 0) pmx_b_pre(scr, T, st, f, col, fn4, fn0, any_full);
            }
            linear_step(ps, ntrunk, any_full, fn0, fn4, dfn);   // ---- L(-h): dispersion negated, the package's trunks
            // ---- 1/N and the loss exp(+alpha/2*h), 1/sqrt(G) on the first step of a span
            const real sc = (real)st->scale, nsc = -sc;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                x[q] = mkc(x[q].x * sc, x[q].y * nsc);
                y[q] = mkc(y[q].x * sc, y[q].y * nsc);
            }
            if constexpr (FILT) {
                const double* hn = (steps.hn, ...);
                cpx u[8], v[8];   // the field, parked while its intensity is filtered
                real pw[8], aux[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    u[q] = x[q];
                    v[q] = y[q];
                    x[q] = f.scalar_field ? mkc(R_ADD(R_MUL(u[q].x, u[q].x), R_MUL(u[q].y, u[q].y)), (real)0)
                                          : pmx_dbp_intensity(u[q], v[q], f);
                    y[q] = mkc((real)0, (real)0);
                }
                // ifft(fft(q) .* H): forward transform, H/N at the thread's bins (conjugated), forward transform = conj(result)
                CtaFFT<R, L>::run(x, y, work, work + L, tt, stw);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const real h = (real)__ldg(&hn[tt + q * T]);
                    x[q] = mkc(x[q].x * h, -(x[q].y * h));
                    y[q] = mkc((real)0, (real)0);
                }
                CtaFFT<R, L>::run(x, y, work, work + L, tt, stw);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    pw[q] = x[q].x;
                    aux[q] = -x[q].y;
                }
                if (f.scalar_field && f.xpm) {   // sum over the columns of the filtered powers, left to right
                    real* sp = reinterpret_cast<real*>(work);
                    if (live) {
#pragma unroll
                        for (int q = 0; q < 8; ++q) sp[t + q * T] = pw[q];
                    }
                    cluster.sync();
#pragma unroll
                    for (int q = 0; q < 8; ++q) aux[q] = (real)0;
                    for (int k = 0; k < f.nfc; ++k) {
                        const real* rp = cluster.map_shared_rank(sp, k);
#pragma unroll
                        for (int q = 0; q < 8; ++q) aux[q] = R_ADD(aux[q], rp[tt + q * T]);
                    }
                    cluster.sync();
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    x[q] = u[q];
                    y[q] = v[q];
                }
                pmx_nl_step_filt(x, y, pw, aux, st->leff, f, col);   // ---- N(-xi*gam) from the filtered intensity
            } else if constexpr (TAPS) {
                const DbpTaps& tp = (steps.taps, ...);
                // the intensity in time order (q at n = t + q*T), then its circular FIR, left to right in the lag
                cpx* sq = work;
                if (live) {
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        sq[t + q * T] = f.scalar_field ? mkc(R_ADD(R_MUL(x[q].x, x[q].x), R_MUL(x[q].y, x[q].y)), (real)0)
                                                       : pmx_dbp_intensity(x[q], y[q], f);
                }
                __syncthreads();
                real pw[8], aux[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int n = tt + q * T;
                    cpx a = mkc((real)0, (real)0);
                    for (int j = 0; j <= 2 * tp.k; ++j) {
                        const real c = (real)tp.c[j];
                        const cpx v = sq[(n + tp.k - j) & (L - 1)];
                        a = mkc(fma(c, v.x, a.x), fma(c, v.y, a.y));
                    }
                    pw[q] = a.x;
                    aux[q] = a.y;
                }
                if (f.scalar_field && f.xpm) {   // sum over the columns of the filtered powers, left to right
                    real* sp = reinterpret_cast<real*>(work + L);   // (the intensity may still be read)
                    if (live) {
#pragma unroll
                        for (int q = 0; q < 8; ++q) sp[t + q * T] = pw[q];
                    }
                    cluster.sync();
#pragma unroll
                    for (int q = 0; q < 8; ++q) aux[q] = (real)0;
                    for (int k = 0; k < f.nfc; ++k) {
                        const real* rp = cluster.map_shared_rank(sp, k);
#pragma unroll
                        for (int q = 0; q < 8; ++q) aux[q] = R_ADD(aux[q], rp[tt + q * T]);
                    }
                    cluster.sync();
                }
                pmx_nl_step_filt(x, y, pw, aux, st->leff, f, col);   // ---- N(-xi*gam) from the FIR of the intensity
            } else {
                if (f.xpm) xpm_sum();   // over the backpropagated columns (the transform has released the exchange buffer)
                pmx_nl_step(x, y, st, f, col);   // ---- N(-xi*gam): the gam of f is the backpropagated one
            }
            __syncthreads();   // the package is read: the next one lands
            if (s + 1 < ds.nstep) {
                land();
                __syncthreads();
            }
        }
    } else {
        for (int i = t; i < (int)(sizeof(StepCtl) / 4); i += blockDim.x) reinterpret_cast<int*>(c)[i] = 0;
        unsigned long long vmax = 0ull;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            ld_sa(fld + 2 * mem(tt + q * T), x[q], y[q]);
            const unsigned long long key = pmx_pow_key((double)power_ref(x[q], y[q]));
            if (live) vmax = key > vmax ? key : vmax;
        }
        __syncthreads();
        int first = 1, parity = 0;
        const double dfn = (double)T * f.inv_nsymb;   // (the thread's bins, as above)
        const double fn0 = (double)tt * f.inv_nsymb;
        const double fn4 = (double)(tt + 4 * T - L) * f.inv_nsymb;
        for (;;) {
            // ---- max |u|^2 of every column of the realization (nextstep, fiber.m:693-698)
            const unsigned long long m = pmx_block_max_t0(vmax, sred);
            if (f.nfc > 1) {
                if (t == 0) xch[parity] = m;
                cluster.sync();
                if (t < f.nfc) c->umax_bits[t] = *cluster.map_shared_rank(&xch[parity], t);
                parity ^= 1;
            } else if (t == 0) {
                c->umax_bits[0] = m;
            }
            __syncthreads();
            // ---- nextstep + checkstep + step package (all CTAs of the cluster compute the same schedule)
            const bool go = pmx_ctl_step(c, st, p, f, first, b, s_go);
            __syncthreads();
            if (!go) break;
            first = 0;
            const int ntrunk = st->ntrunk;
            const bool any_full = (ntrunk > 2) || (st->dzb_first == f.lcorr) || (st->dzb_last == f.lcorr);
            if constexpr (PRE) {
                if (ntrunk > 0) pmx_b_pre(scr, T, st, f, col, fn4, fn0, any_full);
            }
            if (f.xpm) xpm_sum();
            pmx_nl_step(x, y, st, f, col);
            linear_step(p, ntrunk, any_full, fn0, fn4, dfn);
            // ---- 1/N and attenuation exp(-alpha/2*dz) (fiber.m:531-532), running max for the next step
            const real sc = (real)st->scale, nsc = -sc;
            vmax = 0ull;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                x[q] = mkc(x[q].x * sc, x[q].y * nsc);
                y[q] = mkc(y[q].x * sc, y[q].y * nsc);
                const unsigned long long key = pmx_pow_key((double)power_ref(x[q], y[q]));
                if (live) vmax = key > vmax ? key : vmax;
            }
            __syncthreads();   // the package and the exchange buffer are rewritten by the next step
        }
    }
    if (live) {
#pragma unroll
        for (int q = 0; q < 8; ++q) st_sa(fld + 2 * mem(t + q * T), x[q], y[q]);
    }
    if constexpr (!DBP) {
        if (col == 0)
            for (int i = t; i < (int)(sizeof(StepCtl) / 4); i += blockDim.x)
                reinterpret_cast<int*>(&p.ctl[b])[i] = reinterpret_cast<const int*>(c)[i];
    }
    if (f.nfc > 1) cluster.sync();   // no CTA of the cluster exits while another may still read its shared memory
}
