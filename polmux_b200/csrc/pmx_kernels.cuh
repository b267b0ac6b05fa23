// The three HBM passes of one SSFM step (fiber.m:518-537 per iteration) and the
// device-side step control (nextstep fiber.m:693-715, checkstep :739-758).
// The resident field is stored transposed in time (sample n1*N2 + n2 at n2*N1 + n1), see pass A below.
//
//   pass A  rows    : NL step (matrix_nl_step :827-851, or nl_step :786-803 on the scalar path) -> FFT over n1
//                     -> four-step twiddle W_N^(n2*k1)
//   pass B  columns : FFT over n2 -> per-bin Jones/dispersion product over the step's trunks
//                     (matrix_step :907-933) -> IFFT over k2
//   pass C  rows    : W_N^(-n2*k1) -> IFFT over k1 -> 1/N * exp(-alpha/2 dz) (:531-532) ->
//                     max |u|^2 (warp shuffle + one atomicMax per CTA and realization)
//   ctl     one CTA per realization: nextstep + checkstep for the next step, step package for the passes
//   pass C' rows    : (digital backpropagation, pmx_k_passC<..., NL = true>) as pass C, scale exp(+alpha/2 h)/N, then the nonlinear
//                     step with -xi*gam; A without the NL step and B with the dispersion negated complete the step
#pragma once
#include "pmx_fft.cuh"
#include "pmx_tma.cuh"

// ---------------------------------------------------------------------------
// step control (one thread)
__device__ __forceinline__ void pmx_ctl_next(StepCtl* c, const FiberConst& f, bool first, int b,
                                             double* trace_dz, int* trace_ntrunk) {
    if (!first) {
        if (c->state == PMX_ST_LAST) {  // the step just finished was the last one
            c->state = PMX_ST_DONE;
            for (int k = 0; k < f.nfc; ++k) c->umax_bits[k] = 0ull;
            return;
        }
        c->ntot += c->ntrunk - c->nmem;  // fiber.m:529
    }
    // ---- nextstep, fiber.m:693-715
    double pmax = 0.0;
    bool bad = false;
    for (int k = 0; k < f.nfc; ++k) {
        double um = __longlong_as_double((long long)c->umax_bits[k]);
        if (um != um) bad = true;
        double gp = __dmul_rn(f.gam[k], um);
        pmax = (k == 0) ? gp : fmax(pmax, gp);
        c->umax_bits[k] = 0ull;
    }
    if (bad) {
        c->state = PMX_ST_ERROR;
        c->err = -5;  // PMX_ERR_NUMERIC
        return;
    }
    double leff = f.phimax / pmax;
    double dl = __dmul_rn(f.alphalin, leff);
    double dz;
    if (dl >= 1.0) {
        dz = f.dzmax;
    } else {
        double step;
        if (f.alphalin == 0.0)
            step = leff;
        else
            step = __dmul_rn(-1.0 / f.alphalin, log(1.0 - dl));
        dz = (step > f.dzmax) ? f.dzmax : step;
    }
    if (first) {
        if (f.dz_first > 0.0) dz = f.dz_first;  // resumed propagation: the caller hands the step in (fiber.m:603-609)
        c->firstdz = dz;
        c->zprop = __dadd_rn(f.z_start, dz);
        c->ncycle = 1;
        c->ntot = 0;
        c->dz_miss = 0.0;
    } else {
        c->zprop = __dadd_rn(c->zprop, dz);
        c->ncycle += 1;
    }
    c->dz = dz;
    double dz_cur, zend;
    if (c->zprop < f.Lf) {
        dz_cur = dz;
        zend = c->zprop;
        c->state = PMX_ST_RUN;
    } else {
        dz_cur = __dadd_rn(__dadd_rn(f.Lf, -c->zprop), dz);  // fiber.m:538
        zend = f.Lf;
        c->state = PMX_ST_LAST;
    }
    c->dz_cur = dz_cur;
    c->leff = (f.alphalin == 0.0) ? dz_cur : (1.0 - exp(-f.alphalin * dz_cur)) / f.alphalin;  // :827-831
    c->scale = exp(-f.halfalpha * dz_cur) * f.invN;                                           // :531
    // ---- checkstep, fiber.m:739-758
    const double lcorr = f.lcorr;
    double nz = zend / lcorr;
    int nzc = (int)ceil(nz);
    int ntrunk, nmem;
    double dz_miss = c->dz_miss, dzb_first, dzb_last;
    if (dz_miss == 0.0) {
        nmem = 0;
        ntrunk = nzc - c->ntot;
        double dzlast = __dadd_rn(dz_cur, -__dmul_rn(lcorr, (double)(ntrunk - 1)));
        dzb_first = (ntrunk > 1) ? lcorr : dzlast;
        dzb_last = dzlast;
        dz_miss = __dadd_rn(lcorr, -dzlast);
    } else {
        nmem = 1;
        ntrunk = nzc - c->ntot + 1;
        if (ntrunk == 1) {
            dzb_first = dzb_last = dz_cur;
            dz_miss = __dadd_rn(dz_miss, -dz_cur);
        } else {
            double dzlast = __dadd_rn(__dadd_rn(dz_cur, -dz_miss), -__dmul_rn(lcorr, (double)(ntrunk - 2)));
            dzb_first = dz_miss;
            dzb_last = dzlast;
            dz_miss = __dadd_rn(lcorr, -dzlast);
        }
    }
    c->dz_miss = dz_miss;
    c->ntrunk = ntrunk;
    c->nmem = nmem;
    c->dzb_first = dzb_first;
    c->dzb_last = dzb_last;
    c->n_first = c->ntot - nmem;
    if (f.keep_basis)
        c->bmode = (first ? PMX_BM_ENTRY_R : (nmem ? 0 : PMX_BM_ENTRY_C)) | (c->state == PMX_ST_LAST ? PMX_BM_EXIT_R : 0);
    else
        c->bmode = PMX_BM_ENTRY_R | PMX_BM_EXIT_R;
    // largest nonlinear phase of the step: gam*leff*max|u|^2 (the CNLSE rotation angle is at most a third of it)
    if (f.spm && !f.xpm && pmax * c->leff < 0.015625) c->bmode |= PMX_BM_NL_SMALL;
    // (the per-step phasors gpf, gpl, their powers and gd3 are evaluated by pmx_ctl_step, one thread each)
    if (ntrunk > 0 && (c->ntot + ntrunk - nmem > f.nplates || c->n_first < 0)) {
        c->state = PMX_ST_ERROR;  // brf.theta(n) index error in the reference (fiber.m:910)
        c->err = -4;              // PMX_ERR_PLATE_INDEX
        return;
    }
    if (trace_dz && c->ncycle - 1 < f.trace_cap) {
        trace_dz[(size_t)b * f.trace_cap + c->ncycle - 1] = dz_cur;
        trace_ntrunk[(size_t)b * f.trace_cap + c->ncycle - 1] = ntrunk;
    }
}

// Order-preserving key of a power value: non-negative doubles order like their bit
// patterns; NaN maps above +Inf so that it wins the max and the step control flags it.
__device__ __forceinline__ unsigned long long pmx_pow_key(double pw) {
    return (pw != pw) ? 0x7ff8000000000000ull : (unsigned long long)__double_as_longlong(pw);
}

// Block-wide max (warp shuffles, then one fire-and-forget atomicMax per CTA).  The step control that
// consumes the maxima runs in its own one-thread-per-realization kernel (pmx_k_ctl) after the pass, so
// no CTA waits on an atomic's return value or on a fence.  scratch: >= 32 x 8 B of shared memory that
// is not rewritten before the CTA's next __syncthreads().
__device__ __forceinline__ void pmx_block_max(unsigned long long key, void* scratch, StepCtl* c, int col) {
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
    if (threadIdx.x == 0) {
        unsigned long long m = red[0];
        for (int w = 1; w < nwarp; ++w) m = red[w] > m ? red[w] : m;
        atomicMax(&c->umax_bits[col], m);
    }
}

// The step package of a realization (all but its state) from the step's schedule in c, by all threads of a CTA: the
// header, the scalar-mode phasors, the entry / exit matrices and the first plates of the step.  plates: the
// realization's plate table [nplates].  Shared by the step control and the PMD-aware DBP packages (pmx_k_dbp_pkg).
__device__ __forceinline__ void pmx_pkg_fill(const StepCtl* c, StepPkg* g, const FiberConst& f, const PlateConst* plates) {
    const int ntrunk = c->ntrunk, n_first = c->n_first;
    const PlateConst* plg = plates + n_first;
    // Scalar dispersion mode: the step's phasors, one thread each (seven independent evaluations instead of a serial
    // chain on thread 0): per-bin-step factors exp(-i*0.5*dgdrms*domega*dzb/lcorr) of the first / last (partial) trunk
    // with their squares and fourth powers, and exp(-i*dz*b30*domega^3), the third difference of the common phase.
    if (f.disp_scalar && threadIdx.x >= 8 && threadIdx.x < 15) {
        const int k = threadIdx.x - 8;
        const double af = -(0.5 * f.dgdrms * f.domega * c->dzb_first / f.lcorr), al = -(0.5 * f.dgdrms * f.domega * c->dzb_last / f.lcorr);
        const double a3 = -(c->dz_cur * (6.0 * f.b30_6) * f.domega * f.domega * f.domega);
        const double arg = (k == 0) ? af : (k == 1) ? al : (k == 2) ? 2.0 * af : (k == 3) ? 4.0 * af : (k == 4) ? 2.0 * al
                         : (k == 5) ? 4.0 * al : a3;
        double sn, cs;
        pmx_sincos_fast(arg, &sn, &cs);
        double* dst = (k == 0) ? &g->gpf_r : (k == 1) ? &g->gpl_r : (k == 2) ? g->gpf2 : (k == 3) ? g->gpf4 : (k == 4) ? g->gpl2
                    : (k == 5) ? g->gpl4 : &g->gd3_r;
        const bool on = (k == 6) ? (f.gvd_any != 0) : (f.pmd != 0);
        dst[0] = on ? cs : 0.0;
        dst[1] = on ? sn : 0.0;
    }
    if (threadIdx.x == 0) {
        g->dz_cur = c->dz_cur;
        g->leff = c->leff;
        g->scale = c->scale;
        g->dzb_first = c->dzb_first;
        g->dzb_last = c->dzb_last;
        g->db0_last = (f.pmd && ntrunk > 0) ? plg[ntrunk - 1].db0 : 0.0;
        g->ntrunk = ntrunk;
        g->n_first = n_first;
        g->bmode = f.pmd ? c->bmode : (c->bmode & PMX_BM_NL_SMALL);
    }
    if (!f.pmd || ntrunk <= 0) return;
    for (int i = threadIdx.x; i < 16; i += blockDim.x) {
        if (i < 8) {  // entry matrix
            double v = (i == 0 || i == 6) ? 1.0 : 0.0;
            if (c->bmode & PMX_BM_ENTRY_R) {  // R^H: element (r,cc) = conj(R(cc,r))
                const int r = i >> 2, cc = (i >> 1) & 1, im = i & 1;
                v = (&plg[0].r11r)[(cc * 2 + r) * 2 + im];
                if (im) v = -v;
            } else if (c->bmode & PMX_BM_ENTRY_C) {
                v = (&plg[-1].c11r)[i];
            }
            g->E[i] = v;
        } else {      // exit matrix
            g->X[i - 8] = (&plg[ntrunk - 1].r11r)[i - 8];
        }
    }
    constexpr int PLD = (int)(sizeof(PlateConst) / sizeof(double));
    const int n = (ntrunk < PMX_PKG_PLATES ? ntrunk : PMX_PKG_PLATES) * PLD;
    const double* src = reinterpret_cast<const double*>(plg);
    double* dst = reinterpret_cast<double*>(g->plates);
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
}

// nextstep + checkstep for the step about to run and the step package of the realization, by all threads of a CTA
// (thread 0 runs the scalar logic, everybody copies).  c, g: the realization's control block and package (global
// memory for the pass kernels, shared memory in the single-CTA kernel of small fields).  -> false when the realization
// has no further step.
__device__ __forceinline__ bool pmx_ctl_step(StepCtl* c, StepPkg* g, const PassParams& p, const FiberConst& f, int first, int b,
                                             int* s_go) {
    if (threadIdx.x == 0) {
        const int go = first || c->state < PMX_ST_DONE;
        if (go) pmx_ctl_next(c, f, first != 0, b, p.trace_dz, p.trace_ntrunk);
        g->state = c->state;
        *s_go = go && c->state < PMX_ST_DONE;
    }
    __syncthreads();
    if (!*s_go) return false;
    pmx_pkg_fill(c, g, f, p.plates + (f.plate_sets > 1 ? (size_t)b * f.nplates : 0));
    return true;
}

// Step control, one CTA per realization: nextstep + checkstep for the step about to run (first: fiber.m:512; afterwards
// :534-536) from the per-column maxima the previous kernel left, and the step package the pass kernels fetch with
// their tiles.
static __global__ void __launch_bounds__(128) pmx_k_ctl(PassParams p, FiberConst f, int first) {
    const int b = blockIdx.x;
    __shared__ int s_go;
    if (p.pdl) {
        pmx_pdl_launch_dependents();
        pmx_pdl_wait();
    }
    pmx_ctl_step(&p.ctl[b], &p.pkg[b], p, f, first, b, &s_go);
}

// ---------------------------------------------------------------------------
// Initial max |u|^2 of a resident field + first step schedule (fiber.m:512).
static __global__ void __launch_bounds__(256) pmx_k_init(PassParams p, FiberConst f) {
    extern __shared__ cpx smem[];
    const int bc = blockIdx.y, b = bc / f.nfc, col = bc % f.nfc;
    const size_t N = (size_t)p.N1 * p.N2;
    const cpx* fld = reinterpret_cast<const cpx*>(p.field) + (size_t)bc * N * 2;
    unsigned long long vmax = 0ull;
    for (size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (size_t)gridDim.x * blockDim.x) {
        cpx x, y;
        ld_sa(fld + 2 * n, x, y);
        unsigned long long key = pmx_pow_key(power_ref(x, y));
        vmax = key > vmax ? key : vmax;
    }
    pmx_block_max(vmax, smem, &p.ctl[b], col);
}

// smem region stride (in cpx) between the rows/columns a CTA works on: offset so
// that lanes of different regions fall in different 16-byte bank groups.
template <int L, int GROUP>
struct PmxSmem {
    static constexpr int BASE = 2 * L;
#ifdef PMX_F32
    // FP32 exchanges float4 points (16 B = two cpx): the GROUP regions a warp touches at once are offset by 128/GROUP
    // bytes so that their lanes fall in different 16-byte bank groups (and every region stays 16-byte aligned)
    static constexpr int OFF = (GROUP > 1) ? ((16 / GROUP) > 2 ? (16 / GROUP) : 2) : 0;
#else
    static constexpr int OFF = (GROUP > 1) ? ((8 / GROUP) > 0 ? (8 / GROUP) : 1) : 0;
#endif
    static constexpr int STRIDE = BASE + OFF;
};

// Four-step twiddle of one row/column, W_N^(r*m) for m in [0, L): two-level table per row,
// W^(r*m) = lo[m & (2^LO-1)] * hi[m >> LO].  The rows live in a per-plan table in global memory
// ([rows][PER], built once with exact-argument sincospi, L2-resident) and reach shared memory with the
// tile's bulk copy: no per-tile trigonometry, no dependent global load before the store.
template <int L>
struct PmxTw4 {
    static constexpr int LOG = pmx_ilog2(L);
    static constexpr int LO = (LOG + 1) / 2, HI = LOG - LO;
    static constexpr int NLO = 1 << LO, NHI = 1 << HI, PER = NLO + NHI;
};

#define PMX_LIVE_CAP 64    // realizations whose done-flags a CTA caches in shared memory

// Pass B: per-thread phasors (double2 in both builds) that depend on the tile's bins and the step only (not on the
// field) are evaluated BEFORE the CTA waits for its tile and parked here while the forward transform needs the registers.
#define PMX_B_SCR 6

// Shared-memory plan of a pass CTA working on G rows (pass B) or G columns (passes A, C) of
// length L.  PF: the next tile is prefetched by TMA into its own landing buffer while the
// current one is computed; !PF: the tile lands in the exchange buffer itself and the next load
// is issued as soon as the last exchange of the current tile is over.  KIND: 0 = pass A, 1 = B, 2 = C.
// The per-tile auxiliary data (step package of the realization + four-step twiddle rows) is
// double-buffered: tile i uses aux[i & 1] while the bulk copies for tile i+1 land in the other one.
template <int L, int G, bool PF, int KIND>
struct PassSmem {
    static constexpr int T = L / 8;
    static constexpr int THREADS = G * T;
    static constexpr int TILE_BYTES = G * L * PMX_SA_BYTES;
    static constexpr int WORK_BYTES = G * PmxSmem<L, G>::STRIDE * (int)sizeof(cpx);
    static constexpr int WORK_OFF = PF ? ((TILE_BYTES + 1023) / 1024) * 1024 : 0;
    static constexpr int TW_OFF = WORK_OFF + ((WORK_BYTES + 15) / 16) * 16;   // stage twiddles
    static constexpr int PKG_BYTES = (KIND == 1) ? (int)sizeof(StepPkg) : PMX_PKG_HEAD_AC;
    static constexpr int TAB_BYTES = (KIND == 1) ? 0 : ((G * PmxTw4<L>::PER * (int)sizeof(cpx) + 15) / 16) * 16;
    static constexpr int AUX_BYTES = PKG_BYTES + TAB_BYTES;
    static constexpr int AUX_OFF = TW_OFF + ((pmx_tw_total(L) * (int)sizeof(cpx) + 15) / 16) * 16;
    static constexpr int PLATE_OFF = AUX_OFF + 2 * AUX_BYTES;               // pass B: chunks of trunks beyond the package
    static constexpr int SCR_OFF = PLATE_OFF + ((KIND == 1) ? PMX_PKG_PLATES * (int)sizeof(PlateConst) : 0);
    static constexpr int SCR_BYTES = (KIND == 1) ? PMX_B_SCR * THREADS * (int)sizeof(double2) : 0;   // [PMX_B_SCR][THREADS]
    static constexpr int RED_OFF = SCR_OFF + SCR_BYTES;
    static constexpr int LIVE_OFF = RED_OFF + 32 * 8;
    static constexpr int MBAR_OFF = LIVE_OFF + PMX_LIVE_CAP;
    static constexpr int TOTAL = MBAR_OFF + 32;  // the dynamic shared array is declared 1024-byte aligned
    static constexpr int LOAD_BYTES = TILE_BYTES + AUX_BYTES;  // bytes one tile's mbarrier phase expects (passes A, C)
    static_assert(WORK_BYTES >= TILE_BYTES, "exchange buffer must hold a landed tile");
    static_assert(sizeof(StepPkg) % 16 == 0 && PMX_PKG_HEAD % 16 == 0 && PMX_PKG_HEAD_AC % 16 == 0,
                  "bulk copies move multiples of 16 bytes");
};

// copy the per-L stage-twiddle table into shared memory (once per persistent CTA)
template <int L>
__device__ __forceinline__ void pmx_load_stage_tw(cpx* dst, const void* src_) {
    const cpx* __restrict__ src = reinterpret_cast<const cpx*>(src_);
    for (int i = threadIdx.x; i < pmx_tw_total(L); i += blockDim.x) dst[i] = __ldg(&src[i]);
}

// the swizzled TMA landing buffers need a 1024-byte aligned base; the extern array is declared so
__device__ __forceinline__ unsigned char* pmx_checked1024(unsigned char* p) {
    if (pmx_smem_u32(p) & 1023u) __trap();
    return p;
}

// Per-plan four-step twiddle rows: tab[r*PER + e] = W_N^(r*m(e)), m(e) = e for e < NLO, (e-NLO) << LO above.
static __global__ void pmx_k_fill_tw4(cpx* tab, int rows, int lo_bits, int per, int row_stride, double two_over_N) {
    const int nlo = 1 << lo_bits;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)rows * per;
         i += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(i / per), e = (int)(i % per);
        const int m = (e < nlo) ? e : ((e - nlo) << lo_bits);
        double sn, cs;
        sincospi(-(double)((long long)r * m) * two_over_N, &sn, &cs);  // exact argument: N is a power of two
        tab[(size_t)r * row_stride + e] = mkc((real)cs, (real)sn);
    }
}

// done-flags of the realizations, cached per CTA (the step control runs between passes, so they are
// constant while a pass runs)
__device__ __forceinline__ void pmx_cache_live(unsigned char* sdone, const PassParams& p) {
    if (p.batch <= PMX_LIVE_CAP)
        for (int i = threadIdx.x; i < p.batch; i += blockDim.x) sdone[i] = p.pkg[i].state >= PMX_ST_DONE ? 1 : 0;
}
__device__ __forceinline__ bool pmx_is_done(const unsigned char* sdone, const PassParams& p, int b) {
    return (p.batch <= PMX_LIVE_CAP) ? (sdone[b] != 0) : (p.pkg[b].state >= PMX_ST_DONE);
}

// realization / column of a flat realization-column index
__device__ __forceinline__ void pmx_split_bc(int bc, const FiberConst& f, int& b, int& col) {
    if (f.nfc == 1) {
        b = bc;
        col = 0;
    } else {
        b = (int)__umulhi((unsigned)bc, f.nfc_magic);
        col = bc - b * f.nfc;
    }
}

#ifdef PMX_TIMING
#define PMX_T_DECL long long t_ph[8] = {0, 0, 0, 0, 0, 0, 0, 0}; long long t_last = clock64();
#define PMX_T_MARK(i) { long long t_now = clock64(); t_ph[i] += t_now - t_last; t_last = t_now; }
#define PMX_T_FLUSH(kind) if (p.dbg && threadIdx.x == 0) { for (int i = 0; i < 8; ++i) atomicAdd((unsigned long long*)&p.dbg[(kind) * 8 + i], (unsigned long long)t_ph[i]); }
#else
#define PMX_T_DECL
#define PMX_T_MARK(i)
#define PMX_T_FLUSH(kind)
#endif

// resident-CTA target of the launch bounds: 384 (prefetching) / 512 threads per SM in FP64, 768 in FP32
#define PMX_TBUDGET(pf) ((PMX_SA_BYTES == 32) ? ((pf) ? 384 : 512) : 768)
#define PMX_MINB(threads, pf) ((PMX_TBUDGET(pf) / (threads)) > 0 ? (PMX_TBUDGET(pf) / (threads)) : 1)

// ---------------------------------------------------------------------------
// Scalar path with the 'x' flag (nl_step, fiber.m:786-799): the nonlinear phase of column k needs
// sum_j |u_j|^2 of the same sample.  The scalar path has no Y polarization, so the row sum is parked in the
// (zero) Y slot of every column's Sa, where pass A finds it with the sample it already loads; pass A
// clears the slot again.  One read + a 16-byte write per Sa and step.
static __global__ void __launch_bounds__(256) pmx_k_xpm_sum(PassParams p, FiberConst f) {
    const int b = blockIdx.y;
    if (p.pkg[b].state >= PMX_ST_DONE) return;
    const size_t N = (size_t)p.N1 * p.N2;
    cpx* fld = reinterpret_cast<cpx*>(p.field) + (size_t)b * f.nfc * N * 2;
    for (size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (size_t)gridDim.x * blockDim.x) {
        real sum = (real)0;
        for (int k = 0; k < f.nfc; ++k) {  // sum(pow,2), left to right
            const cpx x = fld[((size_t)k * N + n) * 2];
            sum = R_ADD(sum, R_ADD(R_MUL(x.x, x.x), R_MUL(x.y, x.y)));
        }
        for (int k = 0; k < f.nfc; ++k) fld[((size_t)k * N + n) * 2 + 1] = mkc(sum, (real)0);
    }
}

// ---------------------------------------------------------------------------
// The nonlinear step on the eight samples a thread holds: matrix_nl_step (fiber.m:827-851, Manakov or CNLSE) or, on
// the scalar path, nl_step (:786-803; with the 'x' flag y[q].x must hold sum_j |u_j|^2 of the sample).
__device__ __forceinline__ void pmx_nl_step(cpx (&x)[8], cpx (&y)[8], const StepPkg* st, const FiberConst& f, int col) {
    if (f.scalar_field) {  // nl_step (fiber.m:786-803): u .* fastexp(-gam.*pow*leff), Y absent
        if (f.spm || f.xpm) {
            const real ngam = (real)(-f.gam[col]), leff = (real)st->leff;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                real pw = R_ADD(R_MUL(x[q].x, x[q].x), R_MUL(x[q].y, x[q].y));
                if (f.xpm) {  // y.x holds sum(pow,2) of this sample (pmx_k_xpm_sum)
                    const real two_s = R_MUL((real)2, y[q].x);
                    pw = f.spm ? R_ADD(two_s, -pw) : R_MUL((real)2, R_ADD(y[q].x, -pw));
                }
                x[q] = cmul(x[q], pmx_cis_r(R_MUL(R_MUL(ngam, pw), leff)));
            }
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) y[q] = mkc((real)0, (real)0);
    } else if (f.spm) {
        const real gamleff = (real)__dmul_rn(f.gam[col], st->leff);
        const real ngl = -gamleff;
        const bool nl_small = (st->bmode & PMX_BM_NL_SMALL) != 0;  // uniform for the tile
        cpx e[8];
        if (nl_small) {
#pragma unroll
            for (int q = 0; q < 8; ++q) e[q] = pmx_cis_small(R_MUL(ngl, power_ref(x[q], y[q])));
        } else {
#pragma unroll
            for (int q = 0; q < 8; ++q) e[q] = pmx_cis_r(R_MUL(ngl, power_ref(x[q], y[q])));
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            x[q] = cmul(x[q], e[q]);
            y[q] = cmul(y[q], e[q]);
        }
        if (!f.manakov) {  // CNLSE: rotation by gamleff*s3/3 around the third Stokes axis (:841-851)
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const real s3 = (real)2.0 * (x[q].x * y[q].y - x[q].y * y[q].x);
                const real a3 = R_MUL(gamleff, s3) / (real)3.0;
                e[q] = nl_small ? pmx_cis_small(a3) : pmx_cis_r(a3);
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const cpx ux = x[q], uy = y[q];
                const real cs = e[q].x, sn = e[q].y;
                x[q] = mkc(cs * ux.x + sn * uy.x, cs * ux.y + sn * uy.y);
                y[q] = mkc(cs * uy.x - sn * ux.x, cs * uy.y - sn * ux.y);
            }
        }
    }
}

// pmx_nl_step of filtered DBP (pmx_dbp_set_filter): every quantity the step computes from |u|^2 comes filtered, the rest
// is unchanged.  pw: the filtered power (|ux|^2+|uy|^2, on the scalar path |u|^2 of the column); aux: the filtered s3
// (CNLSE) or, on the scalar path with the 'x' flag, the sum over the columns of the filtered powers.
template <int NQ>
__device__ __forceinline__ void pmx_nl_step_filt(cpx (&x)[NQ], cpx (&y)[NQ], const real (&pw)[NQ], const real (&aux)[NQ],
                                                 double leff, const FiberConst& f, int col) {
    if (f.scalar_field) {
        if (f.spm || f.xpm) {
            const real ngam = (real)(-f.gam[col]), rl = (real)leff;
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                real p = pw[q];
                if (f.xpm) p = f.spm ? R_ADD(R_MUL((real)2, aux[q]), -p) : R_MUL((real)2, R_ADD(aux[q], -p));
                x[q] = cmul(x[q], pmx_cis_r(R_MUL(R_MUL(ngam, p), rl)));
            }
        }
#pragma unroll
        for (int q = 0; q < NQ; ++q) y[q] = mkc((real)0, (real)0);
    } else if (f.spm) {
        const real gamleff = (real)__dmul_rn(f.gam[col], leff);
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const cpx e = pmx_cis_r(R_MUL(-gamleff, pw[q]));
            x[q] = cmul(x[q], e);
            y[q] = cmul(y[q], e);
        }
        if (!f.manakov) {   // the s3 rotation with the filtered s3
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                const cpx e = pmx_cis_r(R_MUL(gamleff, aux[q]) / (real)3.0);
                const cpx ux = x[q], uy = y[q];
                x[q] = mkc(e.x * ux.x + e.y * uy.x, e.x * ux.y + e.y * uy.y);
                y[q] = mkc(e.x * uy.x - e.y * ux.x, e.x * uy.y - e.y * ux.y);
            }
        }
    }
}

// The intensity filtered DBP low-passes, P + i*s3 (s3 = 0 for Manakov) of the two-polarization sample (x, y).
__device__ __forceinline__ cpx pmx_dbp_intensity(cpx x, cpx y, const FiberConst& f) {
    return mkc(power_ref(x, y), f.manakov ? (real)0 : (real)2.0 * (x.x * y.y - x.y * y.x));
}

// Filtered DBP on the three passes, two pointwise kernels around the filter plan (grid.y: realization-columns bc).
// pmx_k_dbp_intensity writes P + i*s3 of column bc into the work field, two columns per Sa: column bc/2, slot bc&1 (X, Y);
// an odd last column leaves its Y slot zero.  Both fields have N samples per column in the same layout.
static __global__ void __launch_bounds__(256) pmx_k_dbp_intensity(PassParams p, FiberConst f, cpx* __restrict__ work) {
    const int bc = blockIdx.y, nbc = p.batch * f.nfc;
    const size_t N = (size_t)p.N1 * p.N2;
    const cpx* fld = reinterpret_cast<const cpx*>(p.field) + (size_t)bc * N * 2;
    cpx* w = work + (size_t)(bc >> 1) * N * 2 + (bc & 1);
    const bool pad = (bc & 1) == 0 && bc + 1 == nbc;
    for (size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (size_t)gridDim.x * blockDim.x) {
        cpx x, y;
        ld_sa(fld + 2 * n, x, y);
        w[2 * n] = pmx_dbp_intensity(x, y, f);
        if (pad) w[2 * n + 1] = mkc((real)0, (real)0);
    }
}
// pmx_k_dbp_nl_filt: N(-xi*gam, h) of the step package pkg[b] from the filtered intensity in the work field
static __global__ void __launch_bounds__(256) pmx_k_dbp_nl_filt(PassParams p, FiberConst f, const cpx* __restrict__ work,
                                                                const StepPkg* __restrict__ pkg) {
    const int bc = blockIdx.y, b = bc / f.nfc, col = bc - b * f.nfc;
    const size_t N = (size_t)p.N1 * p.N2;
    cpx* fld = reinterpret_cast<cpx*>(p.field) + (size_t)bc * N * 2;
    const cpx* w = work + (size_t)(bc >> 1) * N * 2 + (bc & 1);
    const double leff = pkg[b].leff;
    for (size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (size_t)gridDim.x * blockDim.x) {
        cpx x[1], y[1];
        ld_sa(fld + 2 * n, x[0], y[0]);
        const cpx q = w[2 * n];
        const real pw[1] = {q.x}, s3[1] = {q.y};
        pmx_nl_step_filt(x, y, pw, s3, leff, f, col);
        st_sa(fld + 2 * n, x[0], y[0]);
    }
}

// Enhanced split-step DBP on the three passes (pmx_dbp_set_taps): N(-xi*gam, h) of the step package pkg[b] from the FIR
//   q~[n] = sum_{m=-k..k} c[m+k] * q[(n - m) mod N]   (left to right in m)
// of the intensity pmx_k_dbp_intensity left in the work field (grid.y: the work column, realization-columns 2y and 2y+1).
// The resident column is time-transposed: sample n1*N2 + n2 sits at n2*N1 + n1, so the time neighbour n - m is row n2 - m
// at the same n1, or across the row wrap row n2 - m +- N2 at n1 -+ 1 (mod N1: circular at n = 0 and n = N - 1; k <= 32
// < N2 wraps once at most).  A CTA takes PMX_FIR_ROWS rows of PMX_FIR_COLS positions along n1 and lands them with a k-row
// halo on either side in shared memory.  It reads the intensity only from the work field, never a sample another CTA
// has already rotated, so the result does not depend on the order the CTAs run in.
#define PMX_FIR_ROWS 64
#define PMX_FIR_COLS 16
#define PMX_FIR_RB 4
static __global__ void __launch_bounds__(256) pmx_k_dbp_nl_fir(PassParams p, FiberConst f, const cpx* __restrict__ work,
                                                               const StepPkg* __restrict__ pkg, DbpTaps tp) {
    constexpr int TY = 256 / PMX_FIR_COLS;
    static_assert(TY * PMX_FIR_RB == PMX_FIR_ROWS, "a thread row per PMX_FIR_RB rows of the tile");
    extern __shared__ __align__(16) unsigned char smf[];
    cpx* sq = reinterpret_cast<cpx*>(smf);   // [PMX_FIR_ROWS + 2k][PMX_FIR_COLS][2]: time row r0 - k + r at row r
    const int K = tp.k, N1 = p.N1, N2 = p.N2;
    const int tiles1 = N1 / PMX_FIR_COLS;
    const int c0 = (int)(blockIdx.x % tiles1) * PMX_FIR_COLS, r0 = (int)(blockIdx.x / tiles1) * PMX_FIR_ROWS;
    const int tx = threadIdx.x % PMX_FIR_COLS, ty = threadIdx.x / PMX_FIR_COLS;
    const size_t N = (size_t)N1 * N2;
    PMX_ASSERT(K >= 0 && K <= 32 && K < N2 && r0 + PMX_FIR_ROWS <= N2 && blockDim.x == 256);
    const cpx* w = work + (size_t)blockIdx.y * N * 2;
    for (int r = ty; r < PMX_FIR_ROWS + 2 * K; r += TY) {
        int rr = r0 - K + r, n1 = c0 + tx;
        if (rr < 0) {
            rr += N2;
            n1 = (n1 - 1) & (N1 - 1);
        } else if (rr >= N2) {
            rr -= N2;
            n1 = (n1 + 1) & (N1 - 1);
        }
        cpx a, b;
        ld_sa(w + 2 * ((size_t)rr * N1 + n1), a, b);
        sq[2 * (r * PMX_FIR_COLS + tx)] = a;
        sq[2 * (r * PMX_FIR_COLS + tx) + 1] = b;
    }
    __syncthreads();
    // a thread takes PMX_FIR_RB consecutive rows: the rows the taps read slide by one from tap to tap, so every tap lands
    // one new row per thread and feeds PMX_FIR_RB independent sums
    const int i0 = ty * PMX_FIR_RB;
    cpx qa[PMX_FIR_RB], qb[PMX_FIR_RB], wa[PMX_FIR_RB], wb[PMX_FIR_RB];
    const cpx* s = sq + 2 * ((i0 + 2 * K) * PMX_FIR_COLS + tx);   // tap 0 (lag m = -k) of row i0 + r: row i0 + r + 2k
#pragma unroll
    for (int r = 0; r < PMX_FIR_RB; ++r) {
        qa[r] = qb[r] = mkc((real)0, (real)0);
        wa[r] = s[2 * r * PMX_FIR_COLS];
        wb[r] = s[2 * r * PMX_FIR_COLS + 1];
    }
    for (int j = 0;;) {
        const real c = (real)tp.c[j];
#pragma unroll
        for (int r = 0; r < PMX_FIR_RB; ++r) {
            qa[r] = mkc(fma(c, wa[r].x, qa[r].x), fma(c, wa[r].y, qa[r].y));
            qb[r] = mkc(fma(c, wb[r].x, qb[r].x), fma(c, wb[r].y, qb[r].y));
        }
        if (++j > 2 * K) break;
#pragma unroll
        for (int r = PMX_FIR_RB - 1; r > 0; --r) {
            wa[r] = wa[r - 1];
            wb[r] = wb[r - 1];
        }
        s -= 2 * PMX_FIR_COLS;
        wa[0] = s[0];
        wb[0] = s[1];
    }
    const int nbc = p.batch * f.nfc;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int bc = 2 * (int)blockIdx.y + h;
        if (bc >= nbc) break;   // an odd last work column: its Y slot is padding
        const int b = bc / f.nfc, col = bc - b * f.nfc;
        cpx* fld = reinterpret_cast<cpx*>(p.field) + (size_t)bc * N * 2;
        const double leff = pkg[b].leff;
#pragma unroll
        for (int r = 0; r < PMX_FIR_RB; ++r) {
            const size_t pos = (size_t)(r0 + i0 + r) * N1 + c0 + tx;
            cpx x[1], y[1];
            ld_sa(fld + 2 * pos, x[0], y[0]);
            const cpx q = h ? qb[r] : qa[r];
            const real pw[1] = {q.x}, s3[1] = {q.y};
            pmx_nl_step_filt(x, y, pw, s3, leff, f, col);
            st_sa(fld + 2 * pos, x[0], y[0]);
        }
    }
}

// ---------------------------------------------------------------------------
// Tile walk shared by the three passes (persistent CTAs): tile -> (realization-column bc, group inside it),
// serpentine direction, skipping finished realizations.
struct PmxWalk {
    int ltpb, tpb_mask, total, reverse;
    __device__ __forceinline__ int phys(int tl) const { return reverse ? total - 1 - tl : tl; }
};

// ---------------------------------------------------------------------------
// The field lives in HBM TRANSPOSED with respect to time: sample n = n1*N2 + n2 sits at n2*N1 + n1 (the
// upload / download kernels do the permutation once per fiber() call).  The two passes that touch the time
// domain (A and C) therefore work on CONTIGUOUS rows (fixed n2, all n1) and only pass B, which has the
// arithmetic to hide it, walks columns (fixed k1, all n2) through narrow TMA boxes:
//   memory [n2][n1] --A: FFT over n1, in place--> [n2][k1] --B: column k1, FFT over n2 / Jones / IFFT over k2,
//   in place--> [n2][k1] --C: IFFT over k1, in place--> [n2][n1].
// (Measured on B200: a TMA copy of 32-byte-wide column tiles runs at 4.4 TB/s, contiguous tiles at 6.5 TB/s.)
//
// pass A: G adjacent rows per tile, thread (t fastest, rl).  Persistent CTAs walk the tile list
// (tile = realization-column bc, row group); finished realizations are skipped.
// FUSED (a batch of ONE realization, the reference-style fiber() call): there is no step-control kernel between pass C
// and pass A.  Every CTA of pass A runs nextstep + checkstep itself from the control block the previous step left
// (deterministic scalar code: all CTAs arrive at the same package), under its first tile load; CTA 0 writes the new
// control block -- into the OTHER of two blocks, so that no CTA reads what another writes -- and the package passes B
// and C fetch.  One dependent launch per step less.
#define PMX_FUSED_BYTES (((int)sizeof(StepCtl) + 15) / 16 * 16 + ((int)sizeof(StepPkg) + 15) / 16 * 16 + 16)
template <typename R, int L, int G, bool PF, bool FUSED = false>
__global__ void __launch_bounds__(G*(L / 8), PMX_MINB(G*(L / 8), PF))
    pmx_k_passA(PassParams p, FiberConst f, const __grid_constant__ CUtensorMap tmap) {
    using S = PassSmem<L, G, PF, 0>;
    using W = PmxTw4<L>;
    constexpr int T = L / 8;
    constexpr int LINES = G * L * PMX_SA_BYTES / 128;  // 128-byte lines per tile
    extern __shared__ __align__(1024) unsigned char smraw[];
    unsigned char* sm = pmx_checked1024(smraw);
    unsigned char* in = sm;  // PF: landing buffer at 0; !PF: WORK_OFF == 0, lands in the exchange buffer
    cpx* work = reinterpret_cast<cpx*>(sm + S::WORK_OFF);
    cpx* stw = reinterpret_cast<cpx*>(sm + S::TW_OFF);
    unsigned char* aux0 = sm + S::AUX_OFF;
    unsigned char* sdone = sm + S::LIVE_OFF;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(sm + S::MBAR_OFF);
    const int rl = threadIdx.x / T, t = threadIdx.x % T;
    const size_t N = (size_t)p.N1 * p.N2;
    PmxWalk wk;
    wk.ltpb = p.log2N2 - pmx_ilog2(G);
    wk.tpb_mask = (1 << wk.ltpb) - 1;
    wk.total = (p.batch * f.nfc) << wk.ltpb;
    wk.reverse = p.reverse;
    const int total = wk.total;

    auto live = [&](int tl) {
        while (tl < total) {
            int b_, col_;
            pmx_split_bc(wk.phys(tl) >> wk.ltpb, f, b_, col_);
            if (!pmx_is_done(sdone, p, b_)) break;
            tl += gridDim.x;
        }
        return tl;
    };
    // a tile = G adjacent rows of the [N2][N1] time-domain matrix = G*L contiguous Sa
    auto issue = [&](int tl, int buf) {  // one thread
        pmx_fence_proxy_async();
        const int tt = wk.phys(tl), bc = tt >> wk.ltpb, row0 = (tt & wk.tpb_mask) * G;
        pmx_mbar_expect_tx(mbar, S::LOAD_BYTES);
        for (int l0 = 0; l0 < LINES; l0 += 256)
            pmx_tma_load_3d(in + l0 * 128, &tmap, 0, (tt & wk.tpb_mask) * LINES + l0, p.bc0 + bc, mbar);
        int b_, col_;
        pmx_split_bc(bc, f, b_, col_);
        unsigned char* a = aux0 + buf * S::AUX_BYTES;
        pmx_bulk_load(a, &p.pkg[b_], S::PKG_BYTES, mbar);
        pmx_bulk_load(a + S::PKG_BYTES, reinterpret_cast<const cpx*>(p.tw4) + (size_t)row0 * W::PER, S::TAB_BYTES, mbar);
    };
    if (threadIdx.x == 0) {
        pmx_mbar_init(mbar, 1);
        pmx_fence_mbar_init();
    }
    pmx_load_stage_tw<L>(stw, p.tw_stage);
    if (p.pdl) {  // everything above is independent of the previous kernel of the stream
        pmx_pdl_launch_dependents();
        pmx_pdl_wait();
    }
    const StepPkg* fpkg = nullptr;
    if constexpr (FUSED) {
        for (int i = threadIdx.x; i < PMX_LIVE_CAP; i += blockDim.x) sdone[i] = 0;   // (one realization; decided below)
    } else {
        pmx_cache_live(sdone, p);
    }
    __syncthreads();
    int tile = live(blockIdx.x), it = 0;
    if (threadIdx.x == 0 && tile < total) issue(tile, 0);
    uint32_t phase = 0;
    if constexpr (FUSED) {
        constexpr int CB = ((int)sizeof(StepCtl) + 15) / 16 * 16, PB = ((int)sizeof(StepPkg) + 15) / 16 * 16;
        unsigned char* fz = sm + ((S::TOTAL + 15) / 16) * 16;
        StepCtl* sc = reinterpret_cast<StepCtl*>(fz);
        StepPkg* sp = reinterpret_cast<StepPkg*>(fz + CB);
        int* s_go = reinterpret_cast<int*>(fz + CB + PB);
        PMX_ASSERT(p.batch == 1 && p.ctl_out != nullptr && p.ctl_out != p.ctl);
        for (int i = threadIdx.x; i < (int)(sizeof(StepCtl) / 4); i += blockDim.x)
            reinterpret_cast<int*>(sc)[i] = reinterpret_cast<const int*>(p.ctl)[i];
        for (int i = threadIdx.x; i < (int)(sizeof(StepPkg) / 4); i += blockDim.x) reinterpret_cast<int*>(sp)[i] = 0;
        __syncthreads();
        PassParams q = p;
        if (blockIdx.x != 0) {   // the schedule trace is written once
            q.trace_dz = nullptr;
            q.trace_ntrunk = nullptr;
        }
        const bool go = pmx_ctl_step(sc, sp, q, f, p.first, 0, s_go);
        __syncthreads();
        if (blockIdx.x == 0) {
            for (int i = threadIdx.x; i < (int)(sizeof(StepCtl) / 4); i += blockDim.x)
                reinterpret_cast<int*>(p.ctl_out)[i] = reinterpret_cast<const int*>(sc)[i];
            for (int i = threadIdx.x; i < (int)(sizeof(StepPkg) / 4); i += blockDim.x)
                reinterpret_cast<int*>(p.pkg)[i] = reinterpret_cast<const int*>(sp)[i];
        }
        if (!go) {   // the fiber is finished: nothing to do (the tile already asked for must still land)
            if (tile < total) pmx_mbar_wait(mbar, phase);
            return;
        }
        fpkg = sp;
    }
    PMX_T_DECL
    while (tile < total) {
        const int tt = wk.phys(tile), bc = tt >> wk.ltpb, row0 = (tt & wk.tpb_mask) * G;
        int b, col;
        pmx_split_bc(bc, f, b, col);
        PMX_ASSERT(tt >= 0 && tt < total && bc < p.batch * f.nfc && b < p.batch && col < f.nfc && b * f.nfc + col == bc);
        PMX_ASSERT(row0 + G <= p.N2 && L == p.N1);
        const unsigned char* aux = aux0 + (it & 1) * S::AUX_BYTES;
        const StepPkg* st = FUSED ? fpkg : reinterpret_cast<const StepPkg*>(aux);
        const cpx* gtab = reinterpret_cast<const cpx*>(aux + S::PKG_BYTES);
        const int next = live(tile + gridDim.x);
        cpx x[8], y[8];
        PMX_T_MARK(0)
        pmx_mbar_wait(mbar, phase);
        phase ^= 1u;
        PMX_T_MARK(1)
#pragma unroll
        for (int q = 0; q < 8; ++q) lds_sa(in, pmx_swz<7>((uint32_t)((rl * L + t + q * T) * PMX_SA_BYTES)), x[q], y[q]);
        __syncthreads();
        if (PF && threadIdx.x == 0 && next < total) issue(next, (it + 1) & 1);
        PMX_T_MARK(2)
        pmx_nl_step(x, y, st, f, col);   // ---- nonlinear step, fiber.m:832-851
        cpx* sx = work + rl * PmxSmem<L, G>::STRIDE;
        cpx* sy = sx + L;
        PMX_T_MARK(3)
        // the next tile lands in the exchange buffer: its load goes out as soon as the last exchange is read, under the
        // last butterfly stage and the store
        CtaFFT<R, L>::run(x, y, sx, sy, t, stw, [&] {
            if (!PF && threadIdx.x == 0 && next < total) issue(next, (it + 1) & 1);
        });
        PMX_T_MARK(4)
        // four-step twiddle W_N^(n2*k1), k1 = t + q*T, from the row's two-level table; straight to HBM (the row is
        // contiguous: 32 lanes x 32 B per store instruction)
        {
            const cpx* tb = gtab + rl * W::PER;
            const cpx wl = tb[t & (W::NLO - 1)];
            cpx* base = reinterpret_cast<cpx*>(p.field) + ((size_t)bc * N + (size_t)(row0 + rl) * L) * 2;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const cpx w = cmul(wl, tb[W::NLO + ((t + q * T) >> W::LO)]);
                st_sa(base + (size_t)(t + q * T) * 2, cmul(x[q], w), cmul(y[q], w));
            }
        }
        PMX_T_MARK(5)
        tile = next;
        ++it;
        __syncthreads();  // everyone is done with this tile's auxiliary buffer
        PMX_T_MARK(6)
    }
    PMX_T_FLUSH(0)
}

// ---------------------------------------------------------------------------
// pass B: G adjacent columns (k1) of the [n2][k1] matrix per tile, thread (cl fastest, t)

// u <- M*u for the eight bins of a thread, M row-major (re,im) in shared memory
__device__ __forceinline__ void pmx_apply2x2(cpx (&x)[8], cpx (&y)[8], const double* M) {
    const cpx m11 = mkc((real)M[0], (real)M[1]), m12 = mkc((real)M[2], (real)M[3]);
    const cpx m21 = mkc((real)M[4], (real)M[5]), m22 = mkc((real)M[6], (real)M[7]);
#pragma unroll
    for (int q = 0; q < 8; ++q) {  // four-term FMA chains: 16 instructions per bin instead of 20
        const cpx a = x[q], b = y[q];
        x[q] = mkc(fma(-m12.y, b.y, fma(m12.x, b.x, fma(-m11.y, a.y, m11.x * a.x))),
                   fma(m12.y, b.x, fma(m12.x, b.y, fma(m11.y, a.x, m11.x * a.y))));
        y[q] = mkc(fma(-m22.y, b.y, fma(m22.x, b.x, fma(-m21.y, a.y, m21.x * a.x))),
                   fma(m22.y, b.x, fma(m22.x, b.y, fma(m21.y, a.x, m21.x * a.y))));
    }
}

// Scalar dispersion mode: what a thread of pass B knows about its eight bins before the field arrives.
// The bins k = k1 + N1*(t + q*T) are equally spaced in frequency; in rising order they are q = 4..7 (negative
// frequencies) then q = 0..3, so with j = (q + 4) & 7 the angular frequency is wb + j*domega.
// The phasors below are DOUBLE in both builds (phases reach 1e3..1e5 rad and progressions over a step's trunks must not
// repeat a float rounding error): they are rounded to the field's precision where they meet the data.
typedef double2 dcpx;
__device__ __forceinline__ dcpx dmk(double a, double b) { return make_double2(a, b); }
__device__ __forceinline__ dcpx dmul(dcpx a, dcpx b) { return dmk(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ dcpx dmulc(dcpx a, dcpx b) { return dmk(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y); }   // a*conj(b)
__device__ __forceinline__ dcpx dcis(double a) {
    dcpx e;
    pmx_sincos_fast(a, &e.y, &e.x);
    return e;
}
__device__ __forceinline__ cpx pmx_to_cpx(dcpx e) { return mkc((real)e.x, (real)e.y); }
struct PmxBPre {
    dcpx E, D1, D2;    // common phase exp(i*phi(j)), phi = -betat*dz: value, first and second difference at j = 4
    dcpx E0, pf, pl;   // exp(-i*db1/2) (whole trunks), first / last trunk phasor (partial trunks), all at j = 0
};

// phi(w) = -dz*(b1*w + b2/2*w^2 + b30/6*w^3) at w = wc; its forward differences over the bin spacing d are evaluated
// from their closed forms (no cancellation):
//   D1 = phi(w+d) - phi(w)   = -dz*d*(b1 + b2*(w + d/2) + b30_6*(3*w*(w + d) + d*d))
//   D2 = D1(w+d) - D1(w)     = -dz*d*d*(b2 + 6*b30_6*(w + d))
//   D3                        = -dz*6*b30_6*d^3          (per step: StepPkg.gd3)
// The six phasors go straight to the thread's scratch slots scr[slot*stride] (PmxBPre order).
__device__ __forceinline__ void pmx_b_pre(dcpx* scr, int stride, const StepPkg* st, const FiberConst& f, int col, double fnb,
                                          double fnc, bool any_full) {
    const double wb = __dmul_rn(f.w0, fnb);   // lowest bin (j = 0): base of the trunk phasor progressions
    if (f.gvd_any) {
        const double wc = __dmul_rn(f.w0, fnc);   // middle bin (j = 4, q = 0): anchor of the common-phase recurrence
        const double b1 = f.beta1[col], b2 = f.beta2[col], d = f.domega, dz = st->dz_cur;
        const double w2 = __dmul_rn(wc, wc);
        double bt = __dadd_rn(__dmul_rn(wc, b1), __dmul_rn(__dmul_rn(0.5, w2), b2));   // betat as fiber.m:355-356
        bt = __dadd_rn(bt, __dmul_rn(__dmul_rn(w2, wc), f.b30_6));
        const double ndzd = -(dz * d);
        const double a1 = ndzd * (b1 + fma(b2, fma(0.5, d, wc), f.b30_6 * fma(3.0 * wc, wc + d, d * d)));
        const double a2 = ndzd * d * fma(6.0 * f.b30_6, wc + d, b2);
        scr[0 * stride] = dcis(-(bt * dz));
        scr[1 * stride] = dcis(a1);
        scr[2 * stride] = dcis(a2);
    }
    if (f.pmd) {
        const double d1b = __dmul_rn(f.dgdrms, wb);  // db1 = dgdrms*omega (:358)
        scr[3 * stride] = any_full ? dcis(-0.5 * d1b) : dmk(1.0, 0.0);
        // partial trunks: deltabeta = 0.5*(db1+db0)*dzb/lcorr  (:925)
        scr[4 * stride] = dcis(-(0.5 * (d1b + st->plates[0].db0) * st->dzb_first / f.lcorr));
        scr[5 * stride] = dcis(-(0.5 * (d1b + st->db0_last) * st->dzb_last / f.lcorr));
    }
}

// One trunk in the PSP basis of its plate is diag(e, conj(e)) with e(j) = b*g^j over the thread's bins (deltabeta is
// linear in omega).  Written as conj(e) * diag(e^2, 1): the scalar conj(e) is common to both polarizations and is
// collected over the trunks of the step in closed form (conj(prod b) * conj(prod g)^j, folded into the common-phase
// recurrence), so a trunk multiplies ONE polarization by e(j)^2 = b2 * g2^j.  Two interleaved chains (even / odd j)
// advanced by g4 = g2^2: three phasors live at a time.  (FP32 fields: the chains run in double and every phasor is
// rounded once where it is applied, so the trunks of a step do not repeat one rounding error.)
__device__ __forceinline__ void pmx_b_diag2(cpx (&x)[8], dcpx b2, dcpx g2, dcpx g4) {
    dcpx ea = b2, eo = dmul(b2, g2);
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
        const int qa = (j + 4) & 7, qo = (j + 5) & 7;
        x[qa] = cmul(x[qa], pmx_to_cpx(ea));
        x[qo] = cmul(x[qo], pmx_to_cpx(eo));
        if (j < 6) {
            ea = dmul(ea, g4);
            eo = dmul(eo, g4);
        }
    }
}
// u <- [ka kb; -conj(kb) ka] * u, ka real: 12 FMAs per bin
__device__ __forceinline__ void pmx_b_applyK(cpx (&x)[8], cpx (&y)[8], double ka_, double kbr_, double kbi_) {
    const real ka = (real)ka_, kbr = (real)kbr_, kbi = (real)kbi_;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const cpx a = x[q], b = y[q];
        x[q] = mkc(fma(-kbi, b.y, fma(kbr, b.x, ka * a.x)), fma(kbi, b.x, fma(kbr, b.y, ka * a.y)));
        y[q] = mkc(fma(-kbi, a.y, fma(-kbr, a.x, ka * b.x)), fma(kbi, a.x, fma(-kbr, a.y, ka * b.y)));
    }
}

// common phase of the eight bins by a difference recurrence anchored at the thread's MIDDLE bin (j = 4, i.e. q = 0):
//   upwards    E(j+1) = E(j)*D1(j),        D1(j+1) = D1(j)*D2(j),        D2(j+1) = D2(j)*D3
//   downwards  E(j-1) = E(j)*conj(D1(j-1)), D1(j-1) = D1(j)*conj(D2(j-1)), D2(j-1) = D2(j)*conj(D3)
// three evaluations + 18 complex products instead of eight evaluations; a rounding error of the first / second
// difference is amplified by at most 4 / 6 (binomials of the distance to the anchor).
__device__ __forceinline__ void pmx_b_common(cpx (&x)[8], cpx (&y)[8], dcpx E, dcpx D1, dcpx D2, dcpx D3) {
    {
        const cpx e0 = pmx_to_cpx(E);
        x[0] = cmul(x[0], e0);
        y[0] = cmul(y[0], e0);
    }
    {   // j = 5, 6, 7  <->  q = 1, 2, 3
        dcpx e = E, d1 = D1, d2 = D2;
#pragma unroll
        for (int q = 1; q < 4; ++q) {
            e = dmul(e, d1);
            const cpx ef = pmx_to_cpx(e);
            x[q] = cmul(x[q], ef);
            y[q] = cmul(y[q], ef);
            if (q < 3) d1 = dmul(d1, d2);
            if (q < 2) d2 = dmul(d2, D3);
        }
    }
    {   // j = 3, 2, 1, 0  <->  q = 7, 6, 5, 4
        dcpx e = E, d1 = D1, d2 = D2;
#pragma unroll
        for (int q = 7; q >= 4; --q) {
            d2 = dmulc(d2, D3);
            d1 = dmulc(d1, d2);
            e = dmulc(e, d1);
            const cpx ef = pmx_to_cpx(e);
            x[q] = cmul(x[q], ef);
            y[q] = cmul(y[q], ef);
        }
    }
}

// ---------------------------------------------------------------------------
// The linear step on the eight bins a thread holds after a forward transform (matrix_step, fiber.m:907-933, and
// lin_step on the scalar path): entry basis change, the step's trunks, exit basis change, common phase.  The bins
// are k = k1 + N1*(t + q*T) (q = 0..7) of a length-N spectrum: pass B calls it with the four-step split of the
// field, the single-CTA kernel of small fields with N1 = 1, k1 = 0.  All threads of the CTA must call it together
// (steps with more trunks than the package holds reload plate chunks behind __syncthreads).
//   scr / scr_stride : the thread's pre-evaluated phasors (pmx_b_pre, double2), scalar dispersion mode
//   schunk           : shared buffer of PMX_PKG_PLATES plates
template <bool SC, bool PRE>
__device__ __forceinline__ void pmx_linear_bins(cpx (&x)[8], cpx (&y)[8], const StepPkg* st, const FiberConst& f,
                                                const PassParams& p, const dcpx* scr, int scr_stride, PlateConst* schunk,
                                                int b, int col, int k1, int t, int T, size_t N, double fn0, double fn4,
                                                double dfn, bool any_full) {
    constexpr int PLD = (int)(sizeof(PlateConst) / sizeof(double));
    const int ntrunk = st->ntrunk, bmode = st->bmode;
    PMX_ASSERT((size_t)k1 + (size_t)p.N1 * (size_t)(t + 7 * T) < N && ntrunk >= 0 && st->n_first >= 0 &&
               st->n_first + ntrunk <= f.nplates);
    (void)scr;
    (void)scr_stride;
    (void)fn0;
    (void)dfn;
    if constexpr (!SC) {
        if (p.hfilt) {   // a linear filter: u(k) <- H(k) * u(k) from the plan's table, the product taken in double
            const double2* h = p.hfilt + (size_t)col * (size_t)p.hfilt_stride + (size_t)k1 * p.N2;
            PMX_ASSERT((size_t)k1 * p.N2 + (size_t)(t + 7 * T) < N && (p.hfilt_stride == 0 || (size_t)p.hfilt_stride == N));
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const double2 e = __ldg(&h[t + q * T]);
                const double xr = x[q].x, xi = x[q].y, yr = y[q].x, yi = y[q].y;
                x[q] = mkc((real)(xr * e.x - xi * e.y), (real)(xr * e.y + xi * e.x));
                y[q] = mkc((real)(yr * e.x - yi * e.y), (real)(yr * e.y + yi * e.x));
            }
            return;
        }
    }
        const double dz_cur = st->dz_cur;
        // scalar phase common to both polarizations collected over the trunks: conj(Bacc) * conj(Gacc)^j
        dcpx Bacc = dmk(1.0, 0.0), Gacc = dmk(1.0, 0.0);
        if (f.pmd) {
            const double lcorr = f.lcorr, dzb_first = st->dzb_first, dzb_last = st->dzb_last;
            if (bmode & (PMX_BM_ENTRY_R | PMX_BM_ENTRY_C)) pmx_apply2x2(x, y, st->E);  // (:920-921)
            // vector dispersion mode: db1 of the thread's bins; whole trunks share exp(-i*db1/2) per bin.  (FP32: that
            // factor is kept in double and each trunk's exp(-i*(db1+db0)/2) is formed in double and rounded once,
            // otherwise the same float-rounded phasor would repeat its phase error in up to nplates factors.)
            double d1[(SC) ? 1 : 8];
#ifdef PMX_F32
            double2 Ed[(SC) ? 1 : 8];
#else
            cpx e1[(SC) ? 1 : 8];
#endif
            // scalar dispersion mode: phasors of the step's whole / first / last trunk at the thread's lowest bin (from
            // the pre-phase); db1 is linear in omega, so the other bins follow by a geometric progression (pmx_b_diag2)
            dcpx E0b = dmk(1.0, 0.0), pfb = E0b, plb = E0b, pprev = E0b;
            if constexpr (SC) {
                E0b = scr[3 * scr_stride];
                pfb = scr[4 * scr_stride];
                plb = scr[5 * scr_stride];
            } else {
                const double* d1p = p.db1_p + (size_t)col * N + (size_t)k1 * p.N2;
#pragma unroll
                for (int q = 0; q < 8; ++q) d1[q] = __ldg(&d1p[t + q * T]);
                if (any_full) {
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
#ifdef PMX_F32
                        pmx_sincos_fast(-0.5 * d1[q], &Ed[q].y, &Ed[q].x);
#else
                        e1[q] = pmx_cis(-0.5 * d1[q]);
#endif
                    }
                }
            }
            for (int k0 = 0; k0 < ntrunk; k0 += PMX_PKG_PLATES) {
                const PlateConst* pl = st->plates;
                if (k0 > 0) {  // more trunks than the package holds (one-step 'gp--' runs): next chunk
                    __syncthreads();
                    const PlateConst* plg = p.plates + (f.plate_sets > 1 ? (size_t)b * f.nplates : 0) + st->n_first + k0;
                    const int n = ((ntrunk - k0) < PMX_PKG_PLATES ? (ntrunk - k0) : PMX_PKG_PLATES) * PLD;
                    const double* s_ = reinterpret_cast<const double*>(plg);
                    double* d_ = reinterpret_cast<double*>(schunk);
                    for (int i = threadIdx.x; i < n; i += blockDim.x) d_[i] = __ldg(&s_[i]);
                    __syncthreads();
                    pl = schunk;
                }
                const int kend = (ntrunk - k0) < PMX_PKG_PLATES ? ntrunk : k0 + PMX_PKG_PLATES;
                for (int k = k0; k < kend; ++k) {
                    const PlateConst& P = pl[k - k0];
                    const double dzb = (k == 0) ? dzb_first : ((k == ntrunk - 1) ? dzb_last : lcorr);
                    if constexpr (SC) {
                        dcpx bb, g, g2, g4;
                        if (dzb == lcorr) {  // whole trunk: exp(-i*0.5*(db1+db0)) = exp(-i*db1/2) * exp(-i*db0/2)
                            bb = dmul(E0b, dmk(P.h0r, P.h0i));
                            g = dmk(f.g1r, f.g1i);
                            g2 = dmk(f.g2r, f.g2i);
                            g4 = dmk(f.g4r, f.g4i);
                        } else if (k == 0) {  // partial trunk (first or last of the step)
                            bb = pfb;
                            g = dmk(st->gpf_r, st->gpf_i);
                            g2 = dmk(st->gpf2[0], st->gpf2[1]);
                            g4 = dmk(st->gpf4[0], st->gpf4[1]);
                        } else {
                            bb = plb;
                            g = dmk(st->gpl_r, st->gpl_i);
                            g2 = dmk(st->gpl2[0], st->gpl2[1]);
                            g4 = dmk(st->gpl4[0], st->gpl4[1]);
                        }
                        bb = dmul(bb, pprev);        // left phase of the boundary matrix just applied
                        Bacc = dmul(Bacc, bb);
                        Gacc = dmul(Gacc, g);
                        pmx_b_diag2(x, dmul(bb, bb), g2, g4);
                        if (k < ntrunk - 1) {        // basis change matR(n+1)' * matR(n) = diag(p, p*) * K
                            pmx_b_applyK(x, y, P.ka, P.kbr, P.kbi);
                            pprev = dmk(P.pr, P.pi);
                        }
                        continue;
                    } else {
                        if (dzb == lcorr) {  // whole trunk: exp(-i*db1/2) * exp(-i*db0/2)
                            const cpx h0 = mkc((real)P.h0r, (real)P.h0i);
#pragma unroll
                            for (int q = 0; q < 8; ++q) {
#ifdef PMX_F32
                                const cpx e = mkc((real)(Ed[q].x * P.h0r - Ed[q].y * P.h0i), (real)(Ed[q].x * P.h0i + Ed[q].y * P.h0r));
                                (void)h0;
#else
                                const cpx e = cmul(e1[q], h0);
#endif
                                x[q] = cmul(x[q], e);
                                y[q] = cmulc(y[q], e);
                            }
                        } else {  // partial trunk: deltabeta = 0.5*(db1+db0)*dzb/lcorr  (:925)
#pragma unroll
                            for (int q = 0; q < 8; ++q) {
                                const cpx e = pmx_cis(-(0.5 * (d1[q] + P.db0) * dzb / lcorr));
                                x[q] = cmul(x[q], e);
                                y[q] = cmulc(y[q], e);
                            }
                        }
                    }
                    if (k < ntrunk - 1) pmx_apply2x2(x, y, &P.c11r);  // basis change matR(n+1)' * matR(n)
                }
            }
            if (bmode & PMX_BM_EXIT_R) pmx_apply2x2(x, y, st->X);  // back to the laboratory basis (:931-932)
        }
        if constexpr (PRE) {  // common phase exp(-i*betat*sum(dzb)) (:924,927-928) times the trunks' common scalar
            // at the anchor bin (j = 4) the collected scalar is conj(Bacc * Gacc^4)
            const dcpx G2 = dmul(Gacc, Gacc);
            const dcpx S4 = dmul(Bacc, dmul(G2, G2));
            if (f.gvd_any)
                pmx_b_common(x, y, dmulc(scr[0 * scr_stride], S4), dmulc(scr[1 * scr_stride], Gacc),
                             scr[2 * scr_stride], dmk(st->gd3_r, st->gd3_i));
            else if (f.pmd)
                pmx_b_common(x, y, dmk(S4.x, -S4.y), dmk(Gacc.x, -Gacc.y), dmk(1.0, 0.0), dmk(1.0, 0.0));
        } else if (f.gvd_any) {  // common phase exp(-i*betat*sum(dzb))  (:924,927-928)
            double a[8];
            if constexpr (SC) {  // betat regenerated per bin (:355-356)
                const double b1 = f.beta1[col], b2 = f.beta2[col];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const double fn = (q < 4) ? fn0 + (double)q * dfn : fn4 + (double)(q - 4) * dfn;  // exact
                    const double w = __dmul_rn(f.w0, fn);
                    const double w2 = __dmul_rn(w, w);
                    double bt = __dadd_rn(__dmul_rn(w, b1), __dmul_rn(__dmul_rn(0.5, w2), b2));
                    bt = __dadd_rn(bt, __dmul_rn(__dmul_rn(w2, w), f.b30_6));
                    a[q] = -(bt * dz_cur);
                }
            } else {
                const double* bt = p.betat_p + (size_t)col * N + (size_t)k1 * p.N2;
#pragma unroll
                for (int q = 0; q < 8; ++q) a[q] = -(__ldg(&bt[t + q * T]) * dz_cur);
            }
            cpx e[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) e[q] = pmx_cis(a[q]);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                x[q] = cmul(x[q], e[q]);
                y[q] = cmul(y[q], e[q]);
            }
        }
}

template <typename R, int L, int G, bool PF, bool SC>
__global__ void __launch_bounds__(G*(L / 8), PMX_MINB(G*(L / 8), PF))
    pmx_k_passB(PassParams p, FiberConst f, const __grid_constant__ CUtensorMap tmap) {
    using S = PassSmem<L, G, PF, 1>;
    constexpr int T = L / 8, SA = PMX_SA_BYTES, PITCH = G * SA, MASK = PITCH / 16 - 1;
    constexpr bool PRE = SC;   // scalar dispersion mode: data-independent phasors before the tile wait
    extern __shared__ __align__(1024) unsigned char smraw[];
    unsigned char* sm = pmx_checked1024(smraw);
    unsigned char* in = sm;
    cpx* work = reinterpret_cast<cpx*>(sm + S::WORK_OFF);
    cpx* stw = reinterpret_cast<cpx*>(sm + S::TW_OFF);
    unsigned char* aux0 = sm + S::AUX_OFF;
    PlateConst* schunk = reinterpret_cast<PlateConst*>(sm + S::PLATE_OFF);
    dcpx* scr = reinterpret_cast<dcpx*>(sm + S::SCR_OFF) + threadIdx.x;   // [slot][THREADS]
    unsigned char* sdone = sm + S::LIVE_OFF;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(sm + S::MBAR_OFF);      // [0]: tile, [1]: step package
    const int cl = threadIdx.x % G, t = threadIdx.x / G;
    const size_t N = (size_t)p.N1 * p.N2;
    PmxWalk wk;
    wk.ltpb = p.log2N1 - pmx_ilog2(G);
    wk.tpb_mask = (1 << wk.ltpb) - 1;
    wk.total = (p.batch * f.nfc) << wk.ltpb;
    wk.reverse = p.reverse;
    const int total = wk.total;

    auto live = [&](int tl) {
        while (tl < total) {
            int b_, col_;
            pmx_split_bc(wk.phys(tl) >> wk.ltpb, f, b_, col_);
            if (!pmx_is_done(sdone, p, b_)) break;
            tl += gridDim.x;
        }
        return tl;
    };
    // The step package travels on its own mbarrier: it is a few KB out of the L2 and lands long before the tile, so
    // the threads can evaluate everything that does not depend on the field while the tile is still in flight.
    auto issue_pkg = [&](int tl, int buf) {  // one thread
        pmx_fence_proxy_async();
        const int tt = wk.phys(tl), bc = tt >> wk.ltpb;
        int b_, col_;
        pmx_split_bc(bc, f, b_, col_);
        pmx_mbar_expect_tx(mbar + 1, S::PKG_BYTES);
        pmx_bulk_load(aux0 + buf * S::AUX_BYTES, &p.pkg[b_], S::PKG_BYTES, mbar + 1);
    };
    auto issue_tile = [&](int tl) {  // one thread
        pmx_fence_proxy_async();
        const int tt = wk.phys(tl), bc = tt >> wk.ltpb, c0 = (tt & wk.tpb_mask) * G;
        pmx_mbar_expect_tx(mbar, S::TILE_BYTES);
        for (int r0 = 0; r0 < L; r0 += 256) pmx_tma_load_3d(in + r0 * PITCH, &tmap, c0 * 4, r0, p.bc0 + bc, mbar);
    };
    auto issue = [&](int tl, int buf) {  // one thread
        issue_pkg(tl, buf);
        issue_tile(tl);
    };
    if (threadIdx.x == 0) {
        pmx_mbar_init(mbar, 1);
        pmx_mbar_init(mbar + 1, 1);
        pmx_fence_mbar_init();
    }
    pmx_load_stage_tw<L>(stw, p.tw_stage);
    if (p.pdl) {  // everything above is independent of the previous kernel of the stream
        pmx_pdl_launch_dependents();
        pmx_pdl_wait();
    }
    pmx_cache_live(sdone, p);
    __syncthreads();
    int tile = live(blockIdx.x), it = 0;
    if (threadIdx.x == 0 && tile < total) issue(tile, 0);
    uint32_t phase = 0;
    PMX_T_DECL
    while (tile < total) {
        const int tt = wk.phys(tile), bc = tt >> wk.ltpb, c0 = (tt & wk.tpb_mask) * G;
        int b, col;
        pmx_split_bc(bc, f, b, col);
        const int k1 = c0 + cl;
        PMX_ASSERT(tt >= 0 && tt < total && bc < p.batch * f.nfc && b < p.batch && col < f.nfc && b * f.nfc + col == bc);
        PMX_ASSERT(k1 < p.N1 && L == p.N2);
        const unsigned char* aux = aux0 + (it & 1) * S::AUX_BYTES;
        const StepPkg* st = reinterpret_cast<const StepPkg*>(aux);
        const int next = live(tile + gridDim.x);
        cpx x[8], y[8];
        PMX_T_MARK(0)
        pmx_mbar_wait(mbar + 1, phase);
        const int ntrunk = st->ntrunk;
        // Scalar dispersion mode: a thread's bins are k = k1 + N1*(t + q*T): q < 4 on the positive-frequency side,
        // q >= 4 on the negative one, equally spaced by domega; bin 4 lies four spacings BELOW bin 0.
        const long long kb = (long long)k1 + (long long)p.N1 * t;
        const double dfn = (double)((long long)p.N1 * T) * f.inv_nsymb;
        const double fn0 = (double)kb * f.inv_nsymb;
        const double fn4 = (double)(kb + (long long)p.N1 * 4 * T - (long long)N) * f.inv_nsymb;
        const bool any_full = (ntrunk > 2) || (st->dzb_first == f.lcorr) || (st->dzb_last == f.lcorr);
        if constexpr (PRE) {
            if (ntrunk > 0) pmx_b_pre(scr, S::THREADS, st, f, col, fn4, fn0, any_full);
        }
        PMX_T_MARK(7)
        pmx_mbar_wait(mbar, phase);
        phase ^= 1u;
        PMX_T_MARK(1)
#pragma unroll
        for (int q = 0; q < 8; ++q) lds_sa(in, pmx_swz<MASK>((uint32_t)((t + q * T) * PITCH + cl * SA)), x[q], y[q]);
        if (threadIdx.x == 0) pmx_tma_wait_read();  // previous tile's store has left the exchange buffer
        __syncthreads();
        if (PF && threadIdx.x == 0 && next < total) issue(next, (it + 1) & 1);
        cpx* sx = work + cl * PmxSmem<L, G>::STRIDE;
        cpx* sy = sx + L;
        PMX_T_MARK(2)
        // forward transform, per-bin product, inverse transform (= conj o forward o conj): one copy of
        // the transform code, run twice
#pragma unroll 1
        for (int dir = 0; dir < 2; ++dir) {
            CtaFFT<R, L>::run(x, y, sx, sy, t, stw);
            if (dir == 1) break;
            PMX_T_MARK(3)

            // ---- linear step in the frequency domain, fiber.m:907-933
            if (ntrunk > 0) {
                pmx_linear_bins<SC, PRE>(x, y, st, f, p, scr, S::THREADS, schunk, b, col, k1, t, T, N, fn0, fn4, dfn, any_full);
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                x[q] = cconj(x[q]);
                y[q] = cconj(y[q]);
            }
            PMX_T_MARK(4)
        }
        PMX_T_MARK(5)
        // the second transform was run on conj(spectrum): conj(result) is the inverse transform.  Its four-step
        // twiddle W_N^(-n2*k1) is applied by pass C when it loads the sample (pass C has FP64 slots to spare).
        // The column tile is staged (same swizzled layout as it landed) in the exchange buffer and TMA-stored.
        unsigned char* outb = reinterpret_cast<unsigned char*>(work);
#pragma unroll
        for (int q = 0; q < 8; ++q)
            sts_sa(outb, pmx_swz<MASK>((uint32_t)((t + q * T) * PITCH + cl * SA)), cconj(x[q]), cconj(y[q]));
        pmx_fence_proxy_async();
        __syncthreads();  // tile staged; everyone is done with this tile's auxiliary buffer and plate chunk
        if (threadIdx.x == 0) {
            for (int r0 = 0; r0 < L; r0 += 256) pmx_tma_store_3d(&tmap, c0 * 4, r0, p.bc0 + bc, outb + r0 * PITCH);
            pmx_tma_commit();
            if (!PF && next < total) {  // the next tile lands in this same buffer
                pmx_tma_wait_read();
                issue(next, (it + 1) & 1);
            }
        }
        tile = next;
        ++it;
        PMX_T_MARK(6)
    }
    PMX_T_FLUSH(1)
    if (threadIdx.x == 0) pmx_tma_wait_read();
}

// ---------------------------------------------------------------------------
// pass C: rows like pass A: four-step twiddle, inverse transform over k1, attenuation, max reduction.  The
// running maximum stays in registers across the tiles a CTA handles for one realization-column and is published
// (one atomicMax per CTA) when the CTA moves on to another one.
// NL (pass C' of a digital-backpropagation step, pmx_dbp_exec): after the scale exp(+alpha/2*h)/N of the step package
// (times 1/sqrt(G) on the first step of a span), the nonlinear step N(-xi*gam) of pmx_nl_step on the rows the CTA holds,
// in time, before the store.  The caller hands in a FiberConst whose gam is -xi*gam and a package whose bmode has no
// PMX_BM_NL_SMALL.  The schedule is known before the first launch, so there is no max reduction and no step control.
template <typename R, int L, int G, bool PF, bool NL>
__global__ void __launch_bounds__(G*(L / 8), PMX_MINB(G*(L / 8), PF))
    pmx_k_passC(PassParams p, FiberConst f, const __grid_constant__ CUtensorMap tmap) {
    using S = PassSmem<L, G, PF, 2>;
    using W = PmxTw4<L>;
    constexpr int T = L / 8;
    constexpr int LINES = G * L * PMX_SA_BYTES / 128;
    extern __shared__ __align__(1024) unsigned char smraw[];
    unsigned char* sm = pmx_checked1024(smraw);
    unsigned char* in = sm;
    cpx* work = reinterpret_cast<cpx*>(sm + S::WORK_OFF);
    void* sred = sm + S::RED_OFF;
    cpx* stw = reinterpret_cast<cpx*>(sm + S::TW_OFF);
    unsigned char* aux0 = sm + S::AUX_OFF;
    unsigned char* sdone = sm + S::LIVE_OFF;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(sm + S::MBAR_OFF);
    const int rl = threadIdx.x / T, t = threadIdx.x % T;
    const size_t N = (size_t)p.N1 * p.N2;
    PmxWalk wk;
    wk.ltpb = p.log2N2 - pmx_ilog2(G);
    wk.tpb_mask = (1 << wk.ltpb) - 1;
    wk.total = (p.batch * f.nfc) << wk.ltpb;
    wk.reverse = p.reverse;
    const int total = wk.total;

    auto live = [&](int tl) {
        while (tl < total) {
            int b_, col_;
            pmx_split_bc(wk.phys(tl) >> wk.ltpb, f, b_, col_);
            if (!pmx_is_done(sdone, p, b_)) break;
            tl += gridDim.x;
        }
        return tl;
    };
    // a tile = G adjacent rows of the [N2][N1] time-domain matrix = G*L contiguous Sa
    auto issue = [&](int tl, int buf) {  // one thread
        pmx_fence_proxy_async();
        const int tt = wk.phys(tl), bc = tt >> wk.ltpb, row0 = (tt & wk.tpb_mask) * G;
        pmx_mbar_expect_tx(mbar, S::LOAD_BYTES);
        for (int l0 = 0; l0 < LINES; l0 += 256)
            pmx_tma_load_3d(in + l0 * 128, &tmap, 0, (tt & wk.tpb_mask) * LINES + l0, p.bc0 + bc, mbar);
        int b_, col_;
        pmx_split_bc(bc, f, b_, col_);
        unsigned char* a = aux0 + buf * S::AUX_BYTES;
        pmx_bulk_load(a, &p.pkg[b_], S::PKG_BYTES, mbar);
        pmx_bulk_load(a + S::PKG_BYTES, reinterpret_cast<const cpx*>(p.tw4) + (size_t)row0 * W::PER, S::TAB_BYTES, mbar);
    };
    if (threadIdx.x == 0) {
        pmx_mbar_init(mbar, 1);
        pmx_fence_mbar_init();
    }
    pmx_load_stage_tw<L>(stw, p.tw_stage);
    if (p.pdl) {  // everything above is independent of the previous kernel of the stream
        pmx_pdl_launch_dependents();
        pmx_pdl_wait();
    }
    pmx_cache_live(sdone, p);
    __syncthreads();
    int tile = live(blockIdx.x), it = 0;
    if (threadIdx.x == 0 && tile < total) issue(tile, 0);
    uint32_t phase = 0;
    unsigned long long vmax = 0ull;  // running max of this thread for the current realization-column
    PMX_T_DECL
    while (tile < total) {
        const int tt = wk.phys(tile), bc = tt >> wk.ltpb, row0 = (tt & wk.tpb_mask) * G;
        int b, col;
        pmx_split_bc(bc, f, b, col);
        PMX_ASSERT(tt >= 0 && tt < total && bc < p.batch * f.nfc && b < p.batch && col < f.nfc && b * f.nfc + col == bc);
        PMX_ASSERT(row0 + G <= p.N2 && L == p.N1);
        const unsigned char* aux = aux0 + (it & 1) * S::AUX_BYTES;
        const StepPkg* st = reinterpret_cast<const StepPkg*>(aux);
        const cpx* gtab = reinterpret_cast<const cpx*>(aux + S::PKG_BYTES);
        const int next = live(tile + gridDim.x);
        cpx x[8], y[8];
        PMX_T_MARK(0)
        pmx_mbar_wait(mbar, phase);
        phase ^= 1u;
        PMX_T_MARK(1)
#pragma unroll
        for (int q = 0; q < 8; ++q) lds_sa(in, pmx_swz<7>((uint32_t)((rl * L + t + q * T) * PMX_SA_BYTES)), x[q], y[q]);
        {   // Pass B left v = conj(z), z = its transform output before the four-step twiddle W_N^(-n2*k1), k1 = t + q*T.
            // The inverse transform over k1 = conj o forward o conj applied to conj(z)*conj(W): its input is z*W.
            const cpx* tb = gtab + rl * W::PER;
            const cpx wl = tb[t & (W::NLO - 1)];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const cpx w = cmul(wl, tb[W::NLO + ((t + q * T) >> W::LO)]);
                x[q] = cmul(cconj(x[q]), w);
                y[q] = cmul(cconj(y[q]), w);
            }
        }
        const real sc = (real)st->scale, nsc = -sc;
        __syncthreads();  // every thread has seen this phase complete before the barrier is armed again
        if (PF && threadIdx.x == 0 && next < total) issue(next, (it + 1) & 1);
        PMX_T_MARK(2)
        cpx* sx = work + rl * PmxSmem<L, G>::STRIDE;
        cpx* sy = sx + L;
        PMX_T_MARK(3)
        CtaFFT<R, L>::run(x, y, sx, sy, t, stw, [&] {
            if (!PF && threadIdx.x == 0 && next < total) issue(next, (it + 1) & 1);
        });
        PMX_T_MARK(4)
        {
            cpx* base = reinterpret_cast<cpx*>(p.field) + ((size_t)bc * N + (size_t)(row0 + rl) * L) * 2;
            if constexpr (NL) {
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    x[q] = mkc(x[q].x * sc, x[q].y * nsc);
                    y[q] = mkc(y[q].x * sc, y[q].y * nsc);
                }
                pmx_nl_step(x, y, st, f, col);   // ---- N(-xi*gam): the gam of f is the backpropagated one
#pragma unroll
                for (int q = 0; q < 8; ++q) st_sa(base + (size_t)(t + q * T) * 2, x[q], y[q]);
            } else {
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    x[q] = mkc(x[q].x * sc, x[q].y * nsc);
                    y[q] = mkc(y[q].x * sc, y[q].y * nsc);
                    unsigned long long key = pmx_pow_key((double)power_ref(x[q], y[q]));
                    vmax = key > vmax ? key : vmax;
                    st_sa(base + (size_t)(t + q * T) * 2, x[q], y[q]);
                }
            }
        }
        PMX_T_MARK(5)
        if constexpr (!NL) {
            if (next >= total || (wk.phys(next) >> wk.ltpb) != bc) {  // moving on: publish the maximum (pmx_k_ctl consumes it)
                pmx_block_max(vmax, sred, &p.ctl[b], col);
                vmax = 0ull;
            }
        }
        tile = next;
        ++it;
        __syncthreads();  // everyone is done with this tile's auxiliary buffer
        PMX_T_MARK(6)
    }
    PMX_T_FLUSH(NL ? 3 : 2)
}
