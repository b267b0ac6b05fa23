// Instantiates the pass kernels for one in-CTA FFT length (-DPMX_L=<L>) in one precision
// (FP64, or FP32 with -DPMX_F32) and exports their launchers through a PmxLaunchTable.
#include "pmx_kernels.cuh"
#include "pmx_onchip.cuh"
#include "pmx_launch.h"

#ifndef PMX_L
#error "compile with -DPMX_L=<fft length>"
#endif

namespace {
constexpr int L = PMX_L;
// Tile shapes.  Rows/columns per tile are chosen so that a tile is <= 32 KiB when possible (1024 Sa in FP64,
// 2048 Sa in FP32: the FP32 tiles have twice the rows/columns, i.e. the same bytes and the same TMA box rows):
// landing buffer + exchange buffer then fit three CTAs per SM with the next tile prefetched.  Longer
// transforms land in the exchange buffer itself (no separate prefetch).
constexpr int PSCALE = 32 / PMX_SA_BYTES;  // 1 (FP64) or 2 (FP32)
constexpr int GAC = PSCALE * ((L >= 1024) ? 1 : (L == 512 ? 2 : 4));
constexpr int GB_ROWS = (PSCALE * ((L >= 1024) ? 1 : (L == 512 ? 2 : 4)) * (L / 8) > 1024) ? 1 : PSCALE * ((L >= 1024) ? 1 : (L == 512 ? 2 : 4));
constexpr int TILE_CAP = 32 * 1024;
// ... unless pass B would then need more shared memory than a CTA can have (227 KiB): FP32 at L = 4096 takes one column
// per tile (as FP64 does), since two would need 251 KB and the kernel could not be launched at all.
constexpr int GB = (PassSmem<L, GB_ROWS, (GB_ROWS * L * PMX_SA_BYTES <= TILE_CAP / 2), 1>::TOTAL > 227 * 1024) ? 1 : GB_ROWS;
// Since passes A and C read and write contiguous rows straight from / to registers they no longer stage a
// tile for a TMA store, and a fourth resident CTA (the tile lands in the exchange buffer, 42 KB per CTA) beats a
// separate prefetch buffer with three (measured 49.0 against 50.3 ps per Sa and step at N = 2^20).
constexpr bool PFAC = false;
// pass B is compute-bound: it prefers a fourth resident CTA to a separate prefetch buffer
constexpr bool PFB = (GB * L * PMX_SA_BYTES <= TILE_CAP / 2);
static_assert(GAC * (L / 8) <= 1024 && GB * (L / 8) <= 1024, "CTA too large");
using SA = PassSmem<L, GAC, PFAC, 0>;
using SB = PassSmem<L, GB, PFB, 1>;
using SC = PassSmem<L, GAC, PFAC, 2>;

cudaError_t setup(int* ctasA, int* ctasB, int* ctasC, int* ctasCnl) {
    cudaError_t e;
    auto prep = [](auto kern, int smem, int threads, int* ctas) -> cudaError_t {
        cudaError_t r = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (r != cudaSuccess) return r;
        cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas, kern, threads, smem);
    };
    e = prep(pmx_k_passA<real, L, GAC, PFAC>, SA::TOTAL, SA::THREADS, ctasA);
    if (e != cudaSuccess) return e;
    {
        int dummy = 0;
        e = prep(pmx_k_passA<real, L, GAC, PFAC, true>, ((SA::TOTAL + 15) / 16) * 16 + PMX_FUSED_BYTES, SA::THREADS, &dummy);
        if (e != cudaSuccess) return e;
    }
    e = prep(pmx_k_passB<real, L, GB, PFB, false>, SB::TOTAL, SB::THREADS, ctasB);
    if (e != cudaSuccess) return e;
    e = prep(pmx_k_passB<real, L, GB, PFB, true>, SB::TOTAL, SB::THREADS, ctasB);
    if (e != cudaSuccess) return e;
    e = prep(pmx_k_passC<real, L, GAC, PFAC, false>, SC::TOTAL, SC::THREADS, ctasC);
    if (e != cudaSuccess) return e;
    return prep(pmx_k_passC<real, L, GAC, PFAC, true>, SC::TOTAL, SC::THREADS, ctasCnl);
}
// p.pdl: launch with programmatic stream serialization (the kernel's prologue then overlaps the previous kernel's tail)
template <typename K>
cudaError_t launch(K kern, int gx, int threads, int smem, cudaStream_t s, const PassParams& p, const FiberConst& f, const CUtensorMap& m) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(gx);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = p.pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, p, f, m);
}
cudaError_t passA(int gx, cudaStream_t s, const PassParams& p, const FiberConst& f, const CUtensorMap& m) {
    if (p.ctl_out)   // fused step control (a batch of one)
        return launch(pmx_k_passA<real, L, GAC, PFAC, true>, gx, SA::THREADS, ((SA::TOTAL + 15) / 16) * 16 + PMX_FUSED_BYTES, s, p, f, m);
    return launch(pmx_k_passA<real, L, GAC, PFAC>, gx, SA::THREADS, SA::TOTAL, s, p, f, m);
}
cudaError_t passB(int gx, cudaStream_t s, const PassParams& p, const FiberConst& f, const CUtensorMap& m) {
    if (f.disp_scalar)
        return launch(pmx_k_passB<real, L, GB, PFB, true>, gx, SB::THREADS, SB::TOTAL, s, p, f, m);
    return launch(pmx_k_passB<real, L, GB, PFB, false>, gx, SB::THREADS, SB::TOTAL, s, p, f, m);
}
cudaError_t passC(int gx, cudaStream_t s, const PassParams& p, const FiberConst& f, const CUtensorMap& m) {
    return launch(pmx_k_passC<real, L, GAC, PFAC, false>, gx, SC::THREADS, SC::TOTAL, s, p, f, m);
}
cudaError_t passC_nl(int gx, cudaStream_t s, const PassParams& p, const FiberConst& f, const CUtensorMap& m) {
    return launch(pmx_k_passC<real, L, GAC, PFAC, true>, gx, SC::THREADS, SC::TOTAL, s, p, f, m);
}
// precision-dependent helpers that do not depend on L (every table carries them)
void init_max(dim3 grid, cudaStream_t s, const PassParams& p, const FiberConst& f) {
    pmx_k_init<<<grid, 256, 256, s>>>(p, f);
}
void xpm_sum(dim3 grid, cudaStream_t s, const PassParams& p, const FiberConst& f) { pmx_k_xpm_sum<<<grid, 256, 0, s>>>(p, f); }
void fill_tw4(void* tab, int rows, double two_over_N, cudaStream_t s) {
    const size_t n = (size_t)rows * PmxTw4<L>::PER;
    const int blocks = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
    pmx_k_fill_tw4<<<blocks, 256, 0, s>>>(reinterpret_cast<cpx*>(tab), rows, PmxTw4<L>::LO, PmxTw4<L>::PER, PmxTw4<L>::PER,
                                          two_over_N);
}
// ---- single-CTA kernel of small fields
using SO = OnchipSmem<L>;
constexpr int ONCHIP_THREADS = (L / 8) < 32 ? 32 : (L / 8);
cudaError_t onchip_setup() {
    cudaError_t e = cudaFuncSetAttribute(pmx_k_onchip<real, L, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SO::TOTAL);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(pmx_k_onchip<real, L, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SO::TOTAL);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(pmx_k_onchip<real, L, true, true, DbpSteps>, cudaFuncAttributeMaxDynamicSharedMemorySize, SO::TOTAL);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(pmx_k_onchip<real, L, false, true, DbpSteps>, cudaFuncAttributeMaxDynamicSharedMemorySize, SO::TOTAL);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(pmx_k_onchip<real, L, true, true, DbpFiltSteps>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             SO::TOTAL);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(pmx_k_onchip<real, L, false, true, DbpFiltSteps>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             SO::TOTAL);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(pmx_k_onchip<real, L, true, true, DbpTapSteps>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             SO::TOTAL);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(pmx_k_onchip<real, L, false, true, DbpTapSteps>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                SO::TOTAL);
}
// the forward run (no step table) or digital backpropagation (one DbpSteps)
template <bool DBP, typename... Steps>
cudaError_t onchip_launch(int nfc, int batch, cudaStream_t s, const PassParams& p, const FiberConst& f, const Steps&... steps) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(nfc, batch);
    cfg.blockDim = dim3(ONCHIP_THREADS);
    cfg.dynamicSmemBytes = SO::TOTAL;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;   // the columns of a realization exchange maxima / powers through DSMEM
    at[0].val.clusterDim.x = nfc;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = nfc > 1 ? 1 : 0;
    if (f.disp_scalar) return cudaLaunchKernelEx(&cfg, pmx_k_onchip<real, L, true, DBP, Steps...>, p, f, steps...);
    return cudaLaunchKernelEx(&cfg, pmx_k_onchip<real, L, false, DBP, Steps...>, p, f, steps...);
}
cudaError_t onchip(int nfc, int batch, cudaStream_t s, const PassParams& p, const FiberConst& f) {
    return onchip_launch<false>(nfc, batch, s, p, f);
}
cudaError_t onchip_dbp(int nfc, int batch, cudaStream_t s, const PassParams& p, const FiberConst& f, const DbpSteps& ds) {
    return onchip_launch<true>(nfc, batch, s, p, f, ds);
}
cudaError_t onchip_dbp_filt(int nfc, int batch, cudaStream_t s, const PassParams& p, const FiberConst& f, const DbpFiltSteps& ds) {
    return onchip_launch<true>(nfc, batch, s, p, f, ds);
}
// filtered DBP on the three passes: the pointwise kernels around the filter plan (grid.y = batch * nfc)
void dbp_intensity(dim3 grid, cudaStream_t s, const PassParams& p, const FiberConst& f, void* work) {
    pmx_k_dbp_intensity<<<grid, 256, 0, s>>>(p, f, reinterpret_cast<cpx*>(work));
}
void dbp_nl_filt(dim3 grid, cudaStream_t s, const PassParams& p, const FiberConst& f, const void* work, const StepPkg* pkg) {
    pmx_k_dbp_nl_filt<<<grid, 256, 0, s>>>(p, f, reinterpret_cast<const cpx*>(work), pkg);
}
// enhanced split-step DBP: the taps on the M-sample grid of a single-launch plan, and on the three passes the nonlinear
// step from the FIR of the intensity in the work field (one CTA per tile of rows and work column)
cudaError_t onchip_dbp_taps(int nfc, int batch, cudaStream_t s, const PassParams& p, const FiberConst& f, const DbpTapSteps& ds) {
    return onchip_launch<true>(nfc, batch, s, p, f, ds);
}
cudaError_t dbp_nl_fir(cudaStream_t s, const PassParams& p, const FiberConst& f, const void* work, const StepPkg* pkg,
                       const DbpTaps& taps) {
    const int smem = (PMX_FIR_ROWS + 2 * taps.k) * PMX_FIR_COLS * 2 * (int)sizeof(cpx);
    cudaError_t e = cudaFuncSetAttribute(pmx_k_dbp_nl_fir, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    const dim3 grid((unsigned)((p.N1 / PMX_FIR_COLS) * (p.N2 / PMX_FIR_ROWS)), (unsigned)((p.batch * f.nfc + 1) / 2));
    pmx_k_dbp_nl_fir<<<grid, 256, smem, s>>>(p, f, reinterpret_cast<const cpx*>(work), pkg, taps);
    return cudaGetLastError();
}
}  // namespace

#define PMX_CAT2(a, b) a##b
#define PMX_CAT(a, b) PMX_CAT2(a, b)
#ifdef PMX_F32
#define PMX_TABLE_NAME PMX_CAT(pmx_table_f32_, PMX_L)
#else
#define PMX_TABLE_NAME PMX_CAT(pmx_table_, PMX_L)
#endif
extern const PmxLaunchTable PMX_TABLE_NAME = {
    L, GAC, GB, PFAC ? 1 : 0, PFB ? 1 : 0, SA::THREADS, SB::THREADS, (size_t)SA::TOTAL, (size_t)SB::TOTAL,
    pmx_tw_total(L), pmx_tw_layout(L), PmxTw4<L>::LO, PmxTw4<L>::PER, PMX_PRECISION, (int)sizeof(cpx),
    setup, passA, passB, passC, init_max, fill_tw4, xpm_sum, (size_t)SO::TOTAL, onchip_setup, onchip, passC_nl, onchip_dbp,
    onchip_dbp_filt, dbp_intensity, dbp_nl_filt, onchip_dbp_taps, dbp_nl_fir};
