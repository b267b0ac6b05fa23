// Per-L launch table: one translation unit per in-CTA FFT length (pmx_passes_inst.cu
// compiled with -DPMX_L=<L>) exports its three pass launchers through this struct.
#pragma once
#include <cuda.h>
#include "pmx_common.cuh"

struct PmxLaunchTable {
    int L;
    int gAC;       // columns per tile in passes A / C
    int gB;        // rows per tile in pass B
    int pfAC, pfB; // 1: next tile prefetched into its own landing buffer
    int threadsAC, threadsB;
    size_t smemAC, smemB;
    int tw_total;  // cpx entries of the stage-twiddle table for this L
    int tw_layout; // 0: first stage 2/4/8 then radix-8 stages; 1: L = 1024 as 8 * 16 * 8 (pmx_fft.cuh)
    int tw4_lo_bits, tw4_per;  // four-step twiddle row layout (PmxTw4<L>)
    int precision;             // 0 = FP64, 1 = FP32 (pmx_precision)
    int cpx_bytes;             // sizeof one complex number of that precision
    // opt in to the dynamic shared memory, report resident CTAs per SM of each kernel (ctasCnl: passC_nl)
    cudaError_t (*setup)(int* ctasA, int* ctasB, int* ctasC, int* ctasCnl);
    // grid_x persistent CTAs
    // (every launcher returns the launch status)
    cudaError_t (*passA)(int grid_x, cudaStream_t s, const PassParams& p, const FiberConst& f, const CUtensorMap& cols);
    cudaError_t (*passB)(int grid_x, cudaStream_t s, const PassParams& p, const FiberConst& f, const CUtensorMap& rows);
    cudaError_t (*passC)(int grid_x, cudaStream_t s, const PassParams& p, const FiberConst& f, const CUtensorMap& cols);
    // first max |u|^2 of a resident field (pmx_k_init) and the four-step twiddle rows, in this precision
    void (*init_max)(dim3 grid, cudaStream_t s, const PassParams& p, const FiberConst& f);
    void (*fill_tw4)(void* tab, int rows, double two_over_N, cudaStream_t s);
    // scalar XPM: sum over the columns of |u|^2 per sample, written to the Y slot of every column (grid.y = realizations)
    void (*xpm_sum)(dim3 grid, cudaStream_t s, const PassParams& p, const FiberConst& f);
    // small fields (nfft == L <= 4096): the whole fiber in one launch, one CTA per realization-column, the nfc CTAs of a
    // realization in one thread-block cluster (pmx_onchip.cuh)
    size_t smemOnchip;
    cudaError_t (*onchip_setup)();
    cudaError_t (*onchip)(int nfc, int batch, cudaStream_t s, const PassParams& p, const FiberConst& f);
    // digital backpropagation: pass C with the nonlinear step after the scale and no max reduction (pmx_k_passC<..., true>)
    cudaError_t (*passC_nl)(int grid_x, cudaStream_t s, const PassParams& p, const FiberConst& f, const CUtensorMap& cols);
    // digital backpropagation of a small field: the on-chip kernel walking the plan's step table (pmx_k_onchip<..., true>),
    // launched like onchip (set up by onchip_setup)
    cudaError_t (*onchip_dbp)(int nfc, int batch, cudaStream_t s, const PassParams& p, const FiberConst& f, const DbpSteps& ds);
    // filtered DBP (pmx_dbp_set_filter): the on-chip kernel with the Gaussian response (pmx_k_onchip<..., DbpFiltSteps>), and
    // on the three passes the intensity into the work field and the nonlinear step from the filtered one (grid.y = batch*nfc)
    cudaError_t (*onchip_dbp_filt)(int nfc, int batch, cudaStream_t s, const PassParams& p, const FiberConst& f,
                                   const DbpFiltSteps& ds);
    void (*dbp_intensity)(dim3 grid, cudaStream_t s, const PassParams& p, const FiberConst& f, void* work);
    void (*dbp_nl_filt)(dim3 grid, cudaStream_t s, const PassParams& p, const FiberConst& f, const void* work, const StepPkg* pkg);
    // enhanced split-step DBP (pmx_dbp_set_taps): the on-chip kernel with the taps (pmx_k_onchip<..., DbpTapSteps>), and on
    // the three passes the nonlinear step from the FIR of dbp_intensity's work field (pmx_k_dbp_nl_fir, its own grid)
    cudaError_t (*onchip_dbp_taps)(int nfc, int batch, cudaStream_t s, const PassParams& p, const FiberConst& f,
                                   const DbpTapSteps& ds);
    cudaError_t (*dbp_nl_fir)(cudaStream_t s, const PassParams& p, const FiberConst& f, const void* work, const StepPkg* pkg,
                              const DbpTaps& taps);
};

const PmxLaunchTable* pmx_get_table(int L, int precision = 0);  // nullptr if L is not built

// Host: fill the stage-twiddle table of length L (layout documented in pmx_fft.cuh).
void pmx_fill_stage_twiddles(int L, cpx* out, int layout);
