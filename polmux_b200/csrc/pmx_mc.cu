// Monte-Carlo BER over independent realizations on the GPUs of ONE node, behind the C ABI (pmx_mc_run).
//
// The reference runs realizations one after another in a `while cond` loop and feeds the integer error count of each
// block to ber_estimate (ex20_coherent_polmux.m:131-181, ber_estimate.m:118).  The realizations share nothing but the
// Tx field and the fiber, so they are the one axis the path shards on (SURVEY 8e): contiguous realization groups per
// GPU, one host thread and one pmx_ctx per GPU, no data-path collective.  Every GPU writes the counts of its own
// realizations straight into its slice of a zero-initialised [nreal] int64 device vector -- the NCCL send buffer --
// and ONE ncclAllReduce(sum) over NVLink leaves the complete vector everywhere (integer, hence order-independent and
// bit-exact).  Written against the public header only; NCCL is bound at run time (dlopen of libnccl.so.2: whichever
// copy the process already holds, e.g. PyTorch's), so the library has no link-time NCCL dependency.
#include <dlfcn.h>
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <future>
#include <string>
#include <thread>
#include <vector>

#include "../../include/polmux_ssfm.h"

namespace {
// the handful of NCCL entry points used, with the types of nccl.h (opaque comm, enums as int)
typedef struct ncclComm* ncclComm_t;
typedef int ncclResult_t;
struct Nccl {
    void* h = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool load() {
        if (h) return true;
        h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return false;
        CommInitAll = (decltype(CommInitAll))dlsym(h, "ncclCommInitAll");
        CommDestroy = (decltype(CommDestroy))dlsym(h, "ncclCommDestroy");
        AllReduce = (decltype(AllReduce))dlsym(h, "ncclAllReduce");
        GetErrorString = (decltype(GetErrorString))dlsym(h, "ncclGetErrorString");
        return CommInitAll && CommDestroy && AllReduce;
    }
};
Nccl g_nccl;
constexpr int NCCL_INT64 = 4, NCCL_SUM = 0;   // ncclInt64, ncclSum (nccl.h)

struct Worker {
    int rc = PMX_OK;
    std::string err;
    long long sa_steps = 0;
    int64_t* counts_dev = nullptr;
    pmx_ctx* ctx = nullptr;
};

#define MC_CK(call)                                                    \
    do {                                                               \
        int rc__ = (call);                                             \
        if (rc__ != PMX_OK) {                                          \
            w.rc = rc__;                                               \
            w.err = std::string(#call) + ": " + pmx_last_error(w.ctx); \
            goto done;                                                 \
        }                                                              \
    } while (0)

// realizations [r0, r1) on one device
void run_shard(Worker& w, int dev, int r0, int r1, const pmx_fiber_desc& fd, const pmx_mc_desc& m, const pmx_field& tx) {
    pmx_devfield *ftx = nullptr, *work = nullptr, *work2 = nullptr;
    pmx_plan *plan = nullptr, *inv = nullptr, *fo = nullptr, *fe = nullptr, *dbp = nullptr, *dbpl = nullptr;
    pmx_ctx* rxctx = nullptr;   // the receive chain's own context (stream): it runs beside the next group's propagation
    int64_t *tmp = nullptr, *tmp2 = nullptr;
    std::future<int> pending;
    std::string rxerr;
    const int B = m.batch, np = fd.nplates, nspan = m.nspan, nfc = fd.nfc;
    const size_t span_stride = (size_t)m.nreal * np;
    std::vector<double> pl[3], ipl[3], nb1, nb2, nbt, ndb1;
    std::vector<uint64_t> seeds(nspan);
    std::vector<int32_t> ncyc((size_t)nspan * B);
    for (auto& v : pl) v.resize((size_t)nspan * B * np);
    for (auto& v : ipl) v.resize((size_t)B * np);
    if (pmx_ctx_create(&w.ctx, dev) != PMX_OK) {
        w.rc = PMX_ERR_CUDA;
        w.err = std::string("pmx_ctx_create: ") + pmx_last_error(nullptr);
        return;
    }
    {
        cudaStream_t st = (cudaStream_t)pmx_ctx_stream(w.ctx);
        if (cudaMalloc(&w.counts_dev, (size_t)m.nreal * sizeof(int64_t)) != cudaSuccess ||
            cudaMalloc(&tmp, (size_t)B * sizeof(int64_t)) != cudaSuccess ||
            cudaMemsetAsync(w.counts_dev, 0, (size_t)m.nreal * sizeof(int64_t), st) != cudaSuccess) {
            w.rc = PMX_ERR_CUDA;
            w.err = "count buffers: out of device memory";
            goto done;
        }
        MC_CK(pmx_field_create(w.ctx, fd.nfft, nfc, 1, fd.precision, &ftx));
        MC_CK(pmx_field_upload(ftx, &tx, 0, 1));
        MC_CK(pmx_field_create(w.ctx, fd.nfft, nfc, B, fd.precision, &work));
        // plates of a group: [span][b][plate] gathered from the caller's [span][realization][plate]
        auto gather = [&](int g0) {
            const double* src[3] = {m.db0, m.theta, m.epsilon};
            for (int k = 0; k < nspan; ++k)
                for (int b = 0; b < B; ++b) {
                    const int r = std::min(g0 + b, m.nreal - 1);   // (slots past the last realization repeat it; not counted)
                    for (int i = 0; i < 3; ++i)
                        memcpy(&pl[i][((size_t)k * B + b) * np], src[i] + (size_t)k * span_stride + (size_t)r * np,
                               (size_t)np * sizeof(double));
                }
        };
        gather(r0);
        pmx_fiber_desc d = fd;
        d.batch = B;
        d.plate_sets = B;
        d.db0 = pl[0].data();
        d.theta = pl[1].data();
        d.epsilon = pl[2].data();
        MC_CK(pmx_plan_create(w.ctx, &d, &plan));
        if (m.dbp && !m.rx) {   // PMD-aware DBP with the group's plates in place of the equaliser
            const int rc = pmx_dbp_create(w.ctx, &d, m.dbp, &dbpl);
            if (rc != PMX_OK) {
                w.rc = rc;
                w.err = std::string("pmx_dbp_create: ") + pmx_last_error(w.ctx);
                goto done;
            }
        } else if (m.equalize) {   // one linear single-step fiber per span with the plate order reversed and every phase negated
            pmx_fiber_desc e = d;
            e.fls[2] = e.fls[3] = 0;
            e.dphimaxt = INFINITY;
            e.dzmaxt = e.length;
            e.alphalin = 0.0;
            e.manakov = 0;
            e.precision = PMX_F64;
            if (e.disp_mode == PMX_DISP_SCALAR) {
                nb1.assign(fd.beta1, fd.beta1 + nfc);
                nb2.assign(fd.beta2, fd.beta2 + nfc);
                for (auto& v : nb1) v = -v;
                for (auto& v : nb2) v = -v;
                e.beta1 = nb1.data();
                e.beta2 = nb2.data();
                e.b30 = -fd.b30;
                e.dgdrms = -fd.dgdrms;
            } else {
                nbt.assign(fd.betat, fd.betat + (size_t)nfc * fd.nfft);
                for (auto& v : nbt) v = -v;
                e.betat = nbt.data();
                if (fd.db1) {
                    ndb1.assign(fd.db1, fd.db1 + (size_t)nfc * fd.nfft);
                    for (auto& v : ndb1) v = -v;
                    e.db1 = ndb1.data();
                }
            }
            if (fd.precision != PMX_F64) {
                w.rc = PMX_ERR_UNSUPPORTED;
                w.err = "the equaliser and the error counter take FP64 fields";
                goto done;
            }
            MC_CK(pmx_plan_create(w.ctx, &e, &inv));
        }
        if (m.rx) {   // the receive chain's two filter plans (receiver_cohmix.m:169,293), for the resident batch
            if (nfc != 1 || fd.precision != PMX_F64 || !m.rx->hf_opt || !m.rx->hf_el || !m.rx->ref_patmat) {
                w.rc = PMX_ERR_UNSUPPORTED;
                w.err = "the receive chain takes single-column FP64 fields, both filter responses and the reference pattern";
                goto done;
            }
            if (pmx_ctx_create(&rxctx, dev) != PMX_OK) {
                w.rc = PMX_ERR_CUDA;
                w.err = std::string("pmx_ctx_create (receive chain): ") + pmx_last_error(nullptr);
                goto done;
            }
            MC_CK(pmx_field_create(w.ctx, fd.nfft, nfc, B, fd.precision, &work2));
            if (cudaMalloc(&tmp2, (size_t)B * sizeof(int64_t)) != cudaSuccess) {
                w.rc = PMX_ERR_CUDA;
                w.err = "count buffers: out of device memory";
                goto done;
            }
            if (pmx_filter_create(rxctx, fd.nfft, 1, B, PMX_F64, m.rx->hf_opt, 1, &fo) != PMX_OK) {
                w.rc = PMX_ERR_CUDA;
                w.err = std::string("pmx_filter_create: ") + pmx_last_error(rxctx);
                goto done;
            }
            std::vector<double> hh(2 * (size_t)fd.nfft);   // Hermitian part: two real currents on one complex transform
            const size_t N = (size_t)fd.nfft;
            for (size_t k = 0; k < N; ++k) {
                const size_t mk = (N - k) & (N - 1);
                hh[2 * k] = 0.5 * (m.rx->hf_el[2 * k] + m.rx->hf_el[2 * mk]);
                hh[2 * k + 1] = 0.5 * (m.rx->hf_el[2 * k + 1] - m.rx->hf_el[2 * mk + 1]);
            }
            if (pmx_filter_create(rxctx, fd.nfft, 1, B, PMX_F64, hh.data(), 1, &fe) != PMX_OK) {
                w.rc = PMX_ERR_CUDA;
                w.err = std::string("pmx_filter_create: ") + pmx_last_error(rxctx);
                goto done;
            }
            if (m.rx->dbp) {   // digital backpropagation of the link, first thing of the receive chain
                const int rc = pmx_dbp_create(rxctx, &d, m.rx->dbp, &dbp);
                if (rc != PMX_OK) {
                    w.rc = rc;
                    w.err = std::string("pmx_dbp_create: ") + pmx_last_error(rxctx);
                    goto done;
                }
            }
        }
        for (int g0 = r0, gi = 0; g0 < r1; g0 += B, ++gi) {
            const int nb = std::min(B, r1 - g0);
            pmx_devfield* const cur = (m.rx && (gi & 1)) ? work2 : work;   // two work fields alternate under the receive chain
            int64_t* const ctmp = (m.rx && (gi & 1)) ? tmp2 : tmp;
            if (g0 != r0) gather(g0);
            MC_CK(pmx_field_broadcast(cur, ftx));
            for (int k = 0; k < nspan; ++k)   // the seed convention of polmux_b200.mc.Link.ase_seed
                seeds[k] = ((m.ase_seed & 0xffffffull) << 40) + ((uint64_t)k << 32);
            pmx_link_desc l;
            memset(&l, 0, sizeof l);
            l.nspan = nspan;
            l.plate_sets = B;
            l.db0 = pl[0].data();
            l.theta = pl[1].data();
            l.epsilon = pl[2].data();
            l.gain = m.gain;
            l.sigma = m.sigma;
            l.seeds = seeds.data();
            l.realization0 = (uint64_t)g0;   // the ASE of a realization does not depend on its group
            pmx_fiber_result res;
            memset(&res, 0, sizeof res);
            res.ncycle = ncyc.data();
            MC_CK(pmx_link_exec(plan, cur, &l, &res));
            for (int k = 0; k < nspan; ++k)
                for (int b = 0; b < nb; ++b) w.sa_steps += (long long)ncyc[(size_t)k * B + b] * fd.nfft * nfc;
            if (dbpl) {
                MC_CK(pmx_dbp_set_plates(dbpl, B, pl[0].data(), pl[1].data(), pl[2].data()));
                MC_CK(pmx_dbp_exec(dbpl, cur));
            }
            if (inv) {
                for (int k = nspan - 1; k >= 0; --k) {
                    for (int b = 0; b < B; ++b)
                        for (int n = 0; n < np; ++n) {
                            const size_t s = ((size_t)k * B + b) * np + (np - 1 - n), t = (size_t)b * np + n;
                            ipl[0][t] = -pl[0][s];
                            ipl[1][t] = pl[1][s];
                            ipl[2][t] = pl[2][s];
                        }
                    MC_CK(pmx_plan_set_plates(inv, B, ipl[0].data(), ipl[1].data(), ipl[2].data()));
                    MC_CK(pmx_fiber_exec(inv, cur, nullptr));
                }
            }
            // the error counter writes the group's counts; they land in this rank's slice of the NCCL send buffer
            if (m.rx) {
                // the previous group's chain ran beside this group's link; now this group's chain starts beside the next link
                if (pending.valid() && pending.get() != PMX_OK) {
                    w.rc = PMX_ERR_CUDA;
                    w.err = rxerr;
                    goto done;
                }
                if (dbp && m.rx->dbp->pmd) {   // this group's plates, before the next gather() overwrites pl
                    const int rc = pmx_dbp_set_plates(dbp, B, pl[0].data(), pl[1].data(), pl[2].data());
                    if (rc != PMX_OK) {
                        w.rc = rc;
                        w.err = std::string("pmx_dbp_set_plates: ") + pmx_last_error(rxctx);
                        goto done;
                    }
                }
                int64_t* const dst = w.counts_dev + g0;
                pending = std::async(std::launch::async, [=, &m, &rxerr]() -> int {
                    int rc = dbp ? pmx_dbp_exec(dbp, cur) : PMX_OK;
                    if (rc == PMX_OK) rc = pmx_fiber_exec(fo, cur, nullptr);
                    if (rc == PMX_OK) rc = pmx_cohmix_exec(rxctx, cur, m.rx->lo_ecw, m.rx->lo_detune, m.rx->lo_phase, m.rx->balanced);
                    if (rc == PMX_OK) rc = pmx_fiber_exec(fe, cur, nullptr);
                    if (rc == PMX_OK) rc = pmx_dsp_count(rxctx, cur, &m.rx->dsp, m.rx->ref_patmat, ctmp, nullptr);
                    if (rc == PMX_OK) {
                        cudaStream_t rs = (cudaStream_t)pmx_ctx_stream(rxctx);
                        if (cudaMemcpyAsync(dst, ctmp, (size_t)nb * sizeof(int64_t), cudaMemcpyDeviceToDevice, rs) != cudaSuccess ||
                            cudaStreamSynchronize(rs) != cudaSuccess) {
                            rxerr = "count copy failed";
                            return PMX_ERR_CUDA;
                        }
                    } else {
                        rxerr = std::string("receive chain: ") + pmx_last_error(rxctx);
                    }
                    return rc;
                });
                continue;
            }
            // the error counter writes the group's counts; they land in this rank's slice of the NCCL send buffer
            MC_CK(pmx_qpsk_count(w.ctx, cur, m.sym, m.nsymb, m.nt, ctmp));
            if (cudaMemcpyAsync(w.counts_dev + g0, ctmp, (size_t)nb * sizeof(int64_t), cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
                w.rc = PMX_ERR_CUDA;
                w.err = "count copy failed";
                goto done;
            }
        }
        if (pending.valid() && pending.get() != PMX_OK) {
            w.rc = PMX_ERR_CUDA;
            w.err = rxerr;
            goto done;
        }
        MC_CK(pmx_ctx_sync(w.ctx));
    }
done:
    if (pending.valid()) pending.wait();   // (an error path: the chain must not outlive its buffers)
    if (tmp) cudaFree(tmp);
    if (tmp2) cudaFree(tmp2);
    pmx_plan_destroy(fo);
    pmx_plan_destroy(fe);
    pmx_plan_destroy(dbp);
    pmx_plan_destroy(dbpl);
    pmx_plan_destroy(inv);
    pmx_plan_destroy(plan);
    pmx_field_destroy(work);
    pmx_field_destroy(work2);
    pmx_field_destroy(ftx);
    if (rxctx) pmx_ctx_destroy(rxctx);
}
}  // namespace

extern "C" int pmx_mc_run(const pmx_fiber_desc* fiber, const pmx_mc_desc* mc, const pmx_field* tx, int64_t* counts,
                          int64_t* sa_steps, char* errbuf, int32_t errlen) {
    auto fail = [&](int code, const std::string& msg) {
        if (errbuf && errlen > 0) {
            strncpy(errbuf, msg.c_str(), (size_t)errlen - 1);
            errbuf[errlen - 1] = 0;
        }
        return code;
    };
    if (!fiber || !mc || !tx || !counts) return fail(PMX_ERR_INVALID, "pmx_mc_run: null argument");
    if (mc->ndev < 1 || mc->nreal < 1 || mc->batch < 1 || mc->nspan < 1 || !mc->device_ids || !mc->sym)
        return fail(PMX_ERR_INVALID, "pmx_mc_run: ndev, nreal, batch, nspan must be >= 1; device_ids and sym are required");
    if (fiber->fls[1] && (!mc->db0 || !mc->theta || !mc->epsilon))
        return fail(PMX_ERR_INVALID, "pmx_mc_run: plate draws [nspan][nreal][nplates] are required with the 'p' flag");
    if (mc->dbp && !mc->rx && !mc->dbp->pmd)
        return fail(PMX_ERR_INVALID, "pmx_mc_run: dbp without a receive chain must be PMD-aware (pmd = 1): the data-aided "
                                     "decision needs the PMD undone");
    if ((mc->dbp && mc->dbp->pmd && !mc->rx) || (mc->rx && mc->rx->dbp && mc->rx->dbp->pmd))
        if (!fiber->fls[1]) return fail(PMX_ERR_INVALID, "pmx_mc_run: PMD-aware DBP needs the fiber's 'p' flag");
    const int ndev = mc->ndev;
    const bool have_nccl = g_nccl.load();
    if (ndev > 1 && !have_nccl) return fail(PMX_ERR_UNSUPPORTED, "pmx_mc_run: libnccl.so.2 not found (needed for more than one GPU)");
    std::vector<ncclComm_t> comms(ndev, nullptr);
    if (have_nccl) {
        ncclResult_t r = g_nccl.CommInitAll(comms.data(), ndev, mc->device_ids);
        if (r != 0) return fail(PMX_ERR_CUDA, std::string("ncclCommInitAll: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "failed"));
    }
    std::vector<Worker> ws(ndev);
    {
        std::vector<std::thread> th;
        for (int g = 0; g < ndev; ++g) {
            const int r0 = (int)((long long)g * mc->nreal / ndev), r1 = (int)((long long)(g + 1) * mc->nreal / ndev);
            th.emplace_back([&, g, r0, r1] { run_shard(ws[g], mc->device_ids[g], r0, r1, *fiber, *mc, *tx); });
        }
        for (auto& t : th) t.join();
    }
    int rc = PMX_OK;
    std::string msg;
    for (int g = 0; g < ndev; ++g)
        if (ws[g].rc != PMX_OK && rc == PMX_OK) {
            rc = ws[g].rc;
            msg = "GPU " + std::to_string(mc->device_ids[g]) + ": " + ws[g].err;
        }
    if (rc == PMX_OK && have_nccl) {   // one all-reduce of the zero-padded count vector (all ranks enqueue, then wait)
        for (int g = 0; g < ndev && rc == PMX_OK; ++g) {
            cudaSetDevice(mc->device_ids[g]);
            // ncclGroupStart/End are not needed: every rank's call is issued from its own thread below
        }
        std::vector<std::thread> th;
        std::vector<int> nr(ndev, 0);
        for (int g = 0; g < ndev; ++g)
            th.emplace_back([&, g] {
                cudaSetDevice(mc->device_ids[g]);
                cudaStream_t st = (cudaStream_t)pmx_ctx_stream(ws[g].ctx);
                nr[g] = g_nccl.AllReduce(ws[g].counts_dev, ws[g].counts_dev, (size_t)mc->nreal, NCCL_INT64, NCCL_SUM, comms[g], st);
                if (nr[g] == 0 && cudaStreamSynchronize(st) != cudaSuccess) nr[g] = -1;
            });
        for (auto& t : th) t.join();
        for (int g = 0; g < ndev; ++g)
            if (nr[g] != 0 && rc == PMX_OK) {
                rc = PMX_ERR_CUDA;
                msg = "ncclAllReduce failed on GPU " + std::to_string(mc->device_ids[g]);
            }
    }
    if (rc == PMX_OK) {
        cudaSetDevice(mc->device_ids[0]);
        if (cudaMemcpy(counts, ws[0].counts_dev, (size_t)mc->nreal * sizeof(int64_t), cudaMemcpyDeviceToHost) != cudaSuccess) {
            rc = PMX_ERR_CUDA;
            msg = "count read-back failed";
        }
        long long total = 0;
        for (auto& w : ws) total += w.sa_steps;
        if (sa_steps) *sa_steps = total;
    }
    for (int g = 0; g < ndev; ++g) {
        cudaSetDevice(mc->device_ids[g]);
        if (ws[g].counts_dev) cudaFree(ws[g].counts_dev);
        if (comms[g]) g_nccl.CommDestroy(comms[g]);
        pmx_ctx_destroy(ws[g].ctx);
    }
    return rc == PMX_OK ? PMX_OK : fail(rc, msg);
}

extern "C" int pmx_mc_nccl_available(void) { return g_nccl.load() ? 1 : 0; }
