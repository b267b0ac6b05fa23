/*
 * ssfm_mex.c -- MEX gateway to the B200 split-step Fourier library (libpolmux_ssfm.so).
 *
 * Written in the style of the reference's own gateways (fastexp.c:46-68,
 * cmaadaptivefilter.c:93-174): split real/imaginary storage through mxGetPr/mxGetPi, outputs
 * from mxCreateDoubleMatrix, failures through mexErrMsgTxt, no toolbox / gpuArray dependency.
 *
 * It replaces the body of matrix_ssfm (fiber.m:459-555) and takes that function's argument
 * list, with the three brf vectors passed separately:
 *
 *   [ux,uy,firstdz,ncycle] = ssfm_mex(ux,uy,betat,db1,dzmaxt,dphimaxt,gam,alphalin, ...
 *                                     nfc,Lf,nplates,manakov,fls,db0,theta,epsilon[,scal])
 *
 *   ux, uy     Nfft x nfc complex (uy may be real or empty -> zeros, fiber.m:286)
 *   betat,db1  Nfft x nfc real                        (fiber.m:350-362)
 *   gam        1 x nfc (or scalar) [1/mW/m], before the Manakov 8/9
 *   manakov    logical / 0-1 scalar: strcmp(x.manakov,'yes')
 *   fls        1 x 4 flag vector                      (fiber.m:157)
 *   db0,theta,epsilon   nplates x 1                   (brf.*, fiber.m:266-276)
 *   scal       optional [symbolrate nsymb nt b30 dgdrms beta1(1:nfc) beta2(1:nfc)]: the library
 *              regenerates betat/db1 on the device and the two vectors are not uploaded ([] to skip)
 *
 * Span loop in one call (the loop  for k=1:Nspan, fiber(x,flag); ampliflat(G,'gain',opt); end  of
 * ex06_ber.m:110-115; the field crosses PCIe once in and once out, pmx_link_run):
 *
 *   [ux,uy,firstdz,ncycle] = ssfm_mex(..., db0,theta,epsilon, scal, amp)
 *
 *   db0,theta,epsilon   nplates x Nspan: column k holds the waveplates fiber.m:274-276 draws for span k
 *   amp        [gain sigma(1:nfc) seed]: linear power gain 10^(G/10) of the amplifier after every span
 *              (ampliflat.m:62), ASE sigma per column (ampliflat.m:91-106, 0 = noiseless) and the seed of the
 *              device noise generator (span k uses seed+k-1); [] or absent: fibers only
 *   firstdz    first step of span 1;  ncycle  1 x Nspan
 *
 * Command interface (what matlab/fiber.m and matlab/ampliflat.m call; the first argument is a string):
 *
 *   [ux,uy,firstdz,ncycle] = ssfm_mex('fiber', ux, uy, betat, db1, P, gam, fls, plates, scal, opt)
 *       P      [dzmaxt dphimaxt alphalin Lf nplates manakov]        (matrix_ssfm's scalars, fiber.m:459-460)
 *       plates nplates x 3  [db0 theta epsilon]                      (brf.*, fiber.m:266-276); [] without the 'p' flag
 *       scal   [] or [symbolrate nsymb nt b30 dgdrms beta1(1:nfc) beta2(1:nfc)] (betat / db1 may then be [])
 *       opt    [scalar_field precision resident tolflag ltol safety], trailing entries optional:
 *              scalar_field 1 = the scalar_ssfm / scalar_a_ssfm dispatches (fiber.m:372-380,386-387; uy = [] in and out)
 *              precision    0 = FP64, 1 = FP32 arithmetic on the device (host arrays stay double)
 *              resident     1 = keep the propagated field in HBM as well: the next in-line device call that is handed
 *                           the very arrays this call returned (same data pointers, same fingerprint) skips its upload
 *              tolflag      0 | 1 (x.dphiadapt: first step by the local error) | 2 (x.ltol: every step), with ltol and
 *                           the safety factor of fiber.m:130
 *   [ux,uy] = ssfm_mex('ampliflat', ux, uy, gain, sigma, noise, asepol, opt)
 *       gain   linear power gain; sigma 1 x nfc; noise = Nfft x 2*nfc complex (options.noise, ampliflat.m:123-129) or a
 *              scalar seed of the device generator; asepol 1 = X, 2 = Y, 3 = both (options.onepol); opt as above
 *   [ux,uy] = ssfm_mex('dbp', ux, uy, betat, db1, P, gam, fls, plates, scal, D, steplen, spansteps, band, opt[, taps])
 *       digital backpropagation of a link (matlab/dbp.m; pmx_dbp_create / pmx_dbp_channel_create, pmx_dbp_exec)
 *       ux ... scal, opt   as for 'fiber' (opt = [scalar_field precision resident]); the resident field is used the same way
 *       D      [nspan gain steps_per_span xi pmd] or [nspan gain steps_per_span xi pmd bw]: linear amplifier gain after
 *              every span (0: none), uniform steps per span (0: the explicit schedule), fraction of gamma backpropagated,
 *              1 = PMD-aware DBP, and for filtered DBP the Gaussian's one-sided -3 dB bandwidth in bins (pmx_dbp_set_filter)
 *       steplen   [] or the steps in forward order: one span's steps for every span, or with spansteps (1 x nspan step
 *              counts) all spans' steps concatenated
 *       plates [] or (nplates*nspan) x 3 [db0 theta epsilon], span k in rows (k-1)*nplates+1 .. k*nplates, forward order
 *              (needs pmd = 1 and the 'p' flag)
 *       band   [] or [shift decim]: single-channel DBP of the channel shift bins bring to baseband, on Nfft/decim samples
 *       taps   absent or [], or enhanced split-step DBP: the real FIR c(1..2K+1) on the intensity of every nonlinear step,
 *              c(K+1) at lag 0 (pmx_dbp_set_taps)
 *   ssfm_mex('reset')                    drops the resident field
 *   c = ssfm_mex('stats')                [uploads downloads resident_hits] since the MEX file was loaded
 *
 * Build (not verifiable in the image this was written in -- it has no mex.h):
 *   mex ssfm_mex.c -I../include -L../polmux_b200/lib -lpolmux_ssfm
 *   mkoctfile --mex ssfm_mex.c -I../include -L../polmux_b200/lib -lpolmux_ssfm
 * The native test driver mex/test_ssfm_mex.c links this very file against mex_shim/mex.h.
 */
#include <math.h>
#include <string.h>
#include "mex.h"

#define PMX_MEX_MAX_NFC 64 /* the library's limit on field columns (polmux_ssfm.h: pmx_fiber_desc.nfc) */
#include "polmux_ssfm.h"

static pmx_ctx *g_ctx = NULL; /* one device context for the life of the MEX file */

static void drop_resident(void);

static void ssfm_at_exit(void)
{
    drop_resident();
    if (g_ctx) {
        pmx_ctx_destroy(g_ctx);
        g_ctx = NULL;
    }
}

static void fail(const char *what)
{
    static char msg[768];
    const char *detail = pmx_last_error(g_ctx);
    strncpy(msg, what, sizeof msg - 1);
    msg[sizeof msg - 1] = 0;
    if (detail && detail[0]) {
        strncat(msg, ": ", sizeof msg - strlen(msg) - 1);
        strncat(msg, detail, sizeof msg - strlen(msg) - 1);
    }
    mexErrMsgTxt(msg);
}

static void command(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]);

void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[])
{
    pmx_fiber_desc d;
    pmx_field io;
    pmx_fiber_result res;
    pmx_link_desc lk;
    double gam_buf[PMX_MEX_MAX_NFC], beta_buf[2 * PMX_MEX_MAX_NFC], sigma_buf[PMX_MEX_MAX_NFC];
    double *firstdz;
    int32_t *ncycle, *ntot, *status;
    uint64_t *seeds;
    size_t nfft, nfc, n, k, nspan;
    mxArray *uy_out, *work;
    int rc, is_link;

    if (nrhs >= 1 && mxIsChar(prhs[0])) {
        command(nlhs, plhs, nrhs, prhs);
        return;
    }
    if (nrhs < 16 || nrhs > 18)
        mexErrMsgTxt("ssfm_mex: 16 to 18 input arguments expected (see the header of ssfm_mex.c).");
    if (nlhs > 4)
        mexErrMsgTxt("ssfm_mex: at most 4 outputs [ux,uy,firstdz,ncycle].");

    nfft = mxGetM(prhs[0]);
    nfc = mxGetN(prhs[0]);
    n = nfft * nfc;
    if (n == 0)
        mexErrMsgTxt("ssfm_mex: empty x field.");
    if (nfc > PMX_MEX_MAX_NFC)
        mexErrMsgTxt("ssfm_mex: at most 64 field columns.");
    if (mxGetNumberOfElements(prhs[1]) != 0 && (mxGetM(prhs[1]) != nfft || mxGetN(prhs[1]) != nfc))
        mexErrMsgTxt("ssfm_mex: ux and uy must have the same size.");
    if ((size_t)mxGetScalar(prhs[8]) != nfc)
        mexErrMsgTxt("ssfm_mex: nfc does not match the number of columns of ux.");
    if (mxGetNumberOfElements(prhs[12]) != 4)
        mexErrMsgTxt("ssfm_mex: fls must have 4 elements.");

    memset(&d, 0, sizeof d);
    d.nfft = (int64_t)nfft;
    d.nfc = (int32_t)nfc;
    d.batch = 1;
    d.precision = PMX_F64;
    d.dzmaxt = mxGetScalar(prhs[4]);
    d.dphimaxt = mxGetScalar(prhs[5]);
    d.alphalin = mxGetScalar(prhs[7]);
    d.length = mxGetScalar(prhs[9]);
    d.nplates = (int32_t)mxGetScalar(prhs[10]);
    d.manakov = mxGetScalar(prhs[11]) != 0.0;
    for (k = 0; k < 4; k++)
        d.fls[k] = mxGetPr(prhs[12])[k] != 0.0;
    /* gam: scalar (nfc == 1) or one value per column */
    for (k = 0; k < nfc; k++)
        gam_buf[k] = mxGetPr(prhs[6])[mxGetNumberOfElements(prhs[6]) == 1 ? 0 : k];
    d.gam = gam_buf;
    /* one column of plates per span: a vector (either orientation) is one span */
    nspan = (d.nplates > 0) ? mxGetNumberOfElements(prhs[14]) / (size_t)d.nplates : 0;
    if (nspan < 1 || nspan * (size_t)d.nplates != mxGetNumberOfElements(prhs[14]) ||
        mxGetNumberOfElements(prhs[13]) != mxGetNumberOfElements(prhs[14]) ||
        mxGetNumberOfElements(prhs[15]) != mxGetNumberOfElements(prhs[14]))
        mexErrMsgTxt("ssfm_mex: db0, theta and epsilon must have nplates elements (nplates x Nspan for a span loop).");
    if (nspan > 1 && mxGetM(prhs[14]) != (size_t)d.nplates)
        mexErrMsgTxt("ssfm_mex: span loop: db0, theta and epsilon must be nplates x Nspan.");
    is_link = nspan > 1 || (nrhs == 18 && mxGetNumberOfElements(prhs[17]) != 0);
    d.plate_sets = 1;
    d.db0 = mxGetPr(prhs[13]);
    d.theta = mxGetPr(prhs[14]);
    d.epsilon = mxGetPr(prhs[15]);
    if (nrhs >= 17 && mxGetNumberOfElements(prhs[16]) != 0) {
        const double *s = mxGetPr(prhs[16]);
        if (mxGetNumberOfElements(prhs[16]) != 5 + 2 * nfc)
            mexErrMsgTxt("ssfm_mex: scal must be [symbolrate nsymb nt b30 dgdrms beta1(1:nfc) beta2(1:nfc)].");
        d.disp_mode = PMX_DISP_SCALAR;
        d.symbolrate = s[0];
        d.nsymb = (int32_t)s[1];
        d.nt = (int32_t)s[2];
        d.b30 = s[3];
        d.dgdrms = s[4];
        for (k = 0; k < 2 * nfc; k++)
            beta_buf[k] = s[5 + k];
        d.beta1 = beta_buf;
        d.beta2 = beta_buf + nfc;
    } else {
        if (mxGetM(prhs[2]) != nfft || mxGetN(prhs[2]) != nfc)
            mexErrMsgTxt("ssfm_mex: betat must be Nfft x nfc.");
        d.disp_mode = PMX_DISP_VECTOR;
        d.betat = mxGetPr(prhs[2]); /* column-major Nfft x nfc == [nfc][nfft] */
        d.db1 = (mxGetNumberOfElements(prhs[3]) == n) ? mxGetPr(prhs[3]) : NULL;
    }

    /* outputs are allocated first and the propagation runs in place on them */
    plhs[0] = mxCreateDoubleMatrix(nfft, nfc, mxCOMPLEX);
    uy_out = mxCreateDoubleMatrix(nfft, nfc, mxCOMPLEX);
    memcpy(mxGetPr(plhs[0]), mxGetPr(prhs[0]), n * sizeof(double));
    if (mxGetPi(prhs[0])) /* purely real arrays carry no imaginary plane (cmaadaptivefilter.c:136-140) */
        memcpy(mxGetPi(plhs[0]), mxGetPi(prhs[0]), n * sizeof(double));
    if (mxGetNumberOfElements(prhs[1]) == n) {
        memcpy(mxGetPr(uy_out), mxGetPr(prhs[1]), n * sizeof(double));
        if (mxGetPi(prhs[1]))
            memcpy(mxGetPi(uy_out), mxGetPi(prhs[1]), n * sizeof(double));
    }
    io.layout = PMX_PLANAR;
    io.reserved = 0;
    io.xr = mxGetPr(plhs[0]);
    io.xi = mxGetPi(plhs[0]);
    io.yr = mxGetPr(uy_out);
    io.yi = mxGetPi(uy_out);

    if (!g_ctx) {
        if (pmx_ctx_create(&g_ctx, 0) != PMX_OK)
            fail("ssfm_mex: no usable B200 (there is no CPU fallback)");
        mexAtExit(ssfm_at_exit);
    }
    /* per-span results live in one scratch matrix owned by the interpreter (freed on error, too) */
    work = mxCreateDoubleMatrix(4 * nspan, 1, mxREAL);
    firstdz = mxGetPr(work);
    ncycle = (int32_t *)(firstdz + nspan);
    ntot = ncycle + nspan;
    status = ntot + nspan;
    seeds = (uint64_t *)(firstdz + 3 * nspan);
    memset(&res, 0, sizeof res);
    res.firstdz = firstdz;
    res.ncycle = ncycle;
    res.ntot = ntot;
    res.status = status;
    if (is_link) {
        memset(&lk, 0, sizeof lk);
        lk.nspan = (int32_t)nspan;
        lk.plate_sets = 1;
        lk.db0 = d.db0; /* nplates x Nspan column-major == [nspan][1][nplates] */
        lk.theta = d.theta;
        lk.epsilon = d.epsilon;
        if (nrhs == 18 && mxGetNumberOfElements(prhs[17]) != 0) {
            const double *a = mxGetPr(prhs[17]);
            if (mxGetNumberOfElements(prhs[17]) != 2 + nfc)
                mexErrMsgTxt("ssfm_mex: amp must be [gain sigma(1:nfc) seed].");
            if (!(a[0] > 0.0))
                mexErrMsgTxt("ssfm_mex: amp(1) is the linear power gain 10^(G/10) and must be positive.");
            lk.gain = a[0];
            for (k = 0; k < nfc; k++)
                sigma_buf[k] = a[1 + k];
            lk.sigma = sigma_buf;
            for (k = 0; k < nspan; k++)
                seeds[k] = (uint64_t)a[1 + nfc] + (uint64_t)k;
            lk.seeds = seeds;
        }
        rc = pmx_link_run(g_ctx, &d, &lk, &io, &res);
    } else {
        rc = pmx_fiber_run(g_ctx, &d, &io, &res);
    }
    if (nlhs > 1)
        plhs[1] = uy_out;
    else
        mxDestroyArray(uy_out);
    if (rc == PMX_ERR_PLATE_INDEX)
        fail("ssfm_mex: index out of bound; value out of bound nplates (fiber.m:910)");
    if (rc != PMX_OK)
        fail("ssfm_mex: propagation failed");

    if (nlhs > 2) {
        plhs[2] = mxCreateDoubleMatrix(1, 1, mxREAL);
        *mxGetPr(plhs[2]) = firstdz[0];
    }
    if (nlhs > 3) {
        plhs[3] = mxCreateDoubleMatrix(1, nspan, mxREAL);
        for (k = 0; k < nspan; k++)
            mxGetPr(plhs[3])[k] = (double)ncycle[k];
    }
    mxDestroyArray(work);
}

/* ------------------------------------------------------------------------------------------------
 * Command interface.  The propagated field may stay in HBM between calls (opt(3) = resident): the
 * interpreter always gets its arrays back (any M code may read GSTATE.FIELDX), but the next in-line
 * device that is handed exactly those arrays -- same data pointers, same fingerprint -- does not
 * upload them again. */
static struct {
    pmx_devfield *f;
    size_t nfft, nfc;
    int precision, has_y;
    const double *p[4];   /* data pointers of the arrays handed back by the last call */
    double fp[4];         /* fingerprints of their contents */
} g_res;
static double g_stats[3]; /* uploads, downloads, resident hits */

static void ensure_ctx(void)
{
    if (!g_ctx) {
        if (pmx_ctx_create(&g_ctx, 0) != PMX_OK)
            fail("ssfm_mex: no usable B200 (there is no CPU fallback)");
        mexAtExit(ssfm_at_exit);
    }
}

static void drop_resident(void)
{
    if (g_res.f)
        pmx_field_destroy(g_res.f);
    memset(&g_res, 0, sizeof g_res);
}

/* a few hundred samples spread over the plane, combined so that an in-place edit is unlikely to go unnoticed */
static double fingerprint(const double *v, size_t n)
{
    double acc = 0.0;
    size_t k, step;
    if (!v || n == 0)
        return 0.0;
    step = n / 509 + 1;
    for (k = 0; k < n; k += step)
        acc = acc * 1.0000001192092896 + v[k];
    return acc + 3.0 * v[0] + 5.0 * v[n - 1] + 7.0 * v[n / 2];
}

static double opt_at(const mxArray *o, size_t k, double dflt)
{
    return (o && mxGetNumberOfElements(o) > k) ? mxGetPr(o)[k] : dflt;
}

/* the field of this call on the device: the resident one when the caller hands back what it was given, else an upload */
static pmx_devfield *acquire(const mxArray *ux, const mxArray *uy, int precision)
{
    const size_t nfft = mxGetM(ux), nfc = mxGetN(ux), n = nfft * nfc;
    const int has_y = uy && mxGetNumberOfElements(uy) == n;
    const double *p[4];
    pmx_field h;
    pmx_devfield *f;
    p[0] = mxGetPr(ux);
    p[1] = mxGetPi(ux);
    p[2] = has_y ? mxGetPr(uy) : NULL;
    p[3] = has_y ? mxGetPi(uy) : NULL;
    if (g_res.f && g_res.nfft == nfft && g_res.nfc == nfc && g_res.precision == precision && g_res.has_y == has_y &&
        p[0] == g_res.p[0] && p[1] == g_res.p[1] && p[2] == g_res.p[2] && p[3] == g_res.p[3] &&
        fingerprint(p[0], n) == g_res.fp[0] && fingerprint(p[1], n) == g_res.fp[1] &&
        fingerprint(p[2], n) == g_res.fp[2] && fingerprint(p[3], n) == g_res.fp[3]) {
        f = g_res.f;
        g_res.f = NULL;
        g_stats[2] += 1.0;
        return f;
    }
    drop_resident();
    if (pmx_field_create(g_ctx, (int64_t)nfft, (int32_t)nfc, 1, precision, &f) != PMX_OK)
        fail("ssfm_mex: device allocation failed");
    h.layout = PMX_PLANAR;
    h.reserved = 0;
    h.xr = (double *)p[0];
    h.xi = (double *)p[1];
    h.yr = (double *)p[2];
    h.yi = (double *)p[3];
    if (pmx_field_upload(f, &h, 0, 1) != PMX_OK) {
        pmx_field_destroy(f);
        fail("ssfm_mex: upload failed");
    }
    g_stats[0] += 1.0;
    return f;
}

/* hand the field back to the interpreter (always) and keep the device copy when asked to */
static void release(pmx_devfield *f, size_t nfft, size_t nfc, int precision, int with_y, int resident, int nlhs,
                    mxArray *plhs[])
{
    const size_t n = nfft * nfc;
    mxArray *ox = mxCreateDoubleMatrix(nfft, nfc, mxCOMPLEX);
    mxArray *oy = mxCreateDoubleMatrix(nfft, nfc, mxCOMPLEX);
    pmx_field h;
    h.layout = PMX_PLANAR;
    h.reserved = 0;
    h.xr = mxGetPr(ox);
    h.xi = mxGetPi(ox);
    h.yr = mxGetPr(oy);
    h.yi = mxGetPi(oy);
    if (pmx_field_download(f, &h, 0, 1) != PMX_OK) {
        pmx_field_destroy(f);
        fail("ssfm_mex: download failed");
    }
    g_stats[1] += 1.0;
    plhs[0] = ox;
    if (with_y && nlhs > 1) {
        plhs[1] = oy;
    } else {
        mxDestroyArray(oy);
        oy = NULL;
        if (nlhs > 1)
            plhs[1] = mxCreateDoubleMatrix(0, 0, mxREAL);
    }
    if (resident && (oy || !with_y)) {
        g_res.f = f;
        g_res.nfft = nfft;
        g_res.nfc = nfc;
        g_res.precision = precision;
        g_res.has_y = oy != NULL;
        g_res.p[0] = mxGetPr(ox);
        g_res.p[1] = mxGetPi(ox);
        g_res.p[2] = oy ? mxGetPr(oy) : NULL;
        g_res.p[3] = oy ? mxGetPi(oy) : NULL;
        g_res.fp[0] = fingerprint(g_res.p[0], n);
        g_res.fp[1] = fingerprint(g_res.p[1], n);
        g_res.fp[2] = fingerprint(g_res.p[2], n);
        g_res.fp[3] = fingerprint(g_res.p[3], n);
    } else {
        pmx_field_destroy(f);
    }
}

static void cmd_fiber(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[])
{
    /* prhs: 'fiber', ux, uy, betat, db1, P, gam, fls, plates, scal, opt */
    pmx_fiber_desc d;
    pmx_fiber_result res;
    pmx_plan *plan = NULL;
    pmx_devfield *f;
    double gam_buf[PMX_MEX_MAX_NFC], beta_buf[2 * PMX_MEX_MAX_NFC], firstdz = 0.0;
    const double *P, *pl;
    int32_t ncycle = 0, ntot = 0, status = 0;
    size_t nfft, nfc, n, k, np;
    int scalar_field, precision, resident, tolflag, rc, has_y;
    const mxArray *opt = nrhs > 10 ? prhs[10] : NULL;

    if (nrhs < 10 || nrhs > 11)
        mexErrMsgTxt("ssfm_mex('fiber',ux,uy,betat,db1,P,gam,fls,plates,scal[,opt]): wrong number of arguments.");
    if (nlhs > 4)
        mexErrMsgTxt("ssfm_mex: at most 4 outputs [ux,uy,firstdz,ncycle].");
    nfft = mxGetM(prhs[1]);
    nfc = mxGetN(prhs[1]);
    n = nfft * nfc;
    if (n == 0)
        mexErrMsgTxt("ssfm_mex: empty x field.");
    if (nfc > PMX_MEX_MAX_NFC)
        mexErrMsgTxt("ssfm_mex: at most 64 field columns.");
    has_y = mxGetNumberOfElements(prhs[2]) != 0;
    if (has_y && (mxGetM(prhs[2]) != nfft || mxGetN(prhs[2]) != nfc))
        mexErrMsgTxt("ssfm_mex: ux and uy must have the same size.");
    if (mxGetNumberOfElements(prhs[5]) != 6)
        mexErrMsgTxt("ssfm_mex: P must be [dzmaxt dphimaxt alphalin Lf nplates manakov].");
    if (mxGetNumberOfElements(prhs[7]) != 4)
        mexErrMsgTxt("ssfm_mex: fls must have 4 elements.");
    scalar_field = opt_at(opt, 0, 0.0) != 0.0;
    precision = opt_at(opt, 1, 0.0) != 0.0 ? PMX_F32 : PMX_F64;
    resident = opt_at(opt, 2, 0.0) != 0.0;
    tolflag = (int)opt_at(opt, 3, 0.0);
    if (scalar_field && has_y)
        mexErrMsgTxt("ssfm_mex: the scalar path takes no y field (fiber.m:253).");

    P = mxGetPr(prhs[5]);
    memset(&d, 0, sizeof d);
    d.nfft = (int64_t)nfft;
    d.nfc = (int32_t)nfc;
    d.batch = 1;
    d.precision = precision;
    d.dzmaxt = P[0];
    d.dphimaxt = P[1];
    d.alphalin = P[2];
    d.length = P[3];
    d.nplates = (int32_t)P[4];
    d.manakov = P[5] != 0.0;
    d.scalar_field = scalar_field;
    for (k = 0; k < 4; k++)
        d.fls[k] = mxGetPr(prhs[7])[k] != 0.0;
    for (k = 0; k < nfc; k++)
        gam_buf[k] = mxGetPr(prhs[6])[mxGetNumberOfElements(prhs[6]) == 1 ? 0 : k];
    d.gam = gam_buf;
    d.plate_sets = 1;
    np = (size_t)d.nplates;
    if (mxGetNumberOfElements(prhs[8]) != 0) {
        if (mxGetM(prhs[8]) != np || mxGetN(prhs[8]) != 3)
            mexErrMsgTxt("ssfm_mex: plates must be nplates x 3 [db0 theta epsilon].");
        pl = mxGetPr(prhs[8]);
        d.db0 = pl;
        d.theta = pl + np;
        d.epsilon = pl + 2 * np;
    } else if (d.fls[1]) {
        mexErrMsgTxt("ssfm_mex: the 'p' flag needs the waveplates.");
    }
    if (mxGetNumberOfElements(prhs[9]) != 0) {
        const double *s = mxGetPr(prhs[9]);
        if (mxGetNumberOfElements(prhs[9]) != 5 + 2 * nfc)
            mexErrMsgTxt("ssfm_mex: scal must be [symbolrate nsymb nt b30 dgdrms beta1(1:nfc) beta2(1:nfc)].");
        d.disp_mode = PMX_DISP_SCALAR;
        d.symbolrate = s[0];
        d.nsymb = (int32_t)s[1];
        d.nt = (int32_t)s[2];
        d.b30 = s[3];
        d.dgdrms = s[4];
        for (k = 0; k < 2 * nfc; k++)
            beta_buf[k] = s[5 + k];
        d.beta1 = beta_buf;
        d.beta2 = beta_buf + nfc;
    } else {
        if (mxGetM(prhs[3]) != nfft || mxGetN(prhs[3]) != nfc)
            mexErrMsgTxt("ssfm_mex: betat must be Nfft x nfc.");
        d.disp_mode = PMX_DISP_VECTOR;
        d.betat = mxGetPr(prhs[3]);
        d.db1 = (mxGetNumberOfElements(prhs[4]) == n) ? mxGetPr(prhs[4]) : NULL;
    }
    ensure_ctx();
    memset(&res, 0, sizeof res);
    res.firstdz = &firstdz;
    res.ncycle = &ncycle;
    res.ntot = &ntot;
    res.status = &status;

    if (tolflag) { /* scalar_a_ssfm (2) / scalar_ssfm with x.dphiadapt (1): host buffers in, host buffers out */
        pmx_field io;
        if (!scalar_field)
            mexErrMsgTxt("adaptive step available in absence of polarization effects"); /* fiber.m:373 */
        drop_resident();
        plhs[0] = mxCreateDoubleMatrix(nfft, nfc, mxCOMPLEX);
        memcpy(mxGetPr(plhs[0]), mxGetPr(prhs[1]), n * sizeof(double));
        if (mxGetPi(prhs[1]))
            memcpy(mxGetPi(plhs[0]), mxGetPi(prhs[1]), n * sizeof(double));
        io.layout = PMX_PLANAR;
        io.reserved = 0;
        io.xr = mxGetPr(plhs[0]);
        io.xi = mxGetPi(plhs[0]);
        io.yr = io.yi = NULL;
        rc = pmx_scalar_adaptive_run(g_ctx, &d, opt_at(opt, 4, 0.0), opt_at(opt, 5, 0.9), tolflag == 1, &io, &res);
        if (rc != PMX_OK)
            fail("ssfm_mex: adaptive propagation failed");
        if (nlhs > 1)
            plhs[1] = mxCreateDoubleMatrix(0, 0, mxREAL);
    } else {
        if (pmx_plan_create(g_ctx, &d, &plan) != PMX_OK) {
            if (d.fls[3] && !scalar_field)
                mexErrMsgTxt("The CNLSE with separate fields is not yet implemented"); /* fiber.m:854 */
            fail("ssfm_mex: plan creation failed");
        }
        f = acquire(prhs[1], prhs[2], precision);
        rc = pmx_fiber_exec(plan, f, &res);
        pmx_plan_destroy(plan);
        if (rc != PMX_OK) {
            pmx_field_destroy(f);
            if (rc == PMX_ERR_PLATE_INDEX)
                fail("ssfm_mex: index out of bound; value out of bound nplates (fiber.m:910)");
            fail("ssfm_mex: propagation failed");
        }
        release(f, nfft, nfc, precision, !scalar_field, resident, nlhs, plhs);
    }
    if (nlhs > 2) {
        plhs[2] = mxCreateDoubleMatrix(1, 1, mxREAL);
        *mxGetPr(plhs[2]) = firstdz;
    }
    if (nlhs > 3) {
        plhs[3] = mxCreateDoubleMatrix(1, 1, mxREAL);
        *mxGetPr(plhs[3]) = (double)ncycle;
    }
}

static void cmd_ampliflat(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[])
{
    /* prhs: 'ampliflat', ux, uy, gain, sigma, noise, asepol, opt */
    double sigma_buf[PMX_MEX_MAX_NFC], *nz = NULL;
    const mxArray *opt = nrhs > 7 ? prhs[7] : NULL;
    pmx_devfield *f;
    size_t nfft, nfc, n, k, c;
    uint64_t seed = 0;
    int precision, resident, asepol, rc;
    mxArray *work = NULL;

    if (nrhs < 7 || nrhs > 8 || nlhs != 2)
        mexErrMsgTxt("[ux,uy] = ssfm_mex('ampliflat',ux,uy,gain,sigma,noise,asepol[,opt]): wrong number of arguments.");
    nfft = mxGetM(prhs[1]);
    nfc = mxGetN(prhs[1]);
    n = nfft * nfc;
    if (n == 0 || nfc > PMX_MEX_MAX_NFC)
        mexErrMsgTxt("ssfm_mex: bad x field.");
    if (mxGetNumberOfElements(prhs[4]) != nfc)
        mexErrMsgTxt("ssfm_mex: sigma must have one entry per field column.");
    for (k = 0; k < nfc; k++)
        sigma_buf[k] = mxGetPr(prhs[4])[k];
    asepol = (int)mxGetScalar(prhs[6]);
    precision = opt_at(opt, 1, 0.0) != 0.0 ? PMX_F32 : PMX_F64;
    resident = opt_at(opt, 2, 0.0) != 0.0;
    if (mxGetNumberOfElements(prhs[5]) == 2 * n) { /* options.noise: Nfft x 2*nfc complex -> [2*nfc][nfft] interleaved */
        const double *re = mxGetPr(prhs[5]), *im = mxGetPi(prhs[5]);
        work = mxCreateDoubleMatrix(4 * n, 1, mxREAL);
        nz = mxGetPr(work);
        for (c = 0; c < 2 * nfc; c++)
            for (k = 0; k < nfft; k++) {
                nz[2 * (c * nfft + k)] = re[c * nfft + k];
                nz[2 * (c * nfft + k) + 1] = im ? im[c * nfft + k] : 0.0;
            }
    } else if (mxGetNumberOfElements(prhs[5]) == 1) {
        seed = (uint64_t)mxGetScalar(prhs[5]);
    } else if (mxGetNumberOfElements(prhs[5]) != 0) {
        mexErrMsgTxt("ssfm_mex: noise must be Nfft x 2*nfc (options.noise) or a scalar seed.");
    }
    ensure_ctx();
    f = acquire(prhs[1], prhs[2], precision);
    rc = pmx_ampliflat_exec_pol(g_ctx, f, mxGetScalar(prhs[3]), sigma_buf, nz, seed, asepol);
    if (work)
        mxDestroyArray(work);
    if (rc != PMX_OK) {
        pmx_field_destroy(f);
        fail("ssfm_mex: ampliflat failed");
    }
    release(f, nfft, nfc, precision, 1, resident, nlhs, plhs);
}

static void cmd_dbp(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[])
{
    /* prhs: 'dbp', ux, uy, betat, db1, P, gam, fls, plates, scal, D, steplen, spansteps, band, opt[, taps] */
    pmx_fiber_desc d;
    pmx_dbp_desc g;
    pmx_dbp_band b;
    pmx_plan *plan = NULL;
    pmx_devfield *f;
    double gam_buf[PMX_MEX_MAX_NFC], beta_buf[2 * PMX_MEX_MAX_NFC];
    const double *P, *D, *pl = NULL;
    size_t nfft, nfc, n, k, j, np, nspan, nsteps = 0;
    int scalar_field, precision, resident, rc, has_y, channel;
    mxArray *work = NULL;
    const mxArray *opt = prhs[14];

    if ((nrhs != 15 && nrhs != 16) || nlhs > 2)
        mexErrMsgTxt("[ux,uy] = ssfm_mex('dbp',ux,uy,betat,db1,P,gam,fls,plates,scal,D,steplen,spansteps,band,opt[,taps]): "
                     "wrong number of arguments.");
    nfft = mxGetM(prhs[1]);
    nfc = mxGetN(prhs[1]);
    n = nfft * nfc;
    if (n == 0)
        mexErrMsgTxt("ssfm_mex: empty x field.");
    if (nfc > PMX_MEX_MAX_NFC)
        mexErrMsgTxt("ssfm_mex: at most 64 field columns.");
    has_y = mxGetNumberOfElements(prhs[2]) != 0;
    if (has_y && (mxGetM(prhs[2]) != nfft || mxGetN(prhs[2]) != nfc))
        mexErrMsgTxt("ssfm_mex: ux and uy must have the same size.");
    if (mxGetNumberOfElements(prhs[5]) != 6)
        mexErrMsgTxt("ssfm_mex: P must be [dzmaxt dphimaxt alphalin Lf nplates manakov].");
    if (mxGetNumberOfElements(prhs[7]) != 4)
        mexErrMsgTxt("ssfm_mex: fls must have 4 elements.");
    if (mxGetNumberOfElements(prhs[10]) != 5 && mxGetNumberOfElements(prhs[10]) != 6)
        mexErrMsgTxt("ssfm_mex: D must be [nspan gain steps_per_span xi pmd] or [nspan gain steps_per_span xi pmd bw].");
    scalar_field = opt_at(opt, 0, 0.0) != 0.0;
    precision = opt_at(opt, 1, 0.0) != 0.0 ? PMX_F32 : PMX_F64;
    resident = opt_at(opt, 2, 0.0) != 0.0;
    if (scalar_field && has_y)
        mexErrMsgTxt("ssfm_mex: the scalar path takes no y field (fiber.m:253).");

    /* the fiber: the same parsing as 'fiber' */
    P = mxGetPr(prhs[5]);
    memset(&d, 0, sizeof d);
    d.nfft = (int64_t)nfft;
    d.nfc = (int32_t)nfc;
    d.batch = 1;
    d.precision = precision;
    d.dzmaxt = P[0];
    d.dphimaxt = P[1];
    d.alphalin = P[2];
    d.length = P[3];
    d.nplates = (int32_t)P[4];
    d.manakov = P[5] != 0.0;
    d.scalar_field = scalar_field;
    for (k = 0; k < 4; k++)
        d.fls[k] = mxGetPr(prhs[7])[k] != 0.0;
    for (k = 0; k < nfc; k++)
        gam_buf[k] = mxGetPr(prhs[6])[mxGetNumberOfElements(prhs[6]) == 1 ? 0 : k];
    d.gam = gam_buf;
    d.plate_sets = 1;
    if (mxGetNumberOfElements(prhs[9]) != 0) {
        const double *s = mxGetPr(prhs[9]);
        if (mxGetNumberOfElements(prhs[9]) != 5 + 2 * nfc)
            mexErrMsgTxt("ssfm_mex: scal must be [symbolrate nsymb nt b30 dgdrms beta1(1:nfc) beta2(1:nfc)].");
        d.disp_mode = PMX_DISP_SCALAR;
        d.symbolrate = s[0];
        d.nsymb = (int32_t)s[1];
        d.nt = (int32_t)s[2];
        d.b30 = s[3];
        d.dgdrms = s[4];
        for (k = 0; k < 2 * nfc; k++)
            beta_buf[k] = s[5 + k];
        d.beta1 = beta_buf;
        d.beta2 = beta_buf + nfc;
    } else {
        if (mxGetM(prhs[3]) != nfft || mxGetN(prhs[3]) != nfc)
            mexErrMsgTxt("ssfm_mex: betat must be Nfft x nfc.");
        d.disp_mode = PMX_DISP_VECTOR;
        d.betat = mxGetPr(prhs[3]);
        d.db1 = (mxGetNumberOfElements(prhs[4]) == n) ? mxGetPr(prhs[4]) : NULL;
    }

    /* the link: D, the step schedule, the waveplates of every span */
    D = mxGetPr(prhs[10]);
    memset(&g, 0, sizeof g);
    g.nspan = (int32_t)D[0];
    g.gain = D[1];
    g.steps_per_span = (int32_t)D[2];
    g.xi = D[3];
    g.pmd = D[4] != 0.0;
    if (g.nspan < 1)
        mexErrMsgTxt("ssfm_mex: D(1), the number of spans, must be at least 1.");
    nspan = (size_t)g.nspan;
    np = (size_t)(d.nplates > 0 ? d.nplates : 0);
    if (g.pmd) {
        if (mxGetM(prhs[8]) != np * nspan || mxGetN(prhs[8]) != 3 || np == 0)
            mexErrMsgTxt("ssfm_mex: PMD-aware DBP: plates must be (nplates*nspan) x 3 [db0 theta epsilon].");
        pl = mxGetPr(prhs[8]);
    } else if (mxGetNumberOfElements(prhs[8]) != 0) {
        mexErrMsgTxt("ssfm_mex: plates are given only for PMD-aware DBP (D(5) = 1).");
    }
    if (mxGetNumberOfElements(prhs[11]) != 0) { /* explicit schedule: steplen in forward order, spansteps per span */
        const double *sl = mxGetPr(prhs[11]), *ss = mxGetPr(prhs[12]);
        const size_t nl = mxGetNumberOfElements(prhs[11]), nss = mxGetNumberOfElements(prhs[12]);
        double *buf;
        int32_t *cnt;
        if (g.steps_per_span != 0)
            mexErrMsgTxt("ssfm_mex: give steps_per_span (D(3)) or steplen, not both.");
        if (nss != 0 && nss != nspan)
            mexErrMsgTxt("ssfm_mex: spansteps must give the steps of every span.");
        nsteps = nss ? nl : nl * nspan; /* without spansteps, steplen is one span's steps, repeated for every span */
        work = mxCreateDoubleMatrix(nsteps + nspan, 1, mxREAL);
        buf = mxGetPr(work);
        cnt = (int32_t *)(buf + nsteps);
        if (nss) {
            size_t tot = 0;
            for (k = 0; k < nspan; k++) {
                if (!(ss[k] >= 1.0) || ss[k] != floor(ss[k]))
                    mexErrMsgTxt("ssfm_mex: spansteps must hold positive integers.");
                cnt[k] = (int32_t)ss[k];
                tot += (size_t)cnt[k];
            }
            if (tot != nl)
                mexErrMsgTxt("ssfm_mex: steplen must hold sum(spansteps) steps.");
            memcpy(buf, sl, nl * sizeof(double));
        } else {
            for (k = 0; k < nspan; k++) {
                cnt[k] = (int32_t)nl;
                for (j = 0; j < nl; j++)
                    buf[k * nl + j] = sl[j];
            }
        }
        g.step_len = buf;
        g.span_steps = cnt;
    } else if (mxGetNumberOfElements(prhs[12]) != 0) {
        mexErrMsgTxt("ssfm_mex: spansteps needs steplen.");
    }
    channel = mxGetNumberOfElements(prhs[13]) != 0;
    if (channel) {
        if (mxGetNumberOfElements(prhs[13]) != 2)
            mexErrMsgTxt("ssfm_mex: band must be [shift decim].");
        memset(&b, 0, sizeof b);
        b.shift = (int64_t)mxGetPr(prhs[13])[0];
        b.decim = (int32_t)mxGetPr(prhs[13])[1];
    }

    ensure_ctx();
    rc = channel ? pmx_dbp_channel_create(g_ctx, &d, &g, &b, &plan) : pmx_dbp_create(g_ctx, &d, &g, &plan);
    if (work)
        mxDestroyArray(work); /* the plan has taken the schedule */
    if (rc != PMX_OK) {
        if (d.fls[3] && !scalar_field)
            mexErrMsgTxt("The CNLSE with separate fields is not yet implemented"); /* fiber.m:854 */
        fail("ssfm_mex: DBP plan creation failed");
    }
    if (g.pmd && pmx_dbp_set_plates(plan, 1, pl, pl + np * nspan, pl + 2 * np * nspan) != PMX_OK) {
        pmx_plan_destroy(plan);
        fail("ssfm_mex: DBP waveplates rejected");
    }
    if (mxGetNumberOfElements(prhs[10]) == 6 && pmx_dbp_set_filter(plan, D[5]) != PMX_OK) {
        pmx_plan_destroy(plan);
        fail("ssfm_mex: DBP filter bandwidth rejected");
    }
    if (nrhs == 16 && mxGetNumberOfElements(prhs[15]) != 0 &&
        pmx_dbp_set_taps(plan, (int32_t)mxGetNumberOfElements(prhs[15]), mxGetPr(prhs[15])) != PMX_OK) {
        pmx_plan_destroy(plan);
        fail("ssfm_mex: DBP taps rejected");
    }
    f = acquire(prhs[1], prhs[2], precision);
    rc = pmx_dbp_exec(plan, f);
    pmx_plan_destroy(plan);
    if (rc != PMX_OK) {
        pmx_field_destroy(f); /* part-way through the link: not usable */
        fail("ssfm_mex: backpropagation failed");
    }
    release(f, nfft, nfc, precision, !scalar_field, resident, nlhs, plhs);
}

/* complex mxArray (split storage) -> interleaved re,im in a fresh mxArray-owned buffer of 2*n doubles */
static double *interleave(const mxArray *a, size_t n, mxArray **owner)
{
    const double *re = mxGetPr(a), *im = mxGetPi(a);
    double *out;
    size_t k;
    *owner = mxCreateDoubleMatrix(2 * n, 1, mxREAL);
    out = mxGetPr(*owner);
    for (k = 0; k < n; k++) {
        out[2 * k] = re[k];
        out[2 * k + 1] = im ? im[k] : 0.0;
    }
    return out;
}

static void cmd_cohmix(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[])
{
    /* [Iric,avgeb] = ssfm_mex('cohmix', sigx, sigy, Hopt, Hel, lo, lophase, band, opt)
     *   sigx, sigy : the channel's column of GSTATE.FIELDX / FIELDY (sigy empty: one polarization)
     *   Hopt, Hel  : Nfft x 1 filter responses over GSTATE.FN (receiver_cohmix.m:169,293)
     *   lo         : [LO_Ecw, 2*pi*kdet/Nfft, balanced]      lophase : Nfft x 1 or []
     *   band       : [ndfn, ndfnl, ndfnr]                     opt     : [0, precision] */
    pmx_cohmix_desc d;
    pmx_field sig;
    mxArray *o1 = NULL, *o2 = NULL;
    const mxArray *opt = nrhs > 8 ? prhs[8] : NULL;
    size_t nfft;
    double avgeb[2] = {0.0, 0.0};
    int rc, two;

    if (nrhs < 8 || nrhs > 9 || nlhs > 2)
        mexErrMsgTxt("[Iric,avgeb] = ssfm_mex('cohmix',sigx,sigy,Hopt,Hel,lo,lophase,band[,opt]): wrong number of arguments.");
    nfft = mxGetNumberOfElements(prhs[1]);
    two = mxGetNumberOfElements(prhs[2]) == nfft;
    if (nfft == 0 || (!two && mxGetNumberOfElements(prhs[2]) != 0))
        mexErrMsgTxt("ssfm_mex: sigx must be a column of Nfft samples and sigy the same, or empty.");
    if (mxGetNumberOfElements(prhs[3]) != nfft || mxGetNumberOfElements(prhs[4]) != nfft)
        mexErrMsgTxt("ssfm_mex: the filter responses must have Nfft elements.");
    if (mxGetNumberOfElements(prhs[5]) != 3 || mxGetNumberOfElements(prhs[7]) != 3)
        mexErrMsgTxt("ssfm_mex: lo = [Ecw, detuning, balanced], band = [ndfn, ndfnl, ndfnr].");
    if (mxGetNumberOfElements(prhs[6]) != 0 && mxGetNumberOfElements(prhs[6]) != nfft)
        mexErrMsgTxt("Incompatible vector."); /* receiver_cohmix.m:204 */
    memset(&d, 0, sizeof d);
    d.nfft = (int64_t)nfft;
    d.precision = opt_at(opt, 1, 0.0) != 0.0 ? PMX_F32 : PMX_F64;
    d.two_pol = two;
    d.hf_opt = interleave(prhs[3], nfft, &o1);
    d.hf_el = interleave(prhs[4], nfft, &o2);
    d.lo_ecw = mxGetPr(prhs[5])[0];
    d.lo_detune = mxGetPr(prhs[5])[1];
    d.balanced = mxGetPr(prhs[5])[2] != 0.0;
    d.lo_phase = mxGetNumberOfElements(prhs[6]) ? mxGetPr(prhs[6]) : NULL;
    d.ndfn = (int64_t)mxGetPr(prhs[7])[0];
    d.ndfnl = (int64_t)mxGetPr(prhs[7])[1];
    d.ndfnr = (int64_t)mxGetPr(prhs[7])[2];
    memset(&sig, 0, sizeof sig);
    sig.layout = PMX_PLANAR;
    sig.xr = mxGetPr(prhs[1]);
    sig.xi = mxGetPi(prhs[1]);
    if (two) {
        sig.yr = mxGetPr(prhs[2]);
        sig.yi = mxGetPi(prhs[2]);
    }
    plhs[0] = mxCreateDoubleMatrix(nfft, two ? 4 : 2, mxREAL);
    ensure_ctx();
    rc = pmx_cohmix_run(g_ctx, &d, &sig, mxGetPr(plhs[0]), nlhs > 1 ? avgeb : NULL);
    mxDestroyArray(o1);
    mxDestroyArray(o2);
    if (rc != PMX_OK)
        fail("ssfm_mex: cohmix failed");
    if (nlhs > 1) {
        plhs[1] = mxCreateDoubleMatrix(1, 2, mxREAL);
        mxGetPr(plhs[1])[0] = avgeb[0];
        mxGetPr(plhs[1])[1] = avgeb[1];
    }
    g_stats[0] += 1.0; /* one upload of the column, one download of the currents */
    g_stats[1] += 1.0;
}

static void cmd_invpmd(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[])
{
    /* [ux,uy,Uinv4,U4] = ssfm_mex('invpmd', ux, uy, plates, ntr, lcorr, betat, db1, mat, flags)
     *   plates : sum(ntr) x 3 = [db0 theta epsilon] of the fibers one after the other      ntr, lcorr : 1 x nfiber
     *   betat, db1 : Nfft x nfiber (brf{k}.betat, brf{k}.db1)      mat : 2 x 2 (options.mat) or []
     *   flags  : [gvd apply]          Uinv4, U4 : 4 x Nfft, column n = [M11; M21; M12; M22] at GSTATE.FN(n) */
    pmx_brf brf[64];
    pmx_field io;
    mxArray *wu = NULL, *wi = NULL;
    double matbuf[8], *U = NULL, *Ui = NULL;
    const double *pl;
    size_t nfft, nfib, k, n, row = 0, tot;
    int gvd, apply, rc;

    if (nrhs != 10 || nlhs < 2 || nlhs > 4)
        mexErrMsgTxt("[ux,uy,Uinv4,U4] = ssfm_mex('invpmd',ux,uy,plates,ntr,lcorr,betat,db1,mat,flags): wrong number of arguments.");
    nfft = mxGetM(prhs[1]);
    nfib = mxGetNumberOfElements(prhs[4]);
    if (mxGetN(prhs[1]) != 1)
        mexErrMsgTxt("inverse_pmd can be used only with a unique field."); /* inverse_pmd.m:63 */
    if (nfib < 1 || nfib > 64 || mxGetNumberOfElements(prhs[5]) != nfib || mxGetM(prhs[6]) != nfft || mxGetN(prhs[6]) != nfib ||
        mxGetM(prhs[7]) != nfft || mxGetN(prhs[7]) != nfib || mxGetN(prhs[3]) != 3 || mxGetNumberOfElements(prhs[9]) != 2)
        mexErrMsgTxt("ssfm_mex: invpmd: inconsistent fiber tables.");
    tot = mxGetM(prhs[3]);
    pl = mxGetPr(prhs[3]);
    for (k = 0; k < nfib; k++) {
        memset(&brf[k], 0, sizeof brf[k]);
        brf[k].ntrunk = (int32_t)mxGetPr(prhs[4])[k];
        brf[k].lcorr = mxGetPr(prhs[5])[k];
        if (brf[k].ntrunk < 1 || row + (size_t)brf[k].ntrunk > tot)
            mexErrMsgTxt("ssfm_mex: invpmd: plates and ntr disagree.");
        brf[k].db0 = pl + row;
        brf[k].theta = pl + tot + row;
        brf[k].epsilon = pl + 2 * tot + row;
        brf[k].betat = mxGetPr(prhs[6]) + k * nfft;
        brf[k].db1 = mxGetPr(prhs[7]) + k * nfft;
        row += (size_t)brf[k].ntrunk;
    }
    if (mxGetNumberOfElements(prhs[8]) == 4) { /* row-major re,im of the column-major 2 x 2 */
        const double *re = mxGetPr(prhs[8]), *im = mxGetPi(prhs[8]);
        static const int order[4] = {0, 2, 1, 3};
        for (k = 0; k < 4; k++) {
            matbuf[2 * k] = re[order[k]];
            matbuf[2 * k + 1] = im ? im[order[k]] : 0.0;
        }
    } else if (mxGetNumberOfElements(prhs[8]) != 0) {
        mexErrMsgTxt("ssfm_mex: invpmd: options.mat must be 2 x 2.");
    }
    gvd = mxGetPr(prhs[9])[0] != 0.0;
    apply = mxGetPr(prhs[9])[1] != 0.0;
    plhs[0] = mxCreateDoubleMatrix(nfft, 1, mxCOMPLEX);
    plhs[1] = mxCreateDoubleMatrix(nfft, 1, mxCOMPLEX);
    memcpy(mxGetPr(plhs[0]), mxGetPr(prhs[1]), nfft * sizeof(double));
    if (mxGetPi(prhs[1])) memcpy(mxGetPi(plhs[0]), mxGetPi(prhs[1]), nfft * sizeof(double));
    memcpy(mxGetPr(plhs[1]), mxGetPr(prhs[2]), nfft * sizeof(double));
    if (mxGetPi(prhs[2])) memcpy(mxGetPi(plhs[1]), mxGetPi(prhs[2]), nfft * sizeof(double));
    memset(&io, 0, sizeof io);
    io.layout = PMX_PLANAR;
    io.xr = mxGetPr(plhs[0]);
    io.xi = mxGetPi(plhs[0]);
    io.yr = mxGetPr(plhs[1]);
    io.yi = mxGetPi(plhs[1]);
    if (nlhs > 2) {
        wi = mxCreateDoubleMatrix(8 * nfft, 1, mxREAL);
        Ui = mxGetPr(wi);
    }
    if (nlhs > 3) {
        wu = mxCreateDoubleMatrix(8 * nfft, 1, mxREAL);
        U = mxGetPr(wu);
    }
    ensure_ctx();
    rc = pmx_inverse_pmd_run(g_ctx, (int64_t)nfft, (int32_t)nfib, brf, mxGetNumberOfElements(prhs[8]) == 4 ? matbuf : NULL, gvd,
                             apply, &io, U, Ui);
    if (rc != PMX_OK) {
        if (wi) mxDestroyArray(wi);
        if (wu) mxDestroyArray(wu);
        fail("ssfm_mex: invpmd failed");
    }
    for (k = 2; k < (size_t)nlhs; k++) { /* interleaved [nfft][4] -> split storage 4 x nfft */
        const double *src = (k == 2) ? Ui : U;
        plhs[k] = mxCreateDoubleMatrix(4, nfft, mxCOMPLEX);
        for (n = 0; n < 4 * nfft; n++) {
            mxGetPr(plhs[k])[n] = src[2 * n];
            mxGetPi(plhs[k])[n] = src[2 * n + 1];
        }
    }
    if (wi) mxDestroyArray(wi);
    if (wu) mxDestroyArray(wu);
    g_stats[0] += apply ? 1.0 : 0.0;
    g_stats[1] += apply ? 1.0 : 0.0;
}

static void command(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[])
{
    char cmd[32];
    if (mxGetString(prhs[0], cmd, sizeof cmd))
        mexErrMsgTxt("ssfm_mex: unknown command.");
    if (!strcmp(cmd, "fiber")) {
        cmd_fiber(nlhs, plhs, nrhs, prhs);
    } else if (!strcmp(cmd, "ampliflat")) {
        cmd_ampliflat(nlhs, plhs, nrhs, prhs);
    } else if (!strcmp(cmd, "cohmix")) {
        cmd_cohmix(nlhs, plhs, nrhs, prhs);
    } else if (!strcmp(cmd, "invpmd")) {
        cmd_invpmd(nlhs, plhs, nrhs, prhs);
    } else if (!strcmp(cmd, "dbp")) {
        cmd_dbp(nlhs, plhs, nrhs, prhs);
    } else if (!strcmp(cmd, "reset")) {
        drop_resident();
    } else if (!strcmp(cmd, "stats")) {
        plhs[0] = mxCreateDoubleMatrix(1, 3, mxREAL);
        memcpy(mxGetPr(plhs[0]), g_stats, sizeof g_stats);
    } else {
        mexErrMsgTxt("ssfm_mex: unknown command (fiber, ampliflat, cohmix, invpmd, dbp, reset, stats).");
    }
}
