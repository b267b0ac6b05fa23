function zbrf = fiber(x, flag)
%FIBER  Optical fiber, split-step Fourier propagation on a B200 (drop-in front-end).
%   ZBRF = FIBER(X,FLAG) keeps the contract of the toolbox's fiber.m: the same fields of X (length,
%   alphadB, aeff, n2, lambda, disp, slope, dzmax, dphimax, and with PMD dgd, nplates, manakov,
%   db0/theta/epsilon; ltol and dphiadapt for the local-error step), the same four-character FLAG
%   ('g','p','s','x' or '-' in positions 1..4), the same effects on GSTATE.FIELDX, GSTATE.FIELDY,
%   GSTATE.DELAY and GSTATE.DISP, and the same birefringence struct ZBRF when an output is asked for.
%
%   Put this directory BEFORE the toolbox on the path.  Everything up to the SSFM dispatch is plain
%   interpreter arithmetic in the toolbox's operation order (the part before the plate draw lives in
%   FIBER_SETUP, which DBP shares); the propagation loop itself -- the
%   toolbox's matrix_ssfm, scalar_ssfm and scalar_a_ssfm sub-functions -- runs inside the MEX gateway
%   ssfm_mex (mex/ssfm_mex.c -> libpolmux_ssfm.so).  There is no CPU fallback: without the gateway
%   the call fails.
%
%   Options of this front-end (fields of the global struct PMXOPT, all optional):
%     precision  'f64' (default) | 'f32'    arithmetic of the device path
%     resident   true (default) | false     keep the propagated field in HBM between in-line devices
%     scalar     true (default) | false     rebuild betat / db1 on the device from a few scalars
%                                           instead of uploading the two Nfft x nfc vectors

global CONSTANTS GSTATE PMXOPT

if nargin < 2
    error('Missing propagation type');
end
c0 = CONSTANTS.CLIGHT;
ncol = size(GSTATE.FIELDX, 2);

% ---- everything up to the plate draw: step-size policy, flag, birefringence parameters, unit conversions,
%      front-end options, dispersion vectors (fiber_setup.m, shared with dbp.m)
[s, x] = fiber_setup(x, flag, nargout > 0);
fls = s.fls;
tolflag = s.tolflag;
ltol = s.ltol;
dphimaxt = s.dphimaxt;
dzmaxt = s.dzmaxt;
isy = s.isy;
vector = s.vector;
manakov = s.manakov;
ispmf = s.ispmf;
nplates = s.nplates;
alphalin = s.alphalin;
b30 = s.b30;
b1 = s.b1;
gam = s.gam;
dch = s.dch;
prec = s.prec;
resident = s.resident;
betat = s.betat;
db1 = s.db1;
scal = s.scal;

% ---- birefringence: the waveplates
if fls(2)
    if ispmf                                     % user-defined plates (e.g. a PMF)
        brf.db0 = x.db0;
        brf.theta = x.theta;
        brf.epsilon = x.epsilon;
    else                                         % random plates, three uniform draws in this order
        brf.db0 = rand(nplates, 1) * 2 * pi - pi;
        brf.theta = rand(nplates, 1) * pi - 0.5 * pi;
        brf.epsilon = 0.5 * asin(rand(nplates, 1) * 2 - 1);
    end
    brf.dgd = x.dgd;
    if ~isy                                      % (isy keeps its value: the DELAY / DISP rows below follow it)
        GSTATE.FIELDY = zeros(size(GSTATE.FIELDX));
        warning('optilux:fiber', ['You are working with two polarizations ', ...
            'but in create_field you initialized just one polarization']);
    end
else
    brf.db0 = 0;
    brf.theta = 0;
    brf.epsilon = 0;
end

% ---- side effects on the global state
nrow = 1 + isy;
GSTATE.DELAY = GSTATE.DELAY + ones(nrow, 1) * (x.length * GSTATE.SYMBOLRATE * b1);
GSTATE.DISP = GSTATE.DISP + ones(nrow, 1) * (fls(1) * dch * x.length * 1e-3);

% ---- the propagation loop: one gateway call for each of the three dispatches
P = [dzmaxt, dphimaxt, alphalin, x.length, nplates, double(manakov)];
if vector
    if tolflag == 2
        error('adaptive step available in absence of polarization effects');
    end
    plates = [];
    if fls(2)
        plates = [brf.db0(:), brf.theta(:), brf.epsilon(:)];
    end
    [GSTATE.FIELDX, GSTATE.FIELDY, firstdz, ncycle] = ssfm_mex('fiber', GSTATE.FIELDX, GSTATE.FIELDY, ...
        betat, db1, P, gam, fls, plates, scal, [0, prec, resident]);
    brf.lcorr = x.length / nplates;
    brf.betat = betat;
    brf.db1 = db1;
    if nargout
        zbrf = brf;
    end
else
    [GSTATE.FIELDX, uy, firstdz, ncycle] = ssfm_mex('fiber', GSTATE.FIELDX, [], betat, db1, P, gam, fls, [], scal, ...
        [1, prec, resident, tolflag, ltol, 0.9]);
end

% ---- summary block of the simulation log (same text as the toolbox writes)
if GSTATE.PRINT
    if alphalin == 0
        leff = x.length;
    else
        leff = (1 - exp(-alphalin * x.length)) / alphalin;
    end
    if ncol == 1
        gamprint = gam * ones(1, GSTATE.NCH);
    else
        gamprint = gam;
    end
    ld = Inf * ones(1, GSTATE.NCH);
    for k = 1:GSTATE.NCH
        if dch(k) ~= 0
            ld(k) = 1 / (GSTATE.SYMBOLRATE^2 * abs(x.lambda^2 / 2 / pi / c0 * dch(k) * 1e-6));
        end
    end
    lnl = 1 ./ (gam .* GSTATE.POWER);
    if b30 ~= 0
        lds = 1 / (GSTATE.SYMBOLRATE^3 * abs(b30));
    else
        lds = Inf;
    end
    loc_delay = x.length * GSTATE.SYMBOLRATE * b1;
    fid = fopen([GSTATE.DIR, '/simul_out'], 'a');
    fprintf(fid, '========================================\n');
    fprintf(fid, '===              fiber               ===\n');
    fprintf(fid, '========================================\n\n');
    fprintf(fid, 'Fiber parameters:\n\n');
    fprintf(fid, 'Length:%17.3f  [km]\n', x.length * 1e-3);
    fprintf(fid, 'Attenuation:%12.2f  [dB/km] (Leff = %7.3f [km])\n', x.alphadB, leff * 1e-3);
    fprintf(fid, 'lambda of Dc:%11.2f  [nm]\n', x.lambda);
    fprintf(fid, 'Dc:%21.4f  [ps/nm/km]\n', x.disp);
    fprintf(fid, 'Slope:%18.4f  [ps/nm^2/km]\n', x.slope);
    fprintf(fid, 'n2:%21.2e  [m^2/W]\n', x.n2);
    fprintf(fid, 'Aeff:%19.2f  [um^2]\n\n', x.aeff);
    if fls(2)
        fprintf(fid, 'DGD:%12.4f  [bits]\n', x.dgd);
        fprintf(fid, '# plates:%d  \n', x.nplates);
        if manakov
            fprintf(fid, 'Manakov Equation: %s\n', 'yes');
        else
            fprintf(fid, 'Manakov Equation: %s\n', 'no');
        end
        if ispmf
            fprintf(fid, 'db0 = %8.2f, theta = %3.2f*pi, epsilon = %3.2f*pi\n', brf.db0(1), brf.theta(1) / pi, ...
                brf.epsilon(1) / pi);
        else
            fprintf(fid, 'Random birefringence\n');
        end
    end
    fprintf(fid, 'Propagation type: ''%s''\n\n', flag);
    if tolflag
        fprintf(fid, 'Local error x step: %.1e\n', x.ltol);
    end
    fprintf(fid, 'Max NL phase rotation x step: %-6.2g  [rad]\n', dphimaxt);
    fprintf(fid, 'Max step: %.2e  [m]\n', dzmaxt);
    fprintf(fid, 'Initial step: %.2e  (num. steps: %d)\n\n', firstdz, ncycle);
    fprintf(fid, 'Channel properties (Ld: disp. length. Lnl: NL length):\n\n');
    for k = 1:GSTATE.NCH
        fprintf(fid, 'ch. #%.2d: Dc = %.4f  [ps/nm/km]   (Ld = %3.2e [km])\n', k, dch(k), ld(k) * 1e-3);
        fprintf(fid, '\t gamma = %.3e [1/mW/km] (Lnl = %3.2e [km])\n', gamprint(k) * 1e3, lnl(k) * 1e-3);
        fprintf(fid, '\t sqrt(Ld/Lnl) = %.4f\n', sqrt(ld(k) / lnl(k)));
        fprintf(fid, '\t local delay = %.3f\n', loc_delay(k));
    end
    fprintf(fid, '\nSlope length Lds: %-3.2e  [km]\n', lds * 1e-3);
    fprintf(fid, '\nGlobal  delay (ch.1 -> %d)\n', GSTATE.NCH);
    for k = 1:GSTATE.NCH
        fprintf(fid, '%.3f  ', GSTATE.DELAY(k));
    end
    fprintf(fid, '\nGlobal cumulated dispersion [ps/nm] ');
    fprintf(fid, '(ch.1 -> %d)\n', GSTATE.NCH);
    for k = 1:GSTATE.NCH
        fprintf(fid, '%.3f  ', GSTATE.DISP(k));
    end
    fprintf(fid, '\n****************************************\n\n');
    fclose(fid);
end
