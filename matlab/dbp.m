function dbp(x, flag, options)
%DBP  Digital backpropagation of a link on the received field (device side; the toolbox has no DBP).
%   DBP(X,FLAG,OPTIONS) runs GSTATE.FIELDX / FIELDY back through OPTIONS.nspan spans of the fiber X, each
%   followed by an amplifier: dispersion, nonlinearity and loss negated, spans last first, the amplifier gain
%   undone before each span.  X and FLAG are what FIBER takes, with the same flag check.  A field without
%   FIELDY runs the scalar path, where the 'x' flag backpropagates the cross-phase modulation of all columns.
%   The whole link is one call of the MEX gateway ssfm_mex('dbp', ...) on the field the previous in-line device
%   left in HBM, so  for k=1:Nspan, fiber(x,flag); ampliflat(G,'gain'); end; dbp(x,flag,opt)  uploads the field
%   once.  There is no CPU fallback.
%
%   OPTIONS (a struct, all fields optional):
%     nspan      number of spans (default 1)
%     gain       gain [dB] of the amplifier after every span, as AMPLIFLAT(GAIN,'gain') takes it (absent: none)
%     steps      uniform steps per span (default 1), or
%     steplen    the steps in forward order: one span's steps, used for every span, or with
%     spansteps  (1 x nspan step counts) all spans' steps concatenated
%     xi         fraction of the nonlinear coefficient backpropagated (default 1)
%     brf        the struct FIBER returned (every span the same plates) or a cell of nspan of them in forward
%                span order; needs the 'p' flag: PMD-aware DBP through those waveplates
%     ich, decim single-channel DBP of channel ICH of a one-column ('unique') field, on Nfft/DECIM samples;
%                afterwards the field holds that channel alone, on its own bins
%     filter_bw  filtered DBP: one-sided -3 dB bandwidth [GHz] of a Gaussian low-pass on the intensity of every
%                nonlinear step (absent: none)
%     taps       enhanced split-step DBP: a row or column of 2K+1 <= 65 real FIR taps, taps(K+1) at lag 0, applied
%                circularly on the time grid to the intensity of every nonlinear step (absent or []: none; not with
%                filter_bw).  With decim the grid is the channel's Nfft/DECIM samples: one tap spans DECIM samples
%
%   Without brf the 'p' flag is dropped: no plates are drawn and nothing is taken from the RAND stream.  The
%   nonlinear model stays the one FIBER used: Manakov when x.manakov is 'yes' and the flag has 'p', else the
%   CNLSE.  With xi = 1 and the forward run's own steps, DBP inverts a noise-free link up to rounding.
%   GSTATE.FIELDX / FIELDY are updated (FIELDY stays empty on the scalar path); GSTATE.DELAY and GSTATE.DISP are
%   left untouched.  PMXOPT.precision, PMXOPT.resident and PMXOPT.scalar act as for FIBER.

global CONSTANTS GSTATE PMXOPT

if nargin < 2
    error('Missing propagation type');
end
if nargin < 3 || ~isstruct(options)
    options = struct();
end
if ~ischar(flag) || length(flag) ~= 4
    error('wrong flag. E.g. flag can be ''g---'',''gp--'',''-s--'', etc');
end
f = lower(flag);
ncol = size(GSTATE.FIELDX, 2);

% ---- the link
nspan = 1;
if isfield(options, 'nspan')
    nspan = options.nspan;
end
gain = 0;
if isfield(options, 'gain')
    gain = 10^(options.gain * 0.1);
end
steps = 1;
steplen = [];
spansteps = [];
if isfield(options, 'steplen')
    if isfield(options, 'steps')
        error('give steps_per_span or step_len, not both');
    end
    steps = 0;
    steplen = options.steplen(:)';
    if isfield(options, 'spansteps')
        spansteps = options.spansteps(:)';
    end
elseif isfield(options, 'steps')
    steps = options.steps;
end
xi = 1;
if isfield(options, 'xi')
    xi = options.xi;
end

% ---- single-channel DBP: the channel's offset in bins, as receiver_cohmix computes its ndfn
band = [];
if isfield(options, 'decim')
    if ~isfield(options, 'ich')
        error('dbp: single-channel DBP (decim) needs the channel ich');
    end
    ich = options.ich;
    if ich < 1 || ich > GSTATE.NCH
        error('The channel does not exist');
    end
    if ncol ~= 1
        error('dbp: single-channel DBP takes a field holding every channel in one column (''unique'')');
    end
    shift = 0;
    if GSTATE.NCH > 1
        maxl = max(GSTATE.LAMBDA);
        minl = min(GSTATE.LAMBDA);
        lamc = 2 * maxl * minl / (maxl + minl);
        minfreq = GSTATE.FN(2) - GSTATE.FN(1);
        deltafn = CONSTANTS.CLIGHT * (1 / lamc - 1 / GSTATE.LAMBDA(ich));
        shift = round(deltafn ./ GSTATE.SYMBOLRATE / minfreq);
    end
    band = [shift, options.decim];
elseif isfield(options, 'ich')
    error('dbp: ich selects a channel for single-channel DBP and needs decim');
end

% ---- the fiber: fiber.m's scalars; without brf the 'p' flag is dropped and no plates are drawn
pflag = f(2) == 'p';
pmd = isfield(options, 'brf');
if pmd && ~pflag
    error('dbp: brf (PMD-aware DBP) needs the ''p'' flag');
end
if ~pmd && pflag
    f = [f(1), '-', f(3:4)];
end
[s, x] = fiber_setup(x, f, false);
plates = [];
if pmd
    brf = options.brf;
    if iscell(brf) && length(brf) ~= nspan
        error('dbp: brf must be one struct or a list of nspan of them');
    end
    for k = 1:nspan                              % span k: rows (k-1)*nplates+1 .. k*nplates, forward order
        if iscell(brf)
            b = brf{k};
        else
            b = brf;
        end
        if numel(b.theta) ~= s.nplates
            error('dbp: brf has %d plates, the fiber %d', numel(b.theta), s.nplates);
        end
        plates = [plates; b.db0(:), b.theta(:), b.epsilon(:)];
    end
end
fls = s.fls;
if fls(4) && s.vector
    error('The CNLSE with separate fields is not yet implemented');
end
if s.vector && ~s.isy                            % the 'p' flag on a single-polarization field
    GSTATE.FIELDY = zeros(size(GSTATE.FIELDX));
end
manakov = pflag && isfield(x, 'manakov') && strcmp(x.manakov, 'yes');

% ---- the backpropagation: one gateway call for the whole link
P = [s.dzmaxt, s.dphimaxt, s.alphalin, x.length, s.nplates, double(manakov)];
D = [nspan, gain, steps, xi, double(pmd)];
if isfield(options, 'filter_bw')                 % in bins of GSTATE.FN
    D = [D, options.filter_bw * GSTATE.NSYMB / GSTATE.SYMBOLRATE];
end
taps = [];                                       % the gateway's optional last argument
if isfield(options, 'taps') && ~isempty(options.taps)
    taps = double(options.taps(:)');
    if mod(numel(taps), 2) ~= 1 || numel(taps) > 65
        error('pmx_dbp_set_taps: ntaps must be odd and at most 65 (0: no taps), got %d', numel(taps));
    end
    bad = find(isnan(taps) | isinf(taps));
    if ~isempty(bad)
        error('pmx_dbp_set_taps: tap %d is not finite', bad(1) - 1);
    end
    if isfield(options, 'filter_bw') && options.filter_bw ~= 0
        error('pmx_dbp_set_taps: the plan has a filter bandwidth (pmx_dbp_set_filter); a plan takes one or the other');
    end
end
if s.vector && isempty(taps)
    [GSTATE.FIELDX, GSTATE.FIELDY] = ssfm_mex('dbp', GSTATE.FIELDX, GSTATE.FIELDY, s.betat, s.db1, P, s.gam, fls, ...
        plates, s.scal, D, steplen, spansteps, band, [0, s.prec, s.resident]);
elseif s.vector
    [GSTATE.FIELDX, GSTATE.FIELDY] = ssfm_mex('dbp', GSTATE.FIELDX, GSTATE.FIELDY, s.betat, s.db1, P, s.gam, fls, ...
        plates, s.scal, D, steplen, spansteps, band, [0, s.prec, s.resident], taps);
elseif isempty(taps)
    GSTATE.FIELDX = ssfm_mex('dbp', GSTATE.FIELDX, [], s.betat, s.db1, P, s.gam, fls, [], s.scal, D, steplen, ...
        spansteps, band, [1, s.prec, s.resident]);
else
    GSTATE.FIELDX = ssfm_mex('dbp', GSTATE.FIELDX, [], s.betat, s.db1, P, s.gam, fls, [], s.scal, D, steplen, ...
        spansteps, band, [1, s.prec, s.resident], taps);
end
