function pbnlc(x, flag, options)
%PBNLC  Perturbation-based nonlinearity compensation of a link on the received field (device side; the toolbox has none).
%   PBNLC(X,FLAG,OPTIONS) compensates GSTATE.FIELDX / FIELDY for OPTIONS.nspan spans of the fiber X, each followed by
%   an amplifier: the all-pass step that undoes the dispersion of the whole link, then the first-order triplet
%   perturbation of the link (Mecozzi, Clausen & Shtaif 2000; Tao et al. 2011), formed at launch scale and subtracted
%   OPTIONS.xi times.  X and FLAG are what FIBER takes, with the same flag check; the nonlinear model is the one FIBER
%   used: Manakov when x.manakov is 'yes' and the flag has 'p', else the CNLSE.  One channel (GSTATE.NCH == 1), two
%   polarizations, one column, FP64.  The M counterpart of pmx.pbnlc (polmux_b200/pbnlc.py): one call of the MEX
%   gateway ssfm_mex('pbnlc', ...), in which the library computes the triplet table on the device (pmx_pb_table), on
%   the field the previous in-line device left in HBM, so  for k=1:Nspan, fiber(x,flag); ampliflat(G,'gain'); end;
%   pbnlc(x,flag,opt)  uploads the field once.  There is no CPU fallback.
%
%   OPTIONS (a struct, all fields optional):
%     nspan      number of spans (default 1)
%     gain       gain [dB] of the amplifier after every span, as AMPLIFLAT(GAIN,'gain') takes it (absent: none)
%     xi         fraction of the perturbation subtracted (default 1)
%     K          half-width of the triplet table, |m|, |n| <= K <= 128 (default 16)
%     prune      keep the entries with |C| >= prune*|C(0,0)| (default 0: all)
%     nquad      Gauss-Legendre nodes per span of the table's integral (default 32)
%     window     symbols of the circular window the table is computed on (default: the smallest power of two that
%                holds the pulse dispersed over the link plus 2K+8 symbols, at most the block)
%     pulse      the real pulse table (default: electricsource's raised-cosine pulse of NT samples per symbol, roll-off
%                0.2; with decim the transmit pulse band-passed and decimated with the channel, at NT/DECIM)
%     ich, decim single-channel PB-NLC of channel ICH of a one-column ('unique') field of any NCH, on Nfft/DECIM
%                samples (DECIM a power of two dividing NT); afterwards the field holds that channel alone, on its
%                own bins
%
%   GSTATE.FIELDX / FIELDY are updated; GSTATE.DELAY and GSTATE.DISP are left untouched.  PMXOPT.resident and
%   PMXOPT.scalar act as for FIBER; PMXOPT.precision = 'f32' is refused (FP64 fields only).

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
nt = GSTATE.NT;
nfft = GSTATE.NSYMB * GSTATE.NT;

% ---- single-channel PB-NLC: the channel's offset in bins, as dbp.m computes it
decim = 0;
shift = 0;
if isfield(options, 'decim')
    if ~isfield(options, 'ich')
        error('pbnlc: single-channel PB-NLC (decim) needs the channel ich');
    end
    ich = options.ich;
    if ich < 1 || ich > GSTATE.NCH
        error('The channel does not exist');
    end
    if ncol ~= 1
        error('pbnlc: single-channel PB-NLC takes a field holding every channel in one column (''unique'')');
    end
    decim = options.decim;
    q = decim;
    while q > 1 && mod(q, 2) == 0
        q = q / 2;
    end
    if decim < 2 || q ~= 1
        error('pmx_pb_channel_create: decim=%d, must be a power of two >= 2', decim);
    end
    if mod(nt, decim) ~= 0
        error('decim=%d must divide nt=%d: the channel keeps every symbol at nt/decim samples', decim, nt);
    end
    if GSTATE.NCH > 1
        maxl = max(GSTATE.LAMBDA);
        minl = min(GSTATE.LAMBDA);
        lamc = 2 * maxl * minl / (maxl + minl);
        minfreq = GSTATE.FN(2) - GSTATE.FN(1);
        deltafn = CONSTANTS.CLIGHT * (1 / lamc - 1 / GSTATE.LAMBDA(ich));
        shift = round(deltafn ./ GSTATE.SYMBOLRATE / minfreq);
    end
elseif isfield(options, 'ich')
    error('pbnlc: ich selects a channel for single-channel PB-NLC and needs decim');
elseif GSTATE.NCH ~= 1
    error('pbnlc: PB-NLC takes a field holding one channel (GSTATE.NCH == 1), got %d', GSTATE.NCH);
end
if isempty(GSTATE.FIELDY)
    error('pbnlc: PB-NLC takes two-polarization fields (FIELDY is empty)');
end
if ncol ~= 1
    error('pbnlc: PB-NLC takes one-column fields');
end

% ---- the options
nspan = 1;
if isfield(options, 'nspan')
    nspan = options.nspan;
end
if nspan < 1
    error('pbnlc: nspan must be >= 1');
end
g = 1;
if isfield(options, 'gain')
    g = 10^(options.gain * 0.1);
end
xi = 1;
if isfield(options, 'xi')
    xi = options.xi;
end
K = 16;
if isfield(options, 'K')
    K = options.K;
end
if K < 0 || K > 128
    error('pmx_pb_create: K=%d, |m| and |n| at most 128', K);
end
prune = 0;
if isfield(options, 'prune')
    prune = options.prune;
end
nquad = 32;
if isfield(options, 'nquad')
    nquad = options.nquad;
end
window = 0;
if isfield(options, 'window')
    window = options.window;
end

% ---- the fiber: fiber.m's scalars and the betat vector the table needs; the 'p' flag is dropped (no plates)
[s, x] = fiber_setup(x, [f(1), '-', f(3:4)], true);
if s.prec
    error('pmx_pb_create: FP64 fields only');
end
manakov = f(2) == 'p' && isfield(x, 'manakov') && strcmp(x.manakov, 'yes');
betat = s.betat(:, 1);

% ---- the table's grid: the link's, or the channel's (pbnlc.channel_setup, channel_pulse)
tbetat = betat;
tnt = nt;
band = [];
if decim
    M = nfft / decim;
    k = [0:M/2-1, -M/2:-1]';                            % the signed bins of the M grid, FFT order
    b = mod(k - shift, nfft) + 1;
    tbetat = betat(b);
    tbetat = tbetat - tbetat(1) - k .* (0.5 * (tbetat(2) - tbetat(M)));   % less the channel's phase and group delay
    tnt = nt / decim;
    band = [shift, decim];
end
if isfield(options, 'pulse')
    pulse = double(options.pulse(:));
else
    pulse = zeros(2 * nt, 1);                             % electricsource.m's raised cosine, roll-off 0.2, duty 1
    nl = round(0.5 * (1 - 0.2) * nt);
    nr = nt - nl - 1;
    pulse(nt+1:nt+nl) = 1;
    hperiod = nt - 2 * nl;
    if hperiod ~= 0
        ncos = nl:nr;
        pulse(ncos + nt + 1) = 0.5 * (1 + cos(pi / hperiod * (ncos - nl + 0.5)));
    end
    pulse(1:nt) = pulse(2*nt:-1:nt+1);
    if decim
        u = zeros(nfft, 1);
        u(mod((0:length(pulse)-1)' - length(pulse) / 2, nfft) + 1) = pulse;
        U = fft(u);
        v = real(ifft(U(mod(k, nfft) + 1) / decim));     % the band-pass at baseband, decimated
        L = min(16 * tnt, M);
        pulse = v(mod((0:L-1)' - L / 2, M) + 1);
    end
end

% ---- model weights, gamma and the launch scale (pbnlc.model_weights, scale_factor)
gam = s.gam(1);
if manakov
    W = [1, 1, 0, gam * 8 / 9];
else
    W = [1, 2 / 3, 1 / 3, gam];
end
scale = (exp(0.5 * s.alphalin * x.length) / sqrt(g))^nspan;
W = [W, xi, scale];

% ---- one gateway call: the all-pass step, the table on the device, the stage
P = [nspan, x.length, s.alphalin, tnt, K, nquad, window, prune];
[GSTATE.FIELDX, GSTATE.FIELDY] = ssfm_mex('pbnlc', GSTATE.FIELDX, GSTATE.FIELDY, betat, s.scal, tbetat, P, W, ...
    pulse, band, [s.prec, s.resident, s.fls(1)]);

