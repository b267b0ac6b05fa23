function [s, x] = fiber_setup(x, flag, vectors)
%FIBER_SETUP  The scalar set-up of a fiber, shared by FIBER and DBP (front-end helper, not a toolbox function).
%   [S,X] = FIBER_SETUP(X,FLAG,VECTORS) does what the toolbox's fiber.m does before its SSFM dispatch, in its
%   operation order, except for the draw of random waveplates and the side effects on GSTATE: the step-size policy,
%   the flag check, the birefringence parameters (number of plates, dgdrms, Manakov), the unit conversions, the
%   front-end options of PMXOPT, and the dispersion vectors betat / db1 (built when VECTORS is true or
%   PMXOPT.scalar is false) or the scalars the gateway rebuilds them from.  X is returned with the defaults fiber.m
%   fills in (dzmax, dphimax, nplates).  FIBER draws the plates after this call; DBP takes them from the brf structs
%   of the forward run and draws nothing.

global CONSTANTS GSTATE PMXOPT

c0 = CONSTANTS.CLIGHT;
ncol = size(GSTATE.FIELDX, 2);
nfft = GSTATE.NSYMB * GSTATE.NT;

% ---- step-size policy
if ~isfield(x, 'dzmax') || x.dzmax > x.length
    x.dzmax = x.length;
end
tolflag = 0;
ltol = 0;
if isfield(x, 'ltol')
    if ~isfield(x, 'dphimax')
        x.dphimax = Inf;
    end
    ltol = x.ltol;
    tolflag = 2;
    if isfield(x, 'dphiadapt') && x.dphiadapt
        tolflag = 1;
    end
end

% ---- flag -> [g p s x]
f = lower(flag);
if ~ischar(f) || length(f) ~= 4
    error('wrong flag. E.g. flag can be ''g---'',''gp--'',''-s--'', etc');
end
letters = 'gpsx';
fls = [0 0 0 0];
for k = 1:4
    if f(k) == letters(k)
        fls(k) = 1;
    elseif f(k) ~= '-'
        error('wrong flag. E.g. flag can be ''g---'',''gp--'',''-s--'', etc');
    end
end
if fls(4) && ncol == 1
    if ~fls(3)
        error(['flag ''', f, ''' available only for channels separated']);
    end
    fls(4) = 0;                                  % a single field has no cross-phase partner
end
onestep = ~fls(3) && ~fls(4);                    % linear flags: one step over the whole fiber
if ncol == 1 && fls(3) && ~fls(1) && ~fls(2)
    onestep = true;                              % pure SPM of one field has an exact solution
end
if onestep
    dphimaxt = Inf;
    dzmaxt = x.length;
else
    dphimaxt = x.dphimax;
    dzmaxt = x.dzmax;
end

% ---- birefringence (the plates themselves are drawn by the caller)
isy = ~isempty(GSTATE.FIELDY);
vector = fls(2) || isy;
given = 0;
if fls(2)
    manakov = isfield(x, 'manakov') && strcmp(x.manakov, 'yes');
    if ~isfield(x, 'dgd')
        error('Missing DGD in fiber');
    end
    given = isfield(x, 'db0') + isfield(x, 'theta') + isfield(x, 'epsilon');
    if given == 3                                % user-defined plates (e.g. a PMF)
        nplates = length(x.theta);
        x.nplates = nplates;
        dgdrms = x.dgd / nplates;
    elseif given == 0                            % random plates
        if ~isfield(x, 'nplates')
            x.nplates = 100;
        end
        nplates = x.nplates;
        dgdrms = sqrt((3 * pi) / 8) * x.dgd / sqrt(nplates);
    else
        error('Missing one of db0, theta or epsilon in fiber');
    end
    dgdrms = dgdrms / GSTATE.SYMBOLRATE;
else
    manakov = false;
    nplates = 1;
    dgdrms = 0;
end

% ---- unit conversions
alphalin = (log(10) * 1e-4) * x.alphadB;
b20 = -x.lambda^2 / 2 / pi / c0 * x.disp * 1e-6;
b30 = (x.lambda / 2 / pi / c0)^2 * (2 * x.lambda * x.disp + x.lambda^2 * x.slope) * 1e-6;
b30 = b30 * fls(1);
maxl = max(GSTATE.LAMBDA);
minl = min(GSTATE.LAMBDA);
lamc = 2 * maxl * minl / (maxl + minl);
w_i0 = 2 * pi * c0 * (1 ./ GSTATE.LAMBDA - 1 / x.lambda);
w_ic = 2 * pi * c0 * (1 ./ GSTATE.LAMBDA - 1 / lamc);
w_c0 = 2 * pi * c0 * (1 ./ lamc - 1 / x.lambda);
b1 = b20 * w_ic + 0.5 * b30 * (w_i0.^2 - w_c0^2);
if ncol == 1
    beta1 = 0;
    w_i0 = 2 * pi * c0 * (1 / lamc - 1 / x.lambda);
    gam = 2 * pi * x.n2 / (lamc * x.aeff) * 1e18;
else
    beta1 = b1;
    gam = 2 * pi * x.n2 ./ (GSTATE.LAMBDA * x.aeff) * 1e18;
end
beta2 = (b20 + b30 * w_i0) * fls(1);
dch = x.disp + x.slope * (GSTATE.LAMBDA - x.lambda);

% ---- front-end options
prec = 0;
resident = 1;
scalmode = 1;
if isstruct(PMXOPT)
    if isfield(PMXOPT, 'precision') && strcmp(PMXOPT.precision, 'f32')
        prec = 1;
    end
    if isfield(PMXOPT, 'resident')
        resident = double(PMXOPT.resident ~= 0);
    end
    if isfield(PMXOPT, 'scalar')
        scalmode = double(PMXOPT.scalar ~= 0);
    end
end

% ---- dispersion vectors (only built when they are returned or uploaded)
betat = [];
db1 = [];
if vectors || ~scalmode
    omega = 2 * pi * GSTATE.SYMBOLRATE * GSTATE.FN';
    betat = zeros(nfft, ncol);
    db1 = zeros(nfft, ncol);
    for k = 1:ncol
        betat(:, k) = omega * beta1(k) + 0.5 * omega.^2 * beta2(k) + omega.^3 * b30 / 6;
        if fls(2)
            db1(:, k) = dgdrms * omega;
        end
    end
end
scal = [];
if scalmode
    scal = [GSTATE.SYMBOLRATE, GSTATE.NSYMB, GSTATE.NT, b30, dgdrms, beta1(:)', beta2(:)'];
end

s.fls = fls;
s.tolflag = tolflag;
s.ltol = ltol;
s.dphimaxt = dphimaxt;
s.dzmaxt = dzmaxt;
s.isy = isy;
s.vector = vector;
s.manakov = manakov;
s.ispmf = (given == 3);
s.nplates = nplates;
s.dgdrms = dgdrms;
s.alphalin = alphalin;
s.b30 = b30;
s.b1 = b1;
s.gam = gam;
s.dch = dch;
s.prec = prec;
s.resident = resident;
s.betat = betat;
s.db1 = db1;
s.scal = scal;
