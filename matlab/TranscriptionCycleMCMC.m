function TranscriptionCycleMCMC(varargin)
%Drop-in for the reference's TranscriptionCycleMCMC.m with the per-cell DRAM
%fits running on the GPU engine (libtcmcmc, through tcmcmc_mex).
%
%Same variable arguments, same defaults and the same output files / struct
%layouts as the reference; 'numParPools' is the number of GPUs to use.
%The parfor body of the reference (per-cell set-up, mcmcrun, summaries,
%best-fit curves) is replaced by ONE call into the engine for all cells.
%New optional arguments: 'files' (cell array of dataset names: skips the
%listdlg dialog, for headless use), 'seed', 'saveChains', 'previousResults'
%(results file of an earlier fit, for 'loadPrevious') and 'numChains'
%(default 1): with numChains > 1 every cell gets that many independent
%chains from independent random starts; MCMCresults pools them (pooled mean,
%pooled population std), MCMCchain concatenates them chain after chain, and
%the extra variable MCMCdiagnostics (cell_index, numChains, Rhat, n_eff,
%Rhat_max: Gelman-Rubin across the chains of a cell) is saved next to
%MCMCresults.  With numChains = 1 the outputs are exactly the reference's.
%'thin' (default 1): MCMCchain keeps every thin-th row (rows n_burn,
%n_burn+thin, ... and s2chain rows 1, 1+thin, ...), a regular subsample of
%the same chain stored on the GPU, and the raw-chain file carries the scalar
%thin; MCMCresults still summarise every row.

%% Variable inputs (defaults of the reference code)
fileDir = pwd; saveLoc = pwd; numParPools = 8; n_burn = 10000; n_steps = 20000;
ratePriorWidth = 50; t_start = 0; t_end = Inf; loadPrevious = false;
construct = 'P2P-MS2v5-LacZ-PP7v4'; files_arg = {}; seed = 20201028; saveChains = true;
prevFile = ''; numChains = 1; thin = 1;
for i = 1:length(varargin)
    if ~(ischar(varargin{i}) || isstring(varargin{i})), continue; end
    switch lower(char(varargin{i}))
        case 'filedir', fileDir = varargin{i+1};
        case 'saveloc', saveLoc = varargin{i+1};
        case 'numparpools', numParPools = varargin{i+1};
        case 'n_burn', n_burn = varargin{i+1};
        case 'n_steps', n_steps = varargin{i+1};
        case 'ratepriorwidth', ratePriorWidth = varargin{i+1};
        case 't_start', t_start = varargin{i+1};
        case 't_end', t_end = varargin{i+1};
        case 'loadprevious', loadPrevious = true;      %presence only, as in the reference
        case 'construct', construct = varargin{i+1};
        case 'files', files_arg = varargin{i+1};
        case 'seed', seed = varargin{i+1};
        case 'savechains', saveChains = varargin{i+1};
        case 'previousresults', prevFile = varargin{i+1};
        case 'numchains', numChains = varargin{i+1};
        case 'thin', thin = varargin{i+1};
    end
end
C = tcmcmc_constructs(construct);   %same table as GetFluorFromPolPos.m; errors on unknown names
if ~(isscalar(thin) && isnumeric(thin) && thin >= 1 && thin == round(thin))
    error('TranscriptionCycleMCMC:thin', '''thin'' must be an integer >= 1');
end

%% Choose datasets (dialog only when a display exists and no 'files' given)
files = dir(fullfile(fileDir, '*.mat')); names = {files.name};
if ~isempty(files_arg)
    s = find(ismember(names, files_arg));
elseif usejava('desktop')
    [s, ~] = listdlg('PromptString', 'Select a dataset:', 'SelectionMode', 'multiple', 'ListString', names);
else
    s = 1:numel(names);
end

for k = 1:length(s)
    dat = load(fullfile(files(s(k)).folder, names{s(k)}));
    if ~isfield(dat, 'data'), continue; end
    data = dat.data; Ncells = length(data); DatasetName = data(1).name;
    prev = [];
    if loadPrevious
        P = load(prevFile); prev = P.MCMCresults;       %results file in this same layout
    end
    %per-cell set-up: truncation, x0, J0, bounds, priors (reference lines 163-255)
    cells = struct('time', {}, 'MS2', {}, 'PP7', {}); keep = [];
    for c = 1:Ncells
        t = data(c).time; i0 = find(t >= t_start, 1, 'first'); i1 = find(t < t_end, 1, 'last');
        if loadPrevious && ~any([prev.cell_index] == c), continue; end
        keep(end+1) = c; %#ok<AGROW>
        cells(end+1) = struct('time', t(i0:i1), 'MS2', data(c).MS2(i0:i1), 'PP7', data(c).PP7(i0:i1)); %#ok<AGROW>
    end
    n = numel(keep); Nmax = max(arrayfun(@(q) numel(q.time), cells)); ld = 7 + Nmax;
    chainCell = repelem(1:n, numChains); nch = numel(chainCell);      %chains of a cell are consecutive columns
    x0 = zeros(ld, nch); J0 = ones(ld, nch); low = zeros(ld, nch); upp = zeros(ld, nch); mu = zeros(ld, nch); sg = inf(ld, nch);
    for j = 1:nch
        q = chainCell(j); t = cells(q).time; N = numel(t); np = 7 + N;
        if loadPrevious
            v0 = prev([prev.cell_index] == keep(q)).mean_v; v_step = 0.0000001; vl = v0 - 0.00001; vu = v0 + 0.00001;
        else
            v0 = 1 + 2*rand; v_step = 0.05; vl = 0; vu = 10;
        end
        x0(1:np, j) = [v0, 4*rand, 4*rand, 10, 5, rand, 15, normrnd(0, 3, 1, N)]';   %[v tau ton MS2b PP7b A R dR]
        J0(1:np, j) = [v_step, 0.1, t(end)-t(end-1), 1, 1, 0.05, 0.5, 0.5*ones(1, N)]';
        low(1:np, j) = [vl, 0, 0, 0, 0, 0, 0, -30*ones(1, N)]';
        upp(1:np, j) = [vu, 20, 10, 50, 50, 1, 40, 30*ones(1, N)]';
        sg(8:np, j) = ratePriorWidth;
    end
    opts = struct('n_steps', n_steps, 'n_burn', n_burn, 'numGPUs', numParPools, 'seed', seed, 'saveChains', saveChains, ...
        'thin', thin);
    if numChains > 1, opts.chainCell = chainCell; end
    out = tcmcmc_mex('fit', C, cells, opts, x0, J0, low, upp, mu, sg);

    %% Pool the chains of a cell (identity with one chain) and pack the reference's structures (field order of lines 149-157)
    nrow = n_steps - n_burn + 1;
    pm = zeros(ld, n); ps = zeros(ld, n); psig = zeros(2, n);
    MCMCdiagnostics = struct('cell_index', {}, 'numChains', {}, 'Rhat', {}, 'n_eff', {}, 'Rhat_max', {});
    for q = 1:n
        cols = (q-1)*numChains + (1:numChains); N = numel(cells(q).time); np = 7 + N;
        m = out.mean(:, cols); sd = out.std(:, cols);
        pm(:, q) = mean(m, 2);
        ps(:, q) = sqrt(mean(sd.^2, 2) + var(m, 1, 2));              %within + between, population normalisation
        psig(1, q) = sqrt(mean(out.sig(1, cols).^2));
        if numChains == 1, psig(2, q) = out.sig(2, cols); else, psig(2, q) = sqrt(mean(out.sig(2, cols).^2)); end
        if numChains > 1
            W = mean(sd(1:np, :).^2, 2) * nrow/(nrow-1); B = nrow * var(m(1:np, :), 0, 2);
            Vp = (nrow-1)/nrow * W + B/nrow;
            Rhat = sqrt(Vp ./ W); neff = min(numChains*nrow*Vp./B, numChains*nrow);
            Rhat(~(W > 0)) = NaN; neff(~(W > 0)) = NaN;
            MCMCdiagnostics(q) = struct('cell_index', keep(q), 'numChains', numChains, 'Rhat', Rhat', 'n_eff', neff', ...
                'Rhat_max', max(Rhat(1:7)));
        end
    end
    if numChains > 1
        sim = tcmcmc_mex('forward', C, cells, pm);                   %best-fit curves at the pooled means (lines 307-309)
    else
        sim = out;
    end
    MCMCchain = struct('v_chain', {}, 'ton_chain', {}, 'A_chain', {}, 'tau_chain', {}, 'MS2_basal_chain', {}, ...
        'PP7_basal_chain', {}, 'R_chain', {}, 'dR_chain', {}, 's2chain', {});
    MCMCresults = struct('mean_v', {}, 'sigma_v', {}, 'mean_ton', {}, 'sigma_ton', {}, 'mean_A', {}, 'sigma_A', {}, ...
        'mean_tau', {}, 'sigma_tau', {}, 'mean_MS2_basal', {}, 'sigma_MS2_basal', {}, 'mean_PP7_basal', {}, ...
        'sigma_PP7_basal', {}, 'mean_R', {}, 'sigma_R', {}, 'mean_dR', {}, 'sigma_dR', {}, 'mean_sigma', {}, ...
        'sigma_sigma', {}, 'cell_index', {}, 'ApprovedFits', {});
    MCMCplot = struct('t_plot', {}, 'MS2_plot', {}, 'PP7_plot', {}, 'simMS2', {}, 'simPP7', {});
    for q = 1:n
        N = numel(cells(q).time); m = pm(:, q); sd = ps(:, q);
        if saveChains
            cols = (q-1)*numChains + (1:numChains);
            ch = reshape(permute(out.chain(:, :, cols), [2 3 1]), [], ld);   %rows n_burn:thin:n_steps, chain after chain
            s2 = reshape(out.s2chain(:, cols), [], 1);
            MCMCchain(q) = struct('v_chain', ch(:,1), 'ton_chain', ch(:,3), 'A_chain', ch(:,6), 'tau_chain', ch(:,2), ...
                'MS2_basal_chain', ch(:,4), 'PP7_basal_chain', ch(:,5), 'R_chain', ch(:,7), 'dR_chain', ch(:,8:7+N), ...
                's2chain', s2);
        end
        R = struct('mean_v', m(1), 'sigma_v', sd(1), 'mean_ton', m(3), 'sigma_ton', sd(3), 'mean_A', m(6), 'sigma_A', sd(6), ...
            'mean_tau', m(2), 'sigma_tau', sd(2), 'mean_MS2_basal', m(4), 'sigma_MS2_basal', sd(4), 'mean_PP7_basal', m(5), ...
            'sigma_PP7_basal', sd(5), 'mean_R', m(7), 'sigma_R', sd(7), 'mean_dR', m(8:7+N)', 'sigma_dR', sd(8:7+N)', ...
            'mean_sigma', psig(1, q), 'sigma_sigma', psig(2, q), 'cell_index', keep(q), 'ApprovedFits', 0);
        if loadPrevious, R.ApprovedFits = prev([prev.cell_index] == keep(q)).ApprovedFits; end
        MCMCresults(q) = R;
        MCMCplot(q) = struct('t_plot', cells(q).time, 'MS2_plot', cells(q).MS2, 'PP7_plot', cells(q).PP7, ...
            'simMS2', sim.simMS2(1:N, q)', 'simPP7', sim.simPP7(1:N, q)');
    end
    filename = [date, '-', DatasetName];
    if numChains > 1
        save(fullfile(saveLoc, [filename, '.mat']), 'MCMCresults', 'MCMCplot', 'DatasetName', 'MCMCdiagnostics');
    else
        save(fullfile(saveLoc, [filename, '.mat']), 'MCMCresults', 'MCMCplot', 'DatasetName');
    end
    if saveChains
        w = whos('MCMCchain');
        extra = {};
        if thin > 1, extra = {'thin'}; end                           %the reference's variables alone when every row is kept
        if w.bytes < 2^31 - 2^24
            save(fullfile(saveLoc, [filename, '_RawChain.mat']), 'MCMCchain', extra{:});    %the reference's file (MAT v5/v7)
        else
            %plain save cannot hold a variable of 2 GiB (the reference's own defaults on TestData give 3.1 GB): parts of
            %whole cells below the limit + an index, the layout of the Python host (LoadRawChains.m reads both)
            full = MCMCchain; sz = arrayfun(@(c) getfield(whos('c'), 'bytes'), full); %#ok<GFLD>
            lim = 2^31 - 2^24; first = 1; k = 0; parts = {}; partOf = zeros(1, numel(full));
            while first <= numel(full)
                last = first; acc = sz(first);
                while last < numel(full) && acc + sz(last+1) <= lim, last = last + 1; acc = acc + sz(last); end
                k = k + 1; MCMCchain = full(first:last); firstCell = first; lastCell = last; part = k; %#ok<NASGU>
                parts{k, 1} = sprintf('%s_RawChain_part%d.mat', filename, k); %#ok<AGROW>
                save(fullfile(saveLoc, parts{k}), 'MCMCchain', 'firstCell', 'lastCell', 'part', extra{:});
                partOf(first:last) = k; first = last + 1;
            end
            MCMCchainParts = parts; MCMCchainPartOfCell = partOf; nParts = k; %#ok<NASGU>
            save(fullfile(saveLoc, [filename, '_RawChain.mat']), 'MCMCchainParts', 'MCMCchainPartOfCell', 'nParts', extra{:});
        end
    end
end
disp(['MCMC analysis complete. Information stored in: ', saveLoc]);
end
