function [G,out] = cmtf_fun_AOADMM(Z,Znorm_const,G,fh,gh,lscalar,uscalar,options) %#ok<INUSL>
% Drop-in replacement of functions/cmtf_fun_AOADMM.m of the AO-ADMM data fusion framework: same signature, same
% outputs, the inner AO-ADMM loop runs on NVIDIA B200 GPUs through the C ABI of include/aoadmm.h (aoadmm_mex).
%
% Put this directory BEFORE the reference's functions/ directory on the MATLAB path:
%     addpath(genpath('.../AOADMM-DataFusionFramework/functions'))
%     addpath('.../matlab-code_b200/matlab', '-begin')
% cmtf_AOADMM.m:193 then calls this file instead of the MATLAB solver; nothing else changes: Z / options are built by
% the user script, constraints_to_prox and init_coupled_AOADMM_CMTF still run in MATLAB (cmtf_AOADMM.m:30-53).
%
% fh, gh, lscalar, uscalar are [] for the Frobenius loss (cmtf_AOADMM.m:158-161) and are not used.  Problems the device
% engine does not cover ('custom' constraints, non-Frobenius losses) raise the MATLAB error
% 'aoadmm:unsupported' (there is deliberately no CPU fallback: remove this directory from the path to run the
% reference's MATLAB solver).
% Engine options (fields of `options`, all optional): b200_gpus = number of B200s of this box the call uses (the
% tensors are cut into mode-3 slabs inside the library, one MATLAB process drives all of them), b200_shard_sparse =
% true (with b200_gpus > 1: sparse objects too are cut, into nonzero-balanced slabs of their last mode),
% b200_sparse_slices = true (PARAFAC2 objects whose slices are all sparse, MATLAB sparse or order-2 sptensor, run without
% densifying them; one GPU, no Z.miss on such an object), b200_dimtree,
% b200_mttkrp_precision, b200_fuse_inner, b200_graph, b200_heldout{p} = an sptensor / sparse matrix of entries of object p
% withheld from training (with their true values; object p needs Z.miss): out.heldout_sse{p} is then the held-out SSE
% after outer iterations 0..OuterIterations.  b200_heldout_patience = P (needs b200_heldout): early stopping on the summed
% held-out SSE; G and the f_* values are those of the best iteration out.heldout_best_iter, and out.exit_flag is
% 'heldoutStop' when the held-out rule ended the run (include/aoadmm.h states the rule).
    % hand the gateway plain numeric arrays: X.data of a Tensor Toolbox tensor shares its memory with X (copy-on-write),
    % whereas mxGetProperty inside a MEX file would deep-copy the whole tensor
    for p = 1:numel(Z.object)
        Z.object{p} = unwrap_data(Z.object{p});
        if isfield(Z,'miss') && numel(Z.miss) >= p && ~isempty(Z.miss{p})
            Z.miss{p} = unwrap_data(Z.miss{p});
        end
    end
    heldout = isfield(options,'b200_heldout');
    if heldout
        options.b200_heldout = unwrap_data(options.b200_heldout);
    end
    [G,out] = aoadmm_mex(Z, Znorm_const, G, options);
    if heldout   % one history per object: a cell, empty where an object has no held-out set
        hs = out.heldout_sse;
        out.heldout_sse = cell(1, size(hs,2));
        for p = 1:numel(options.b200_heldout)
            if ~isempty(options.b200_heldout{p}), out.heldout_sse{p} = hs(:,p).'; end
        end
    else
        out = rmfield(out, 'heldout_sse');
    end
    if ~isfield(options,'b200_heldout_patience') || options.b200_heldout_patience == 0
        out = rmfield(out, 'heldout_best_iter');
    end
    if out.non_finite_mode > 0
        warning('aoadmm:nonFinite', 'a residual of the inner ADMM loop of mode %d was NaN/Inf (a factor or dual of norm 0)', out.non_finite_mode);
    end
    if isfield(options,'Display') && (strcmp(options.Display,'iter') || strcmp(options.Display,'final'))
        % the table of cmtf_fun_AOADMM.m:44-59, :462-468, :498-504 printed from the returned history
        fprintf(1,' Iter  f total      f tensors      f couplings    f constraints    f PAR2 couplings\n');
        fprintf(1,'------ ------------ -------------  -------------- ---------------- ----------------\n');
        n = numel(out.func_val_conv);
        step = 1; if isfield(options,'DisplayIters'), step = options.DisplayIters; end
        rows = n;
        if strcmp(options.Display,'iter'), rows = unique([1, 1+step:step:n, n]); end
        for i = rows
            ft = out.func_val_conv(i); fc = out.func_coupl_conv(i); fz = out.func_constr_conv(i); fp = out.func_PAR2_coupl(i);
            fprintf(1,'%6d %12f %12f %12f %17f %12f\n', i-1, ft+fc+fz+fp, ft, fc, fz, fp);
        end
    end
end

function X = unwrap_data(X)
    if iscell(X)
        for k = 1:numel(X), X{k} = unwrap_data(X{k}); end
    elseif isa(X,'sptensor')
        % sparse objects stay sparse: the gateway hands them to aoadmm_create_sparse (1-based subscripts)
        X = struct('subs',double(X.subs),'vals',double(X.vals),'size',X.size);
    elseif issparse(X)
        [i,j,v] = find(X);
        X = struct('subs',[i j],'vals',full(v),'size',size(X));
    elseif isa(X,'tensor')
        X = X.data;
    end
end
