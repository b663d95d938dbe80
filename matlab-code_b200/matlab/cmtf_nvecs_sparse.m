function U = cmtf_nvecs_sparse(Z,n,r)
% cmtf_nvecs for a mode whose first object is sparse (an sptensor or a MATLAB sparse matrix; functions/cmtf_nvecs.m and
% the cmtf_nvecs.m shim refuse those): the r leading eigenvectors of X_(n)*X_(n)' with the unstored entries counted as
% zero, computed on the GPU through aoadmm_nvecs_sparse_mex (include/aoadmm.h: aoadmm_nvecs_sparse) without forming the
% n x n matrix.  Columns come in descending eigenvalue order, the entry of largest magnitude of each column positive.
% A mode of a dense object is refused (aoadmm:invalidArg): use cmtf_nvecs.
    P = length(Z.object);
    for p = 1:P
        i = find(Z.modes{p} == n, 1);
        if ~isempty(i)
            X = Z.object{p};
            if isa(X,'sptensor')
                S = struct('subs',double(X.subs),'vals',double(X.vals),'size',double(size(X)));
            elseif issparse(X)
                [a,b,v] = find(X);
                S = struct('subs',[a b],'vals',full(v),'size',size(X));
            else
                error('aoadmm:invalidArg','cmtf_nvecs_sparse needs a sparse object (use cmtf_nvecs for dense ones)');
            end
            U = aoadmm_nvecs_sparse_mex(S, i, r);
            return
        end
    end
    error('Mode %d is not part of any object.', n);
end
