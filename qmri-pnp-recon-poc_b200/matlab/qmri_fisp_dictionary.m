function dict = qmri_fisp_dictionary(lut, seq, C, V)
% dict = qmri_fisp_dictionary(lut, seq, C [, V])
% A FISP-MRF dictionary simulated on the GPU, with the fields of dictionaries/real_fisp_cut*_dict/SVD_dict_FISP_cut*.mat
% (loaded at main_recon_tsmis_FFT.m:127-129 and main_synthesize_tsmis.m:50-54):
%   dict.D     K x C single, unit-norm rows d*V / norm(d*V)
%   dict.normD K x 1 single, norm(d*V)
%   dict.lut   K x 2 single, (T1, T2) in seconds: the atoms are simulated at exactly these values
%   dict.V     T x C double, top-C eigenvectors of the Gram matrix of all fingerprints, descending eigenvalues, each column's
%              entry of largest magnitude positive (the first one on a tie)
% seq: struct with flip_deg (T degrees), tr (T seconds), te (seconds), ti (seconds, or [] for no inversion).  The signal model
% is stated in include/qmri.h.  Pass V to project onto a given temporal basis instead (e.g. the one of a larger dictionary).
lut = single(lut);
if nargin < 4 || isempty(V)
    G = qmri_b200_mex('fisp_gram', lut, seq);
    [U, L] = eig((G + G') / 2);                 % G is exactly symmetric; eig then returns real eigenpairs
    [~, order] = sort(diag(L), 'descend');
    V = U(:, order(1:C));
    [~, peak] = max(abs(V), [], 1);
    s = sign(V(sub2ind(size(V), peak, 1:size(V, 2))));
    s(s == 0) = 1;
    V = V .* s;
end
[D, normD] = qmri_b200_mex('fisp_compress', lut, seq, double(V));
dict = struct('D', D, 'normD', normD, 'lut', lut, 'V', double(V));
end
