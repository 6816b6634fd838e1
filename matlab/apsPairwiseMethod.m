function method = apsPairwiseMethod(input)
    %APSPAIRWISEMETHOD  aps_method of the pairwise matcher input selects (0 exhaustive, 1 subsetpdist2, 2 kdtree,
    %   3 pca2nn; matchFeaturesScratch.m:116-163), for featureMatchingPairwiseSets and pairwiseImageMatchingSets.  Warns
    %   when input.useMATLABFeatureMatch = 1 asks for MathWorks matchFeatures, which the GPU path does not run.
    % Nothing may change the match lists silently: input.apsAcceptScratchSemantics = 1 acknowledges.
    accept = isfield(input, 'apsAcceptScratchSemantics') && input.apsAcceptScratchSemantics;
    if ~accept && isfield(input, 'useMATLABFeatureMatch') && input.useMATLABFeatureMatch == 1
        warning('apsmatch:semantics', ['input.useMATLABFeatureMatch = 1 selects MathWorks matchFeatures in the ' ...
            'reference; this GPU path runs the matchFeaturesScratch semantics (featureMatchingPairwise.m:108-117).']);
    end
    method = 0;
    if isfield(input, 'Matchingmethod') && strcmpi(input.Matchingmethod, 'Approximate')
        nn = 'pca2nn';                                   % parser default, matchFeaturesScratch.m:75
        if isfield(input, 'ApproxFloatNNMethod'); nn = lower(char(input.ApproxFloatNNMethod)); end
        switch nn
            case 'subsetpdist2'
                method = 1;
            case 'kdtree'
                method = 2;
            case 'pca2nn'
                method = 3;
            otherwise
                error('Select a approximate method');
        end
    end
end
