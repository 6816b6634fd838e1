function matches = featureMatchingPairwise(input, allDescriptors, numImg)
    %FEATUREMATCHINGPAIRWISE  Drop-in replacement of PP/featureMatching/featureMatchingPairwise.m.
    %   Runs getMatches' matchFeaturesScratch branch (Unique = true) for every image pair i<j on the GPU in one call.
    %   input.Matchingmethod 'Exhaustive', or 'Approximate' with input.ApproxFloatNNMethod 'subsetpdist2' (the
    %   inputs.m default) / 'kdtree' (Euclidean searches, matchFeaturesScratch.m:142-155) / 'pca2nn' (PCA-48 + cosine, :130-141).
    %   (The MathWorks matchFeatures branch, input.useMATLABFeatureMatch = 1, is closed source; with this file on the
    %   path the scratch semantics are used and a warning says so.)
    %   input.apsGPUs (optional, e.g. 1:gpuDeviceCount): spread the image pairs over these GPUs (gpuDevice numbering)
    %   from this one process instead of parfor workers; the match lists are identical to the one-GPU call.
    arguments
        input struct
        allDescriptors cell
        numImg (1, 1) {mustBeNumeric, mustBeFinite, mustBePositive}
    end
    % Nothing may change the match lists silently: input.apsAcceptScratchSemantics = 1 acknowledges.
    accept = isfield(input, 'apsAcceptScratchSemantics') && input.apsAcceptScratchSemantics;
    if ~accept && isfield(input, 'useMATLABFeatureMatch') && input.useMATLABFeatureMatch == 1
        warning('apsmatch:semantics', ['input.useMATLABFeatureMatch = 1 selects MathWorks matchFeatures in the ' ...
            'reference; this GPU path runs the matchFeaturesScratch semantics (featureMatchingPairwise.m:108-117).']);
    end
    method = 0;                                          % aps_method: 0 exhaustive, 1 subsetpdist2, 2 kdtree, 3 pca2nn
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
    if isfield(input, 'apsGPUs')
        matches = aps_featureMatching_mex('pairwise', allDescriptors, numImg, input.Matchingthreshold, ...
            input.Ratiothreshold, method, double(input.apsGPUs));
    else
        matches = aps_featureMatching_mex('pairwise', allDescriptors, numImg, input.Matchingthreshold, input.Ratiothreshold, method);
    end
end
