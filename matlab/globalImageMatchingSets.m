function [allMatchesSets, numMatchesSets, tformsSets, matchesSets] = globalImageMatchingSets(input, descSets, numImgs, keypointsSets)
    %GLOBALIMAGEMATCHINGSETS  featureMatchingGlobal followed by imageMatching over many independent image sets, in one
    %   GPU call.  Element b of each 1 x B output cell is exactly what
    %       matchesSets = featureMatchingGlobalSets(input, descSets, numImgs);
    %       [allMatchesSets, numMatchesSets, tformsSets] = imageMatchingSets(input, numImgs, keypointsSets, matchesSets);
    %   returns, and matchesSets (the fourth output, fetched only when asked for) is the putative lists of the first
    %   call.  The match lists stay on the GPU between the two stages (aps_globalImageMatching_mex -> libapsmatch.so);
    %   no CPU fallback.  keypointsSets{b}{i} has one row per row of descSets{b}{i}.
    arguments
        input (1, 1) struct
        descSets cell
        numImgs (1, :) double {mustBeInteger, mustBePositive}
        keypointsSets cell
    end
    if input.useMATLABImageMatching == 1 || ~strcmpi(input.imageMatchingMethod, 'ransac') || ...
            ~strcmpi(input.transformationType, 'projective')
        error('apsmatch:args', 'GPU path covers imageMatchingMethod = ''ransac'', transformationType = ''projective''.');
    end
    if isfield(input, 'apsGPUs')
        error('apsmatch:args', 'input.apsGPUs is not supported by globalImageMatchingSets; match the sets on one GPU.');
    end
    if numel(descSets) ~= numel(numImgs) || numel(keypointsSets) ~= numel(numImgs)
        error('apsmatch:args', 'numImgs, descSets and keypointsSets must have one element per set.');
    end
    mutual = 0;
    if isfield(input, 'apsMutual'), mutual = double(input.apsMutual); end
    args = {descSets, numImgs, keypointsSets, input.k, input.Ratiothreshold, double(input.BFMatch), ...
        input.mBrownLowe, input.maxDistance, input.inliersConfidence, input.maxIter, 0, mutual};
    if nargout > 3
        [allMatchesSets, numMatchesSets, tformsSets, matchesSets] = aps_globalImageMatching_mex(args{:});
    else
        [allMatchesSets, numMatchesSets, tformsSets] = aps_globalImageMatching_mex(args{:});
    end
end
