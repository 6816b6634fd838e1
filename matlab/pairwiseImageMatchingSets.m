function [allMatchesSets, numMatchesSets, tformsSets, matchesSets] = pairwiseImageMatchingSets(input, descSets, numImgs, keypointsSets)
    %PAIRWISEIMAGEMATCHINGSETS  featureMatchingPairwise followed by imageMatching over many independent image sets, in
    %   one GPU call.  Element b of each 1 x B output cell is exactly what
    %       matchesSets = featureMatchingPairwiseSets(input, descSets, numImgs);
    %       [allMatchesSets, numMatchesSets, tformsSets] = imageMatchingSets(input, numImgs, keypointsSets, matchesSets);
    %   returns, and matchesSets (the fourth output, fetched only when asked for) is the putative lists of the first
    %   call.  The match lists stay on the GPU between the two stages (aps_pairwiseImageMatching_mex -> libapsmatch.so);
    %   no CPU fallback.  keypointsSets{b}{i} has one row per row of descSets{b}{i}.  Reads input.Matchingmethod,
    %   input.ApproxFloatNNMethod, input.Matchingthreshold and input.Ratiothreshold as featureMatchingPairwiseSets does.
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
        error('apsmatch:args', 'input.apsGPUs is not supported by pairwiseImageMatchingSets; match the sets on one GPU.');
    end
    if numel(descSets) ~= numel(numImgs) || numel(keypointsSets) ~= numel(numImgs)
        error('apsmatch:args', 'numImgs, descSets and keypointsSets must have one element per set.');
    end
    method = apsPairwiseMethod(input);                  % aps_method, with the semantics warning
    args = {descSets, numImgs, keypointsSets, input.Matchingthreshold, input.Ratiothreshold, method, ...
        input.mBrownLowe, input.maxDistance, input.inliersConfidence, input.maxIter, 0};
    if nargout > 3
        [allMatchesSets, numMatchesSets, tformsSets, matchesSets] = aps_pairwiseImageMatching_mex(args{:});
    else
        [allMatchesSets, numMatchesSets, tformsSets] = aps_pairwiseImageMatching_mex(args{:});
    end
end
