function [allMatchesSets, numMatchesSets, tformsSets] = imageMatchingSets(input, numImgs, keypointsSets, matchesAllSets)
    %IMAGEMATCHINGSETS  imageMatching over many independent image sets in one GPU call.
    %   Element b of each 1 x B output cell is exactly what imageMatching(input, numImgs(b), keypointsSets{b},
    %   matchesAllSets{b}) returns: top-m partner selection, RANSAC homography per candidate pair ('projective'),
    %   acceptance ni > 8 + 0.3*nf, tforms{i,j} / tforms{j,i} = model / inv(model).  One partner selection and one
    %   RANSAC pass serve every set (aps_imageMatchingSets_mex -> libapsmatch.so); no CPU fallback.
    %
    %   A batch of panoramas, one per dataset folder, in two calls end to end:
    %       for b = 1:B
    %           descSets{b} = allDescriptors_of_folder{b};  keypointsSets{b} = keypoints_of_folder{b};
    %           numImgs(b) = numel(descSets{b});
    %       end
    %       matchesSets = featureMatchingGlobalSets(input, descSets, numImgs);
    %       [allMatchesSets, numMatchesSets, tformsSets] = imageMatchingSets(input, numImgs, keypointsSets, matchesSets);
    arguments
        input (1, 1) struct
        numImgs (1, :) double {mustBeInteger, mustBeNonnegative}
        keypointsSets cell
        matchesAllSets cell
    end
    if input.useMATLABImageMatching == 1 || ~strcmpi(input.imageMatchingMethod, 'ransac') || ...
            ~strcmpi(input.transformationType, 'projective')
        error('apsmatch:args', 'GPU path covers imageMatchingMethod = ''ransac'', transformationType = ''projective''.');
    end
    if numel(keypointsSets) ~= numel(numImgs) || numel(matchesAllSets) ~= numel(numImgs)
        error('apsmatch:args', 'numImgs, keypointsSets and matchesAllSets must have one element per set.');
    end
    for b = 1:numel(numImgs)
        if ~isequal(size(matchesAllSets{b}), [numImgs(b), numImgs(b)])
            error('imageMatching:InvalidMatchesAllSize', 'matchesAllSets{%d} must be an n-by-n cell array.', b);
        end
        if numel(keypointsSets{b}) ~= numImgs(b)
            error('imageMatching:InvalidKeypointsLength', 'keypointsSets{%d} must contain n elements (one per image).', b);
        end
    end
    [allMatchesSets, numMatchesSets, tformsSets] = aps_imageMatchingSets_mex(keypointsSets, matchesAllSets, ...
        input.mBrownLowe, input.maxDistance, input.inliersConfidence, input.maxIter);
end
