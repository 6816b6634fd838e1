function matchesSets = featureMatchingPairwiseSets(input, allDescriptorsSets, numImgs)
    %FEATUREMATCHINGPAIRWISESETS  featureMatchingPairwise over many independent image sets in one GPU call.
    %   matchesSets{b} is exactly featureMatchingPairwise(input, allDescriptorsSets{b}, numImgs(b)): a
    %   numImgs(b) x numImgs(b) cell of [M x 2] double index pairs.  Only the pairs inside a set are matched
    %   (sum of numImgs(b)^2 / 2 pairs, not (sum of numImgs)^2 / 2).  Reads input.Matchingmethod,
    %   input.ApproxFloatNNMethod, input.Matchingthreshold and input.Ratiothreshold as featureMatchingPairwise
    %   does.  Every set must use one descriptor class (single, or binaryFeatures) and one width.  All sets
    %   share one pass on the GPU (aps_featureMatching_mex('pairwisesets', ...) -> libapsmatch.so), so many
    %   panoramas cost about one call instead of one call each.  No device groups here.
    %
    %   A script that loops over dataset folders can extract features first and match every folder at once:
    %
    %       allDescriptorsSets = cell(1, numel(imgFolders));
    %       numImgs = zeros(1, numel(imgFolders));
    %       for f = 1:numel(imgFolders)
    %           [~, ~, numImgs(f)] = loadImages(input, imgFolders(f), myImg);   % as the reference loads one folder
    %           [~, allDescriptorsSets{f}] = getFeaturePoints(input, ...);      % its features, as today
    %       end
    %       matchesSets = featureMatchingPairwiseSets(input, allDescriptorsSets, numImgs);
    %       for f = 1:numel(imgFolders)
    %           matches = matchesSets{f};   % what featureMatchingPairwise returned for folder f
    %           % ... imageMatching, bundle adjustment, rendering of folder f as before
    %       end
    arguments
        input struct
        allDescriptorsSets cell
        numImgs (1, :) {mustBeNumeric, mustBeFinite, mustBePositive, mustBeInteger}
    end
    method = apsPairwiseMethod(input);                  % aps_method, with the semantics warning
    matchesSets = aps_featureMatching_mex('pairwisesets', allDescriptorsSets, numImgs, input.Matchingthreshold, ...
        input.Ratiothreshold, method);
end
