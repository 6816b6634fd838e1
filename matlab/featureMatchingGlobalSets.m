function matchesSets = featureMatchingGlobalSets(input, allDescriptorsSets, numImgs)
    %FEATUREMATCHINGGLOBALSETS  featureMatchingGlobal over many independent image sets in one GPU call.
    %   matchesSets{b} is exactly featureMatchingGlobal(input, allDescriptorsSets{b}, numImgs(b)): a
    %   numImgs(b) x numImgs(b) cell of [M x 2] double index pairs.  Rows of one set never see another
    %   set's rows.  Reads input.k, input.Ratiothreshold, input.BFMatch and the opt-in input.apsMutual.
    %   Every set must use one descriptor class (single, or binaryFeatures) and one width.  All sets
    %   share one pass on the GPU (aps_featureMatching_mex('globalsets', ...) -> libapsmatch.so), so
    %   many panoramas cost about one call instead of one call each.  No device groups here.
    %
    %   A script that loops over dataset folders can extract features first and match every folder at once:
    %
    %       allDescriptorsSets = cell(1, numel(imgFolders));
    %       numImgs = zeros(1, numel(imgFolders));
    %       for f = 1:numel(imgFolders)
    %           [~, ~, numImgs(f)] = loadImages(input, imgFolders(f), myImg);   % as the reference loads one folder
    %           [~, allDescriptorsSets{f}] = getFeaturePoints(input, ...);      % its features, as today
    %       end
    %       matchesSets = featureMatchingGlobalSets(input, allDescriptorsSets, numImgs);
    %       for f = 1:numel(imgFolders)
    %           matches = matchesSets{f};   % what featureMatchingGlobal returned for folder f
    %           % ... imageMatching, bundle adjustment, rendering of folder f as before
    %       end
    arguments
        input struct
        allDescriptorsSets cell
        numImgs (1, :) {mustBeNumeric, mustBeFinite, mustBePositive, mustBeInteger}
    end
    useBF = isfield(input, 'BFMatch') && input.BFMatch;
    mutual = isfield(input, 'apsMutual') && input.apsMutual;
    matchesSets = aps_featureMatching_mex('globalsets', allDescriptorsSets, numImgs, input.k, ...
        input.Ratiothreshold, double(useBF), double(mutual));
end
