function [allMatches, numMatches, tforms, matches] = pairwiseImageMatching(input, allDescriptors, numImg, keypoints)
    %PAIRWISEIMAGEMATCHING  Drop-in for the pair of calls of the reference with input.matchFeaturesPairwise = 1:
    %       matches = featureMatchingPairwise(input, allDescriptors, numImg);                    % main.m:95-99
    %       [allMatches, numMatches, tforms] = imageMatching(input, numImg, keypoints, matches); % imageMatchingPanoramaConComps.m:40
    %   in one GPU call with the match lists kept on the device in between; the outputs are exactly the two calls'.
    %   matches (the fourth output) is fetched only when asked for.  The one-set case of pairwiseImageMatchingSets.
    arguments
        input (1, 1) struct
        allDescriptors cell
        numImg (1, 1) double {mustBeInteger, mustBePositive}
        keypoints cell
    end
    if nargout > 3
        [a, n, t, m] = pairwiseImageMatchingSets(input, {allDescriptors}, numImg, {keypoints});
        matches = m{1};
    else
        [a, n, t] = pairwiseImageMatchingSets(input, {allDescriptors}, numImg, {keypoints});
    end
    allMatches = a{1};
    numMatches = n{1};
    tforms = t{1};
end
