function matches = featureMatchingGlobal(input, allDescriptors, numImg)
    %FEATUREMATCHINGGLOBAL  Drop-in replacement of PP/featureMatching/featureMatchingGlobal.m.
    %   Same signature and output (numImg x numImg cell, [M x 2] double index pairs in the strict
    %   upper triangle, [] elsewhere); pooling, L2 normalisation, global kNN (exact), self / same-image
    %   removal, Lowe ratio test and the scatter into cells all run on the GPU in ONE call
    %   (aps_featureMatching_mex -> libapsmatch.so).  No gpuArray, no CPU fallback: without a B200
    %   the MEX raises apsmatch:nogpu.
    %   input.apsGPUs (optional, e.g. 1:gpuDeviceCount): spread the call over these GPUs (gpuDevice numbering) from this
    %   one process; the match lists are identical to the one-GPU call.
    arguments
        input struct
        allDescriptors cell
        numImg (1, 1) {mustBeNumeric, mustBeFinite, mustBePositive}
    end
    useBF = isfield(input, 'BFMatch') && input.BFMatch;
    if isfield(input, 'apsGPUs')
        matches = aps_featureMatching_mex('global', allDescriptors, numImg, input.k, input.Ratiothreshold, ...
            double(useBF), double(input.apsGPUs));
    else
        matches = aps_featureMatching_mex('global', allDescriptors, numImg, input.k, input.Ratiothreshold, double(useBF));
    end
end
