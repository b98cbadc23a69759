"""depthmapcompression_b200 -- B200 (sm_100a) implementation of the post filter set for decoded depth maps
(Wavelet303/DepthMapCompression, PostFilterSetForDepthCoding/filter.h) behind the reference's own operator names.

The product is libdmc_b200.so (hand-written CUDA kernels + a C ABI, include/dmc_c.h).  The C++ drop-in for the
reference's header is include/filter.h; this Python package is the same interface for numpy / device pointers and
is what tests/ and bench.py drive.  There is no CPU path: importing needs the built library, creating a
Context needs a CUDA device.
"""
from .capi import (FULL_KERNEL, FULL_KERNEL_PAIR, SEPARABLE_KERNEL, FILL_DISPARITY, FILL_DEPTH, DmcError,  # noqa: F401
                   shard_frames)
from .filters import (Context, PostFilterSet, binalyWeightedRangeFilter, jointBinalyWeightedRangeFilter, blurRemoveMinMax, blurRemoveMinMaxBase,  # noqa: F401
                      maxFilter, minFilter, boundaryReconstructionFilter, minmaxBoundaryReconstructionFilter, smallGaussianBlur, medianBlur,
                      disp8U2depth32F, depth32F2disp8U, depth16U2disp8U, disp16S2depth16U, fillOcclusion,
                      reprojectXYZ, transpose, default_context, jpegDecodeGrayBatch, jpegProbe, jpegDecodeColorBatch, jpegProbeColor, jpegEncodeGrayBatch, jpegEncodeBound, degradeJPEG, jpegEncodeColorBatch, jpegEncodeColorBound, degradeJPEGColor, frameSSE, frameSSIM, psnrFromSSE, jpegRateDistortion, jpegViewRateDistortion, boundaryReconstructionFilterBatch, brf_params, prepareDisparityBatch, renderViewBatch, pack_streams, multi_chain_batch, FrameBatchScheduler, hostlink_probe,
                      projectPointsSimple, projectImagefromXYZ, fillSmallHole, pinned_empty, pinned_free, host_register, host_unregister)
