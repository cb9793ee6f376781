"""visfd_b200 -- B200-native (sm_100a) implementation of visfd's filter_mrc membrane /
blob detection hot path behind a C ABI (include/visfd_cuda.h).

  visfd_b200/csrc/        CUDA kernels + the extern "C" layer  -> visfd_b200/libvisfd_cuda.so
  visfd_b200/csrc/visfd_cuda_shim.hpp
                          C++ mirror of the reference's `namespace visfd` entry points
  visfd_b200/csrc/multi.cu        the membrane pipeline, blob detection and the Gaussian / DoG / LoG filters in Z-slabs
                                  behind one C call: on several GPUs (visfd_cuda_membrane_multi, visfd_cuda_blob_dog_multi,
                                  visfd_cuda_filter_multi), or on one GPU slab after slab within a memory budget
                                  (visfd_cuda_membrane_stream, visfd_cuda_blob_dog_stream, visfd_cuda_filter_stream);
                                  the membrane pipeline with -connect (visfd_cuda_membrane_connect_multi / _stream)
  visfd_b200/csrc/connect.cu      LabelConnected: device predicates + ordered host flood
  visfd_b200/capi.py      ctypes binding (tests, bench, multi-GPU driver)
  visfd_b200/slab.py      Z-slab multi-GPU drivers: membrane pipeline, blob detection, image statistics
                          (torch.distributed / NCCL plumbing)
  visfd_b200/mrc.py       MRC / REC file I/O (include/visfd_mrc.h)
  visfd_b200/blobs.py     blob list post-processing (include/visfd_blobs.h)
  visfd_b200/synth.py     synthetic tomograms

There is no CPU fallback anywhere in this package.
"""
from .capi import (Context, VisfdCudaError, MembraneParams, load_library, gen_gauss1d, gauss_halfwidth,
                   tv_halfwidth, INCREASING_EIVALS, DECREASING_EIVALS, SCORE_PLANAR, SCORE_LINEAR,
                   THRESH_SINGLE, THRESH_2, THRESH_4, THRESH_GAUSS, RESCALE, blob_finalize, pack_regions,
                   membrane_multi, blob_dog_multi, FilterParams, filter_multi, ConnectParams,
                   membrane_connect_multi)

__all__ = ["Context", "VisfdCudaError", "MembraneParams", "load_library", "gen_gauss1d", "gauss_halfwidth",
           "tv_halfwidth", "blob_finalize", "pack_regions", "membrane_multi",
           "blob_dog_multi", "FilterParams", "filter_multi", "ConnectParams", "membrane_connect_multi"]
