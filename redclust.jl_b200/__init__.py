"""redclust.jl_b200 -- B200-native sampler hot path of RedClust.jl behind the reference's API.

The directory name contains a dot, so it is loaded under the module name `redclust_jl_b200`
(see __graft_entry__.load_package()).  Only what the hot path needs lives here:
  csrc/        hand-written sm_100a CUDA kernels + the C ABI (include/rcb200.h) -> librcb200.so
  _lib.py      ctypes binding of the C ABI
  host.py      host-side mirror of the reference's API (MCMCData, runsampler, getpointestimate, ...)
  prior.py     host-side fitprior / k-medoids (caller of the hot path)
  h5min.py     minimal HDF5 reader for example_datasets (example_data.jl:33-71)
  data/        the package's copy of the three example data sets
  julia/       the `ccall` twin of host.py for a Julia host
"""
from .host import (Comm, MCMCOptionsList, PriorHyperparamsList, MCMCData, MCMCState, MCMCResult, Sampler, runsampler,
                   getpointestimate, binderloss, infodist, adjacencymatrix, sortlabels, makematrix, uppertriangle,
                   generatemixture, example_dataset, example_datasets, prettytime, prettynumber, evaluateclustering, summarise, params_from_labels, pair_stats, psm, psm_counts_dev, psm_sharded, mpel_loss_sums, binder_loss_sums, mpel_loss_sums_sharded, cyclic_rows, assemble_cyclic_rows, init_rp, ArgumentError,
                   crossdistances, predictivecoclustering, allocationprobabilities, predictive_from_labels)
from ._lib import RCError, LIB_PATH
from .prior import fitprior, fitprior2, sampledist, sampleK, kmedoids, kmedoids_device, kmeans
