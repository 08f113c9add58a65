// The wide instantiations (PMDI_X_GLOBAL): the pool and spec sweeps, and the single-cluster evaluation, for a context
// whose observation cannot be staged in shared memory.  The block operators are the staged kernels' own source; they
// read x[t] and x[t-1] from global memory (DsDev::xstage) instead of the observation ring, and the dynamic shared
// memory holds the log-factorial table and the role tables alone.  Compiled into a cubin of its own, which
// libpmdi_cuda.so carries and loads on first use: in pmdi_cuda.cu's module these kernels would share non-inlined device
// functions with k_sweep_spec and k_sweep_pool and change their code (spec_group.cu).  Nothing else goes here.
#define PMDI_X_GLOBAL
#include "aux_kernels.cuh"
#include "pool_kernel.cuh"
#include "spec_kernel.cuh"
