// The group instantiations of the speculative sweep (k_sweep_spec_group / _dbg, spec_kernel.cuh): several contexts in
// one cooperative launch.  They are compiled into a cubin of their own, which libpmdi_cuda.so carries and loads at run
// time (pmdi_group_create).  In one module with k_sweep_spec the device functions both kernels call would be compiled
// once for both callers, and that changes the register allocation and stack frame of the single-context kernels
// (measured: 352 -> 384 B of stack); in a module of their own the single-context kernels stay as they are.  With
// PMDI_SPEC_GROUP defined spec_kernel.cuh compiles the two group kernels and nothing else: the members' set-up and
// finish kernels run from the library (or a member's run-time compiled program), and any other kernel in this module
// would share its non-inlined device functions with the group kernels and change their code.
#define PMDI_SPEC_GROUP
#include "spec_kernel.cuh"
