// sfma_hbm.cu -- K5, the fused SFMA kernel with its per-agent tables in a global workspace (sfma_kernel<A, MODS, true>),
// for configurations that need the fused kernel on state spaces whose SfmaSmem block exceeds shared memory.  The kernel
// is sfma.cu's, compiled here so that the on-chip instantiations in sfma.cu are built exactly as without it.
#define SFMA_HBM_TU
#include "sfma.cu"
