// mcb_engine_prm.cu -- the step kernels of batches with per-env physics parameters (mcb_env_kernel<TIER, true>).
//
// The same source as mcb_engine.cu, compiled as a translation unit of its own so that the default kernels' module stays as it is
// (see prm_launch_tiers() there).  This unit defines only prm_launch_tiers() and prm_set_tier_smem(); the C ABI lives in
// mcb_engine.cu.
#define MCB_PRM_UNIT
#include "mcb_engine.cu"
