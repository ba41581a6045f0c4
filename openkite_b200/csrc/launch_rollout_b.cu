#include "kite_launch.h"
namespace kite {
template <int UMODE>
static void go(const RolloutArgs& a, bool rigid, bool percoef, cudaStream_t s) {
    dim3 grid(blocks_for(a.B, ROLLOUT_BLOCK)), block(ROLLOUT_BLOCK);
    if constexpr (UMODE != 3) {      // rigid body + synthetic inputs is rejected by kite_rk4_rollout: no such kernel
        if (rigid) { k_rk4_rollout<UMODE, true, false><<<grid, block, rollout_smem_bytes(false), s>>>(a); return; }
    }
    if (percoef) k_rk4_rollout<UMODE, false, true><<<grid, block, rollout_smem_bytes(true), s>>>(a);
    else k_rk4_rollout<UMODE, false, false><<<grid, block, rollout_smem_bytes(false), s>>>(a);
}
void launch_rollout_23(const RolloutArgs& a, int umode, bool rigid, bool percoef, cudaStream_t s) {
    if (umode == 2) go<2>(a, rigid, percoef, s); else go<3>(a, rigid, percoef, s);
}
}  // namespace kite
