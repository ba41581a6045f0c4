#include "kite_launch.h"
namespace kite {
constexpr int COLLOC_NPB = 4;      // node rows per CTA: 128 threads at 255 registers, no spills (11 rows = 352 threads spilled 400+ B)
void launch_colloc_eval(const CollocArgs& a, bool percoef, int fmt, cudaStream_t s) {
    const unsigned gb = blocks_for(a.B, 32);
    dim3 block(32, COLLOC_NPB);
    constexpr int N = COLLOC_NPB;
    if (percoef) {
        if (fmt == 3) k_colloc_eval<true, N, 3><<<gb, block, 0, s>>>(a);
        else if (fmt == 0) k_colloc_eval<true, N, 0><<<gb, block, 0, s>>>(a);
        else if (fmt == 1) k_colloc_eval<true, N, 1><<<gb, block, 0, s>>>(a);
        else k_colloc_eval<true, N, 2><<<gb, block, 0, s>>>(a);
    } else {
        if (fmt == 3) k_colloc_eval<false, N, 3><<<gb, block, 0, s>>>(a);
        else if (fmt == 0) k_colloc_eval<false, N, 0><<<gb, block, 0, s>>>(a);
        else if (fmt == 1) k_colloc_eval<false, N, 1><<<gb, block, 0, s>>>(a);
        else k_colloc_eval<false, N, 2><<<gb, block, 0, s>>>(a);
    }
}
void launch_colloc_cost(const CostArgs& a, cudaStream_t s) {
    dim3 block(32, 4);
    k_colloc_cost<4><<<blocks_for(a.B, 32), block, 0, s>>>(a);
}
}  // namespace kite
