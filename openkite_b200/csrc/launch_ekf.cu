#include "kite_launch.h"
namespace kite {
template <bool ARM, bool RIGID>
static void go_predict(const EkfArgs& a, cudaStream_t s) {
    // per-device attribute, set on every launch (contexts may live on several devices of one process)
    cudaFuncSetAttribute(k_ekf_predict<ARM, RIGID>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EfCfg<ARM>::SMEM);
    const int sms = current_device_sms();
    const long ngroups = (a.B + 31) / 32;
    const long want = (ngroups + EfCfg<ARM>::WARPS - 1) / EfCfg<ARM>::WARPS;
    const unsigned grid = (unsigned)(want < sms ? want : sms);          // persistent: one CTA per SM
    k_ekf_predict<ARM, RIGID><<<grid, EfCfg<ARM>::WARPS * 32, EfCfg<ARM>::SMEM, s>>>(a);
}
template <bool ARM, bool RIGID>
static void go_predict_tma(const EkfTmaArgs& a, cudaStream_t s) {
    cudaFuncSetAttribute(k_ekf_predict_tma<ARM, RIGID>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EtCfg<ARM>::SMEM);
    const int sms = current_device_sms();
    const long ngroups = (a.e.B + 31) / 32;
    const long want = (ngroups + EtCfg<ARM>::WARPS - 1) / EtCfg<ARM>::WARPS;
    const unsigned grid = (unsigned)(want < sms ? want : sms);          // persistent: one CTA per SM
    k_ekf_predict_tma<ARM, RIGID><<<grid, EtCfg<ARM>::WARPS * 32, EtCfg<ARM>::SMEM, s>>>(a);
}
size_t ekf_predict_scratch_bytes() {
    int sms = current_device_sms();        // the scratch is a per-context buffer, sized for the context's (current) device
    if (sms <= 0) sms = 256;
    return sizeof(double) * (size_t)ET_SCRATCH_PER_CTA_MAX * (size_t)sms;      // Jacobian lines of the resident warps (one CTA per SM)
}
void launch_ekf_predict(const EkfArgs& a, bool rigid, bool arm, double* lines, cudaStream_t s) {
    // the covariance moves as TMA boxes when its layout allows it (16-byte aligned base and pitch, even B)
    EkfTmaArgs ta{};
    ta.e = a; ta.Jw = lines;
    if (lines && sens_make_tensor_map(&ta.tmP, const_cast<double*>(a.P), a.B, a.ld, 169, 1) &&
        sens_make_tensor_map(&ta.tmPn, a.Pn, a.B, a.ld, 169, 1)) {
        if (rigid) go_predict_tma<false, true>(ta, s);
        else if (arm) go_predict_tma<true, false>(ta, s);
        else go_predict_tma<false, false>(ta, s);
        return;
    }
    if (rigid) go_predict<false, true>(a, s);
    else if (arm) go_predict<true, false>(a, s);
    else go_predict<false, false>(a, s);
}
void launch_ekf_update(const EkfUpdArgs& a, cudaStream_t s) {
    constexpr int smem = (int)sizeof(double) * (91 + 13) * EKFU_BLOCK;
    cudaFuncSetAttribute(k_ekf_update<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    k_ekf_update<0><<<blocks_for(a.B, EKFU_BLOCK), EKFU_BLOCK, smem, s>>>(a);
}
}  // namespace kite
