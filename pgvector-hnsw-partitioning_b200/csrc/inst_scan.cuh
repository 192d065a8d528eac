// inst_scan.cuh -- instantiates the scan kernels for one (storage type, metric) pair.  Included
// by scan_<type>_<metric>.cu with HBI_T / HBI_IP / HBI_NAME defined, so the four pairs compile in
// parallel.
#include "index.h"
#include "scan_kernel.cuh"
#include "scan_reg.cuh"
#include "scan_cta.cuh"

namespace hb {
cudaError_t HB_CAT(scan_fast_, HBI_NAME)(const ScanParams &p, int sms, int mg, cudaStream_t s, ScanLaunchInfo *i)
{
    return launch_scan_t<HBI_T, HBI_IP, false>(p, sms, mg, s, i);
}
cudaError_t HB_CAT(scan_slow_, HBI_NAME)(const ScanParams &p, int sms, int mg, cudaStream_t s, ScanLaunchInfo *i)
{
    return launch_scan_t<HBI_T, HBI_IP, true>(p, sms, mg, s, i);
}
cudaError_t HB_CAT(scan_reg_, HBI_NAME)(const ScanParams &p, int R, int sms, int mg, cudaStream_t s, ScanLaunchInfo *i)
{
    return launch_scan_reg_t<HBI_T, HBI_IP>(p, R, sms, mg, s, i);
}
cudaError_t HB_CAT(scan_cta_, HBI_NAME)(const ScanParams &p, int sms, cudaStream_t s) { return launch_scan_cta_t<HBI_T, HBI_IP>(p, sms, s); }
cudaError_t HB_CAT(dist_, HBI_NAME)(const DistBatchParams &p, cudaStream_t s) { return launch_dist_t<HBI_T, HBI_IP>(p, s); }
}   // namespace hb

#include "build_kernel.cuh"
#include "iter_kernel.cuh"
namespace hb {
cudaError_t HB_CAT(iter_, HBI_NAME)(const IterParams &p, int grid, cudaStream_t s) { return launch_iter_t<HBI_T, HBI_IP>(p, grid, s); }
cudaError_t HB_CAT(build_search_, HBI_NAME)(const BuildSearchParams &p, int sms, int slow_grid, cudaStream_t s, bool slow)
{
    return slow ? launch_build_search_t<HBI_T, HBI_IP, true>(p, sms, slow_grid, s)
                : launch_build_search_t<HBI_T, HBI_IP, false>(p, sms, slow_grid, s);
}
cudaError_t HB_CAT(build_link_, HBI_NAME)(const LinkParams &p, int sms, int which, cudaStream_t s)
{
    return launch_build_link_t<HBI_T, HBI_IP>(p, sms, which, s);
}
cudaError_t HB_CAT(pair_fill_, HBI_NAME)(const LinkParams &p, int sms, int max_items, cudaStream_t s)
{
    return launch_pair_fill_t<HBI_T, HBI_IP>(p, sms, max_items, s);
}
cudaError_t HB_CAT(nbr_dist_, HBI_NAME)(const NbrDistParams &p, int sms, cudaStream_t s)
{
    return launch_nbr_dist_t<HBI_T, HBI_IP>(p, sms, s);
}
}   // namespace hb
