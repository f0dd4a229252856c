// ocd_inst.cu -- one (H, other cars, lanes, math mode) specialisation of k_solve / k_episode / k_solve_vjp /
// k_episode_jac.
// Compiled once per combination by the Makefile:
//   nvcc -DOCD_HT=5 -DOCD_NO=1 -DOCD_LT=3 -DOCD_PRECISE=0 -c ocd_inst.cu -o build/inst_5_1_3_0.o
//   (+ -DOCD_SOLVE_ONLY for build/solve_<HT>_<NO>_<LT>.o: FAST k_solve alone)
#include "ocd_kernels.cuh"
#define OCD_HD_ONLY          // the hyper-dual arithmetic of ocd_hessian.cuh without its kernel (built by ocd_api.cu)
#include "ocd_vjp.cuh"

#if !defined(OCD_HT) || !defined(OCD_NO) || !defined(OCD_LT) || !defined(OCD_PRECISE)
#error "define OCD_HT, OCD_NO, OCD_LT and OCD_PRECISE"
#endif

namespace ocd {
template int launch_solve_t<OCD_HT, OCD_NO, OCD_LT, (OCD_PRECISE != 0)>(const KParams &, const SolveArgs &, cudaStream_t);
template int launch_solve_vjp_t<OCD_HT, OCD_NO, OCD_LT, (OCD_PRECISE != 0)>(const KParams &, const VjpArgs &, cudaStream_t);
#ifndef OCD_SOLVE_ONLY   // the many-car sweep specialisations build k_solve only
template int launch_episode_t<OCD_HT, OCD_NO, OCD_LT, (OCD_PRECISE != 0)>(const KParams &, const ocd_scenario &,
                                                                  const EpisodeArgs &, cudaStream_t);
// the episode's reverse pass re-runs the iterations of the episode's specialisation (not the solve's)
template int launch_episode_jac_t<OCD_HT, OCD_NO, OCD_LT, (OCD_PRECISE != 0)>(const KParams &, const ocd_scenario &,
                                                                      const EpisodeVjpArgs &, int, cudaStream_t);
#endif
}  // namespace ocd

#ifdef OCD_BLOCK_TIMES   // tuning builds only (scripts/tuning/block_times.py): read back the per-block timestamps
extern "C" int ocd_debug_block_times(void *host_buf) {
    return cudaMemcpyFromSymbol(host_buf, ocd::g_block_times, sizeof(ocd::g_block_times)) == cudaSuccess ? 0 : -1;
}
#endif
