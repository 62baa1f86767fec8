// env_alloc.cu - launcher of the one-warp allocation kernel of the split step (env_alloc.cuh).
#include <atomic>

#include "env_alloc.cuh"

namespace marlsc {

namespace {

// prepare_only: do every check and attribute call but do not launch (the split step calls this before it launches K1a, so
// that a failure cannot leave the state half-stepped)
template <int SPL, int NCH>
int launch_tt(const LaunchArgs& a, const marlsc_step_io_t& io, double* cost_alloc, int t, cudaStream_t s, bool prepare_only) {
  using Cfg = AllocCfg<SPL>;
  const AllocLayout l = alloc_layout(a.ds.W, a.ds.S, a.ds.R, NCH, Cfg::MW, Cfg::kPass, SPL);
  const size_t smem = (size_t)l.t_bytes + 4 * (size_t)l.team_bytes;
  if ((int)smem > a.max_smem_optin) return 0;
  static std::atomic<size_t> configured[kMaxDevices];   // per device: the attributes belong to the device's context
  static std::atomic<bool> carveout[kMaxDevices];
  int dev = 0;
  MARLSC_CUDA(cudaGetDevice(&dev));
  const int di = dev < kMaxDevices ? dev : kMaxDevices - 1;
  if (dev >= kMaxDevices || !carveout[di].load()) {   // the scratch is what bounds residency: ask for the largest shared-memory carveout
    MARLSC_CUDA(cudaFuncSetAttribute((const void*)env_alloc_warp_kernel<SPL, NCH>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                     (int)cudaSharedmemCarveoutMaxShared));
    carveout[di].store(true);
  }
  if (smem > 48 * 1024 && (dev >= kMaxDevices || smem > configured[di].load())) {
    MARLSC_CUDA(cudaFuncSetAttribute((const void*)env_alloc_warp_kernel<SPL, NCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured[di].store(smem);
  }
  if (prepare_only) return 1;
  env_alloc_warp_kernel<SPL, NCH><<<(unsigned)((a.st.num_envs + 3) / 4), 128, smem, s>>>(a.ds, a.st, io, cost_alloc, t);
  MARLSC_CUDA(cudaGetLastError());
  return 1;
}

template <int SPL>
int launch_t(const LaunchArgs& a, const marlsc_step_io_t& io, double* cost_alloc, int t, cudaStream_t s, bool prepare_only) {
  if (!a.ds.prio_perm) return 0;   // needs W <= 16 (availability masks)
  switch (a.ds.perm_chunks) {
    case 1: return launch_tt<SPL, 1>(a, io, cost_alloc, t, s, prepare_only);
    case 2: return launch_tt<SPL, 2>(a, io, cost_alloc, t, s, prepare_only);
    case 3: return launch_tt<SPL, 3>(a, io, cost_alloc, t, s, prepare_only);
    case 4: return launch_tt<SPL, 4>(a, io, cost_alloc, t, s, prepare_only);
    default: return 0;
  }
}

}  // namespace

int launch_alloc_warp(int spl, const LaunchArgs& a, const marlsc_step_io_t& io, double* cost_alloc, int t, cudaStream_t s, bool prepare_only) {
  if (io.order_qty_bytes != 1) return 0;
  switch (spl) {
    case 1: return launch_t<1>(a, io, cost_alloc, t, s, prepare_only);
    case 4: return launch_t<4>(a, io, cost_alloc, t, s, prepare_only);
    case 8: return launch_t<8>(a, io, cost_alloc, t, s, prepare_only);
    default: return 0;
  }
}

}  // namespace marlsc
