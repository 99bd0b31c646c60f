// Dispatch of the per-point backward over the padded input dimension.
#include "gpblur_point_bwd.cuh"

namespace gpblur {

int launch_point_backward_dp16(const PointBwdArgs& a, cudaStream_t st);
int launch_point_backward_dp32(const PointBwdArgs& a, cudaStream_t st);
int launch_point_backward_dp64(const PointBwdArgs& a, cudaStream_t st);
int launch_point_backward_dp128(const PointBwdArgs& a, cudaStream_t st);

int bwd_vector_partials(const WsLayout& L) { return bwd_persistent_grid(L, bwd_tile_points(L)); }

int launch_point_backward(const WsLayout& L, const void* stage, void* ws, const float* x, const SegGrads& seg,
                          const float* var, uint64_t seed, uint64_t offset, uint32_t stream_id,
                          const unsigned long long* offset_dev, float* dx, cudaStream_t st) {
  if (L.N <= 0) return GPBLUR_OK;
  PointBwdArgs a{L, ws, stage, x, var, seed, offset, stream_id, dx, 0, offset_dev, seg};
  switch (L.DP) {
    case 16: return launch_point_backward_dp16(a, st);
    case 32: return launch_point_backward_dp32(a, st);
    case 64: return launch_point_backward_dp64(a, st);
    default: return launch_point_backward_dp128(a, st);
  }
}

}  // namespace gpblur
