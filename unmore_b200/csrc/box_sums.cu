// O(1) box sums from the summed-area tables of sat.cu (north-star op (a)):
//   boxsum = S[y2][x2] - S[y1][x2] - S[y2][x1] + S[y1][x1]   on the snapped window.
// In a file of its own: compiled beside any of the sized (image_hw) kernels, box_sums_kernel's code changes.
#include "unmore_internal.h"

namespace unmore {

__global__ void box_sums_kernel(const double* __restrict__ sat, int planes_per_img, int plane, int H, int W,
                                const void* __restrict__ boxes, int boxes_f64, const int* __restrict__ counts, int cap,
                                int n_img, double* __restrict__ sums, double* __restrict__ means) {
  const int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= n_img * cap) return;
  const int img = id / cap, k = id - img * cap;
  if (counts && k >= counts[img]) return;
  double x1, y1, x2, y2;
  load_box<double>(boxes, boxes_f64 != 0, (size_t)id, x1, y1, x2, y2);
  const Window w = snap_window<double>(x1, y1, x2, y2, W, H);
  const double* S = sat + ((size_t)img * planes_per_img + plane) * (H + 1) * (W + 1);
  const int OW = W + 1;
  double s = 0.0;
  if (!w.empty())
    s = S[(size_t)w.y2 * OW + w.x2] - S[(size_t)w.y1 * OW + w.x2] - S[(size_t)w.y2 * OW + w.x1] + S[(size_t)w.y1 * OW + w.x1];
  sums[id] = s;
  if (means) means[id] = w.empty() ? 0.0 : s / ((double)w.w() * (double)w.h());
}

int launch_box_sums(const double* sat, int planes_per_img, int plane, int H, int W, const void* boxes, int boxes_f64,
                    const int* counts, int cap, int n_img, double* sums, double* means, const int* image_hw,
                    cudaStream_t stream) {
  const int total = n_img * cap;
  if (total <= 0) return 0;
  if (image_hw)
    return launch_box_sums_hw(sat, planes_per_img, plane, H, W, boxes, boxes_f64, counts, cap, n_img, sums, means, image_hw,
                              stream);
  box_sums_kernel<<<(total + 255) / 256, 256, 0, stream>>>(sat, planes_per_img, plane, H, W, boxes, boxes_f64, counts, cap,
                                                            n_img, sums, means);
  return (int)cudaGetLastError();
}

}  // namespace unmore
