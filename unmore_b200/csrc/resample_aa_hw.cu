// The antialiased crop on a padded stack of images of different sizes (unmore_crop_resize_aa_hw): the SIZED
// instantiation of the kernels in aa_crop.cuh, in a file of its own so that the uniform kernels keep their code.
#include "aa_crop.cuh"
#include "unmore_internal.h"

namespace unmore {

int launch_crop_resize_aa_hw(const AaCropParams& p, long long tiles, const int* image_hw, cudaStream_t stream) {
  AaCropHwParams hp;
  static_cast<AaCropParams&>(hp) = p;
  hp.image_hw = image_hw;
  return launch_crop_aa_t<true>(hp, tiles, stream);
}

}  // namespace unmore
