// center_reasoning in the second resize mode (antialias=True) straight from the fields: the kernel of center.cuh on the
// antialiased row source (CenterAaRows).
#include "center.cuh"

namespace unmore {

// the same three passes as launch_center on fields: row skipping on the first pass (the one that asks for split boxes)
int launch_center_aa(const CenterParams& p, int num_sms, cudaStream_t stream) {
  if (p.cc_counts) return launch_center_t<true, kAaFields>(p, num_sms, stream);
  if (p.splits) return launch_center_t<false, kAaFields, true>(p, num_sms, stream);
  return launch_center_t<false, kAaFields>(p, num_sms, stream);
}

}  // namespace unmore
