// Instantiation of admm_direct_kernel<PLACE_MIXED, 768, 1> (see direct_instance.h).  The mixed placement
// serves problems whose matrices and index arrays stay in global memory: its parallel phases are bound by
// dependent global loads, so they want as many threads as the register file allows (centroidal H=50,
// 148 instances: 376 ms at 256 threads, 297 at 512, 278 at 768, 298 at 1024).
#include "direct_instance.h"

namespace ocpb200 {
namespace direct {

const EntryPoints kMixed = Instance<PLACE_MIXED, 768, 1>::entry_points;

}  // namespace direct
}  // namespace ocpb200
