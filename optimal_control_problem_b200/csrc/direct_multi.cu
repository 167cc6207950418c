// Instantiation of admm_direct_kernel<PLACE_MULTI, 192, 2> (see direct_instance.h): the throughput plan for the
// problems the compact kernel cannot take.
#include "direct_instance.h"

namespace ocpb200 {
namespace direct {

const EntryPoints kMulti = Instance<PLACE_MULTI, 192, 2>::entry_points;

}  // namespace direct
}  // namespace ocpb200
