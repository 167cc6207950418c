// Instantiation of admm_direct_kernel<PLACE_BIG, 384, 1> (see direct_instance.h).
#include "direct_instance.h"

namespace ocpb200 {
namespace direct {

const EntryPoints kBig = Instance<PLACE_BIG, 384, 1>::entry_points;

}  // namespace direct
}  // namespace ocpb200
