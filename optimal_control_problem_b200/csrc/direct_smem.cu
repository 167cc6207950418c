// Instantiation of admm_direct_kernel<PLACE_SMEM, 384, 1> (see direct_instance.h) and the placement -> entry points
// lookup.
#include "direct_instance.h"

namespace ocpb200 {
namespace direct {

const EntryPoints kSmem = Instance<PLACE_SMEM, 384, 1>::entry_points;

const EntryPoints& entry_points(int place) {
  switch (place) {
    case PLACE_SMEM: return kSmem;
    case PLACE_MULTI: return kMulti;
    case PLACE_BIG: return kBig;
    default: return kMixed;
  }
}

}  // namespace direct
}  // namespace ocpb200
