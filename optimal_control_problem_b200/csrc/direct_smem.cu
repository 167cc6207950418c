// Instantiation of admm_direct_kernel<PLACE_SMEM, 384, 1> (see direct_instance.h), the placement -> entry points
// lookup and the plan helpers.
#include "direct_instance.h"

namespace ocpb200 {
namespace direct {

const EntryPoints kSmem = Instance<PLACE_SMEM, 384, 1>::entry_points;

size_t plan_array_doubles(const PatternDev& P, int id) { return array_doubles(P, id); }
int plan_array_count() { return AR_COUNT; }
bool plan_multi_in_smem(int id) { return multi_in_smem(id); }
bool plan_big_in_smem(int id) { return big_in_smem(id); }
bool plan_smem_in_smem(int id) { return smem_in_smem(id); }
int plan_stage_array() { return AR_STAGE; }
bool plan_is_factor_array(int id) { return id == AR_DINV || id == AR_LSUB || id == AR_LP; }
void plan_mixed_priority(std::vector<int>& order) {
  order = {AR_B, AR_X, AR_W, AR_CTYPE, AR_Q, AR_STAGE, AR_SCRATCH, AR_Z, AR_Y, AR_L, AR_U, AR_D, AR_E,
           AR_AVAL, AR_IDX, AR_PVAL, AR_LP, AR_DINV, AR_LSUB, AR_DX, AR_DY};
}

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
