// noc_ts_inst.cu — instantiation of the streamed tensor-core rollout (noc_ts_rollout.cuh) for the 50-agent swarm (d = 150).
#include "noc_ts_rollout.cuh"

namespace noc {
int launch_ts_swarm50(const RolloutCall<float>& c) { return launch_ts<TsShape<50>>(c); }
}  // namespace noc
