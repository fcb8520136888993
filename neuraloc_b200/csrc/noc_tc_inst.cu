// noc_tc_inst.cu — one translation unit per tensor-core rollout shape (compile with -DNOC_TC_SHAPE=k); see noc_tc_rollout.cuh.
#include "noc_tc_rollout.cuh"

// tuning knobs (overridable with -D for experiments): epilogue chunk and CTAs per SM the register budget is set for
#ifndef NOC_TC_CH0
#define NOC_TC_CH0 16
#endif
#ifndef NOC_TC_SPLIT0
#define NOC_TC_SPLIT0 4
#endif
#ifndef NOC_TC_CH3
#define NOC_TC_CH3 16
#endif
#ifndef NOC_TC_MINB3
#define NOC_TC_MINB3 3
#endif
#ifndef NOC_TC_CH1
#define NOC_TC_CH1 16
#endif
#ifndef NOC_TC_MINB1
#define NOC_TC_MINB1 5
#endif

namespace noc {
//                              kind NA CH minb
#if NOC_TC_SHAPE == 0
using Shape = TcShape<2, 1, NOC_TC_CH0, 1, NOC_TC_SPLIT0>;   // one quadcopter, d = 12 (singlequad: m = 128, one 16-warp CTA per SM, 4 threads per sample)
#elif NOC_TC_SHAPE == 1
using Shape = TcShape<0, 2, NOC_TC_CH1, NOC_TC_MINB1>;     // Cross2D, 2 agents, d = 4 (softcorridor, swap2, hardcorridor)
#elif NOC_TC_SHAPE == 2
using Shape = TcShape<0, 4, 16, 3>;     // Cross2D, 4 agents, d = 8 (midcross4)
#elif NOC_TC_SHAPE == 3
using Shape = TcShape<0, 12, NOC_TC_CH3, NOC_TC_MINB3>;    // Cross2D, 12 agents, d = 24 (swap12)
#elif NOC_TC_SHAPE == 4
using Shape = TcShape<0, 6, 16, 3>;     // Cross2D, 6 agents, d = 12 (swap12_3pair)
#elif NOC_TC_SHAPE == 5
using Shape = TcShape<0, 8, 16, 3>;     // Cross2D, 8 agents, d = 16 (swap12_4pair)
#elif NOC_TC_SHAPE == 6
using Shape = TcShape<0, 10, 16, 3>;    // Cross2D, 10 agents, d = 20 (swap12_5pair)
#else
#error "NOC_TC_SHAPE must be 0..6"
#endif

#define NOC_TC_NAME2(k) launch_tc_##k
#define NOC_TC_NAME(k) NOC_TC_NAME2(k)
int NOC_TC_NAME(NOC_TC_SHAPE)(const RolloutCall<float>& c) { return launch_tc<Shape>(c); }
}  // namespace noc
