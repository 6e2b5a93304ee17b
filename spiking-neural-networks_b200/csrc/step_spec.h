// step_spec.h — the run-time specialisation key of the step kernels and the one place that turns it into their template
// arguments.  Plain C++17 without CUDA, so that tests/cpp/step_dispatch.cpp can check the mapping with a host compiler.
#pragma once
#include "../../include/snn_b200.h"

namespace snn {

// chemg: 0 no chemical gather, 1 one neurotransmitter type in the whole node array, 3 general; ntrel: neurotransmitter /
// receptor state is present and must be stepped; net: several lattices and/or spike trains share the node array
struct StepSpec {
    int model = 0;
    int chemg = 0;
    bool ntrel = false, stdp = false, net = false;
};

// the compile-time image of a StepSpec, passed to the launchers' kernel-specific code
template <int MODEL_, int CHEMG_, bool NTREL_, bool STDP_, bool NET_>
struct Spec {
    static constexpr int MODEL = MODEL_, CHEMG = CHEMG_;
    static constexpr bool NTREL = NTREL_, STDP = STDP_, NET = NET_;
};

namespace detail {
template <int MODEL, int CHEMG, bool NTREL, bool NET, typename R, typename F>
R dispatch_stdp(const StepSpec &s, F &f) {
    if (s.stdp) return f(Spec<MODEL, CHEMG, NTREL, true, NET>{});
    return f(Spec<MODEL, CHEMG, NTREL, false, NET>{});
}

// 7 (CHEMG, NTREL, NET) combinations: networks gather chemistry through per-edge masks only, and chemistry implies NTREL
template <int MODEL, typename R, typename F>
R dispatch_chem(const StepSpec &s, F &f) {
    if (s.net) {
        if (s.chemg) return dispatch_stdp<MODEL, 3, true, true, R>(s, f);
        if (s.ntrel) return dispatch_stdp<MODEL, 0, true, true, R>(s, f);
        return dispatch_stdp<MODEL, 0, false, true, R>(s, f);
    }
    if (s.chemg == 1) return dispatch_stdp<MODEL, 1, true, false, R>(s, f);
    if (s.chemg == 3) return dispatch_stdp<MODEL, 3, true, false, R>(s, f);
    if (s.ntrel) return dispatch_stdp<MODEL, 0, true, false, R>(s, f);
    return dispatch_stdp<MODEL, 0, false, false, R>(s, f);
}
}  // namespace detail

// f(Spec<...>{}) for the instantiation that steps `s`: 9 models x 7 x 2 specialisations; `invalid` for an unknown model
template <typename R, typename F>
R dispatch_step(const StepSpec &s, R invalid, F &&f) {
    switch (s.model) {
    case SNN_MODEL_LEAKY_INTEGRATE_AND_FIRE: return detail::dispatch_chem<SNN_MODEL_LEAKY_INTEGRATE_AND_FIRE, R>(s, f);
    case SNN_MODEL_QUADRATIC_INTEGRATE_AND_FIRE: return detail::dispatch_chem<SNN_MODEL_QUADRATIC_INTEGRATE_AND_FIRE, R>(s, f);
    case SNN_MODEL_ADAPTIVE_LEAKY_INTEGRATE_AND_FIRE: return detail::dispatch_chem<SNN_MODEL_ADAPTIVE_LEAKY_INTEGRATE_AND_FIRE, R>(s, f);
    case SNN_MODEL_ADAPTIVE_EXP_LEAKY_INTEGRATE_AND_FIRE: return detail::dispatch_chem<SNN_MODEL_ADAPTIVE_EXP_LEAKY_INTEGRATE_AND_FIRE, R>(s, f);
    case SNN_MODEL_IZHIKEVICH: return detail::dispatch_chem<SNN_MODEL_IZHIKEVICH, R>(s, f);
    case SNN_MODEL_LEAKY_IZHIKEVICH: return detail::dispatch_chem<SNN_MODEL_LEAKY_IZHIKEVICH, R>(s, f);
    case SNN_MODEL_SIMPLE_LEAKY_INTEGRATE_AND_FIRE: return detail::dispatch_chem<SNN_MODEL_SIMPLE_LEAKY_INTEGRATE_AND_FIRE, R>(s, f);
    case SNN_MODEL_HODGKIN_HUXLEY: return detail::dispatch_chem<SNN_MODEL_HODGKIN_HUXLEY, R>(s, f);
    case SNN_MODEL_BCM_IZHIKEVICH: return detail::dispatch_chem<SNN_MODEL_BCM_IZHIKEVICH, R>(s, f);
    }
    return invalid;
}

}  // namespace snn
