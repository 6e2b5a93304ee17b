// step_dispatch.cpp — checks dispatch_step (spiking-neural-networks_b200/csrc/step_spec.h), the one map from a run's StepSpec to the
// template arguments of the step kernels.  Built and run by tests/test_step_dispatch.py; prints STEP_DISPATCH_OK and the number of
// inputs checked on success.
#include <cstdio>
#include <initializer_list>

#include "step_spec.h"

using snn::StepSpec;

struct Reached {
    int model, chemg;
    bool ntrel, stdp, net;
};

static Reached dispatch(const StepSpec &s) {
    const Reached invalid{-1, -1, false, false, false};
    return snn::dispatch_step(s, invalid, [](auto k) {
        using K = decltype(k);
        return Reached{K::MODEL, K::CHEMG, K::NTREL, K::STDP, K::NET};
    });
}

int main() {
    int checked = 0, failed = 0;
    // every input the engine produces: chemg == 1 only on single lattices, chemg != 0 only with ntrel
    for (int model = 0; model < SNN_MODEL_COUNT; ++model)
        for (int chemg : {0, 1, 3})
            for (int ntrel = 0; ntrel < 2; ++ntrel)
                for (int stdp = 0; stdp < 2; ++stdp)
                    for (int net = 0; net < 2; ++net) {
                        if ((chemg == 1 && net) || (chemg != 0 && !ntrel)) continue;
                        const StepSpec s{model, chemg, ntrel != 0, stdp != 0, net != 0};
                        const Reached r = dispatch(s);
                        const int want_chemg = net ? (chemg ? 3 : 0) : chemg;
                        const bool want_ntrel = chemg != 0 || ntrel;
                        ++checked;
                        if (r.model != model || r.chemg != want_chemg || r.ntrel != want_ntrel || r.stdp != (stdp != 0) || r.net != (net != 0)) {
                            std::printf("model %d chemg %d ntrel %d stdp %d net %d -> Spec<%d, %d, %d, %d, %d>\n", model, chemg, ntrel, stdp, net,
                                        r.model, r.chemg, r.ntrel, r.stdp, r.net);
                            ++failed;
                        }
                    }
    for (int model : {-1, (int)SNN_MODEL_COUNT, SNN_MODEL_COUNT + 7}) {
        ++checked;
        if (dispatch(StepSpec{model, 0, false, false, false}).model != -1) {
            std::printf("model %d was dispatched\n", model);
            ++failed;
        }
    }
    if (failed) return 1;
    std::printf("STEP_DISPATCH_OK %d\n", checked);
    return 0;
}
