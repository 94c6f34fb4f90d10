// Host build of the outlier policy of the C++ façade (ecb::outlierRejection, include/ecb/event_calib.hpp) for the CPU test suite.
// Links libecb.so (loads without a GPU) but makes no compute call.
#include "../../include/ecb/event_calib.hpp"

// groups[n] (ecb_residual_group) -> returns s; *threshold, drop[n]
extern "C" double host_outlier_policy(const ecb_residual_group *groups, int n, double k, double *threshold, uint8_t *drop) {
    std::vector<uint8_t> d;
    const double s = ecb::outlierRejection(std::vector<ecb_residual_group>(groups, groups + n), k, threshold, &d);
    std::copy(d.begin(), d.end(), drop);
    return s;
}
