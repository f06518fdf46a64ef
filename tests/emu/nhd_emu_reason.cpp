/*
 * nhd_emu_reason.cpp — TEST INFRASTRUCTURE.  node_reason (nhd_b200/csrc/nhd_core.cuh, the per-thread logic of
 * explain_kernel) compiled with g++ and driven by a plain serial loop, so that the explanation the device computes
 * can be diffed against the explanation oracle (tests/explain_model.py) on a machine without a GPU.
 * Built by tests/test_explain.py; never linked into the product library.
 */
#include "../../nhd_b200/csrc/nhd_core.cuh"

using namespace nhd;

extern "C" int nhd_emu_reason(double bw, double min_busy, const double* speed, int n_nodes, const nhd_node_rec* recs,
                              const nhd_pod* pod, double now, uint8_t* out)
{
    double cap[NHD_MAX_SPEED_CLASSES];
    for (int i = 0; i < NHD_MAX_SPEED_CLASSES; i++) cap[i] = speed[i] * bw;
    PodType t;
    make_pod_type(*pod, t);
    for (int n = 0; n < n_nodes; n++) out[n] = (uint8_t)node_reason(recs[n], t, cap, now, min_busy);
    return 0;
}
