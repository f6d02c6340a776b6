// host.cc -- host-side pieces of libppq_b200: ABI/version info, error strings, variant knobs and the host
// compute_mse_loss (the reference's is a host function too: /root/reference/ppq/csrc/cpu/hist_mse.cc:3-28).
#include <cuda_runtime.h>
#include <string.h>

#include <atomic>

#include "../../include/ppq_b200.h"
#include "variants.h"

namespace ppqb {
static std::atomic<int> g_variants[kVarCount];
int variant_of(int key) { return (key >= 0 && key < kVarCount) ? g_variants[key].load(std::memory_order_relaxed) : 0; }
static int key_of(const char *name) {
    if (!name) return -1;
    if (!strcmp(name, "linear_quant_t")) return kVarLinearT;
    if (!strcmp(name, "histogram")) return kVarHistogram;
    if (!strcmp(name, "minmax")) return kVarMinMax;
    if (!strcmp(name, "linear_quant_c")) return kVarChannel;
    if (!strcmp(name, "kl_search")) return kVarKlSearch;
    if (!strcmp(name, "select")) return kVarSelect;
    if (!strcmp(name, "multi_histogram")) return kVarMultiHist;
    return -1;
}
}  // namespace ppqb

extern "C" {

int ppq_b200_abi_version(void) { return 1; }

const char *ppq_b200_error_string(int status) {
    if (status == 0) return "success";
    return cudaGetErrorString((cudaError_t)status);
}

const char *ppq_b200_build_info(void) {
    return "libppq_b200 abi 1; sm_100a; host compiler gcc " __VERSION__ "; built " __DATE__;
}

int ppq_b200_set_variant(const char *kernel, int variant) {
    const int k = ppqb::key_of(kernel);
    if (k < 0 || variant < 0) return (int)cudaErrorInvalidValue;
    ppqb::g_variants[k].store(variant, std::memory_order_relaxed);
    return 0;
}
int ppq_b200_get_variant(const char *kernel) {
    const int k = ppqb::key_of(kernel);
    return k < 0 ? -1 : ppqb::variant_of(k);
}

// Per-bin error model of a (start, step, end) quantisation grid laid over the histogram, fp32 accumulation in bin order.
float ppq_b200_compute_mse_loss(const int64_t *hist, int64_t nbins, int start, int step, int end) {
    int64_t total = 0;
    for (int64_t i = 0; i < nbins; i++) total += hist[i];
    const float ftotal = (float)total;
    float loss = 0.0f;
    for (int64_t i = 0; i < nbins; i++) {
        const int idx = (int)i;
        float err;
        if (idx < start) err = (float)((start - idx - 1) + 0.5);
        else if (idx > end) err = (float)((idx - end) + 0.5);
        else {
            const int64_t l = (idx - start) % step, r = step - l - 1;
            if (l == r) err = (float)(l + 0.25);
            else {
                const float le = (float)(l + 0.5), re = (float)(r + 0.5);
                err = le < re ? le : re;
            }
        }
        // three separately rounded fp32 operations (no contraction: this file is built with -ffp-contract=off)
        volatile float a = (float)hist[i] * err;
        volatile float b = a * err;
        volatile float c = b / ftotal;
        loss = loss + c;
    }
    return loss;
}

}  // extern "C"
