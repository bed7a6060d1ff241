#include "host_common.h"

#include <stdlib.h>

#include <new>

#include <mutex>
#include <vector>

#include "../../include/omg_b200.h"

namespace omg {

thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};

bool pdl_enabled() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("OMG_PDL");
        v = (e && e[0] == '1') ? 1 : 0;
    }
    return v == 1;
}

PFN_encodeTiled get_encode_tiled() {
    static PFN_encodeTiled fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    });
    return fn;
}

int make_tmap_16b(CUtensorMap* out, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_elems,
                  const uint32_t* box, CUtensorMapSwizzle swizzle, CUtensorMapDataType dtype) {
    PFN_encodeTiled enc = get_encode_tiled();
    OMG_CHECK(enc != nullptr, "cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
    cuuint64_t gdim[5], gstr[5];
    cuuint32_t bdim[5], estr[5];
    for (int i = 0; i < rank; ++i) {
        gdim[i] = dims[i];
        bdim[i] = box[i];
        estr[i] = 1;
        if (i > 0) {
            gstr[i - 1] = strides_elems[i] * 2;  // bytes
            OMG_CHECK(gstr[i - 1] % 16 == 0, "tensor map stride %d (%llu B) not a multiple of 16 B", i,
                      (unsigned long long)gstr[i - 1]);
        }
        OMG_CHECK(box[i] >= 1 && box[i] <= 256, "tensor map box dim %d = %u out of range", i, box[i]);
    }
    OMG_CHECK((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "tensor map base pointer not 16 B aligned");
    CUresult r = enc(out, dtype, rank, const_cast<void*>(ptr), gdim, gstr, bdim, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    OMG_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return 0;
}

}  // namespace omg

// ------------------------------------------------------------------------------------------------ launch plans
struct omg_plan {
    std::vector<std::function<int(void*)>> steps;
};

namespace omg {
static thread_local omg_plan* g_recording = nullptr;
bool plan_recording() { return g_recording != nullptr; }
void plan_note(std::function<int(void*)> step) {
    if (g_recording) g_recording->steps.push_back(std::move(step));
}
}  // namespace omg

extern "C" omg_plan* omg_plan_create(void) { return new (std::nothrow) omg_plan(); }

extern "C" void omg_plan_destroy(omg_plan* plan) {
    if (plan && omg::g_recording == plan) omg::g_recording = nullptr;
    delete plan;
}

extern "C" int omg_plan_record_begin(omg_plan* plan) {
    OMG_CHECK(plan != nullptr, "omg_plan_record_begin: null plan");
    OMG_CHECK(omg::g_recording == nullptr, "omg_plan_record_begin: this thread is already recording a plan");
    omg::g_recording = plan;
    return 0;
}

extern "C" int omg_plan_record_end(omg_plan* plan) {
    OMG_CHECK(plan != nullptr && omg::g_recording == plan, "omg_plan_record_end: this plan is not being recorded on this thread");
    omg::g_recording = nullptr;
    return 0;
}

extern "C" int omg_plan_length(const omg_plan* plan) { return plan ? (int)plan->steps.size() : -1; }

extern "C" int omg_plan_clear(omg_plan* plan) {
    OMG_CHECK(plan != nullptr && omg::g_recording != plan, "omg_plan_clear: null plan, or the plan is being recorded");
    plan->steps.clear();
    return 0;
}

extern "C" int omg_plan_run(const omg_plan* plan, void* stream) {
    OMG_CHECK(plan != nullptr, "omg_plan_run: null plan");
    OMG_CHECK(omg::g_recording != plan, "omg_plan_run: the plan is still being recorded");
    for (const auto& step : plan->steps) {
        const int rc = step(stream);
        if (rc != 0) return rc;  // omg_last_error() holds the failing launch's message
    }
    return 0;
}

extern "C" const char* omg_last_error(void) { return omg::g_err; }
extern "C" const char* omg_version(void) { return "omg_b200 0.1 sm_100a"; }
extern "C" uint64_t omg_launch_count(void) { return omg::g_launches.load(); }
