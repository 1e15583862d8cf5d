// Library-level entry points: version, error strings, workspace sizing, launch counter.
#include "common.cuh"

namespace ssdhead {
std::atomic<unsigned long long> g_launch_count{0};
size_t loss_workspace_bytes(int B, int P, int C);          // loss.cu
size_t detect_workspace_bytes(int B, int P, int C, int n); // detect.cu
size_t resident_rows_bytes(int B, int P);                   // loss.cu
}  // namespace ssdhead

using namespace ssdhead;

extern "C" {

int ssdhead_abi_version(void) { return SSDHEAD_ABI_VERSION; }

uint64_t ssdhead_launch_count(void) { return (uint64_t)g_launch_count.load(std::memory_order_relaxed); }

const char* ssdhead_error_string(int code)
{
    switch (code) {
        case 0: return "ok";
        case SSDHEAD_E_BADARG: return "ssdhead: bad argument (null pointer or negative size)";
        case SSDHEAD_E_UNSUPPORTED: return "ssdhead: unsupported shape (C must be 21; P limited by shared memory)";
        case SSDHEAD_E_WORKSPACE: return "ssdhead: workspace too small";
        case SSDHEAD_E_ALIGN: return "ssdhead: pointer not 16-byte aligned";
        case SSDHEAD_E_STATE: return "ssdhead: host context misuse";
        default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "ssdhead: unknown error";
}

size_t ssdhead_workspace_bytes(int which, int B, int P, int C, int n)
{
    if (B < 0 || P < 0 || C < 0 || n < 0) return 0;
    switch (which) {
        case SSDHEAD_WS_MATCH:
            return match_ws_bytes(B, n);
        case SSDHEAD_WS_LOSS:
            return loss_workspace_bytes(B, P, C);
        case SSDHEAD_WS_DETECT:
        case SSDHEAD_WS_NMS:
            return detect_workspace_bytes(B, P, C, n);
        case SSDHEAD_WS_ROWS:
            return resident_rows_bytes(B, P);
        default:
            return 0;
    }
}

}  // extern "C"
