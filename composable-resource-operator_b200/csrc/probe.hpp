// probe.hpp — the long-lived probe context behind the C ABI.
//
// Takes the slot of utils.RunNvidiaSmi + utils.CheckGPUVisible in
// handleAttachingState (internal/controller/composableresource_controller.go:259,275;
// internal/utils/gpus.go:666-689, 54-86).  One Device per managed GPU holds the
// resident sweep buffers (2*S bytes: halves A and B), two streams, the timing
// events, the reduction scratch and the device-written result struct, so a warm
// probe is one cudaGraphLaunch and one 512-byte copy-back.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/croprobe.h"
#include "kernels.cuh"

namespace cro {

// Everything ONE probe in flight owns.  A device has two lanes, so a second probe can be enqueued behind a running
// one (cro_probe_begin twice): its kernels start the moment the first probe's finalize kernel retires, with no host
// round trip in between — what keeps a GPU busy when one reconcile worker feeds eight of them.
struct Lane {
    ProbeParams* d_params = nullptr;   // what the graph's kernels read
    ProbeParams* h_params = nullptr;   // pinned; refreshed by the host before each launch
    SweepOut* d_out = nullptr;         // device sweep-result slots (lane 0: kSlotCount, lane 1: the first 64)
    SweepOut* h_out = nullptr;         // pinned host mirror
    cro_probe_result* d_result = nullptr;  // written by the finalize kernels; lane 0's is the all-gather send buffer
    cro_probe_result* h_result = nullptr;  // pinned copy-back target
    std::vector<cudaEvent_t> evpool;   // per-sweep timing events of the full probe (bench / tests read them)
    cudaEvent_t ev_done = nullptr;     // recorded behind the probe's last copy-back
    // the whole probe captured as one CUDA graph (timing events are external event-record nodes)
    cudaGraphExec_t graph_exec = nullptr;
    uint64_t graph_key = 0;
    size_t graph_events = 0;
    bool graph_failed = false;
    size_t events = 0;                 // timing events the in-flight / last probe recorded
    uint32_t reads = 0, copies = 0;
    bool timed = false;                // the events of the last probe on this lane are valid
    bool in_flight = false;
    std::chrono::steady_clock::time_point since{};
};

struct Device {
    int ordinal = -1;              // CUDA ordinal
    int index = -1;                // rank: position in the minor-sorted list
    cro_dev_info info{};
    std::mutex mu;
    cudaStream_t stream = nullptr; // every sweep
    cudaStream_t aux = nullptr;    // the closed-form generator (ALU only) runs beside the copy sweeps
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_fork = nullptr, ev_join = nullptr;
    Lane lanes[2];
    int lane_head = 0;                 // oldest probe in flight
    int lane_count = 0;                // probes in flight (0..2)
    int last_lane = 0;                 // lane of the most recently COLLECTED probe (cro_probe_sweep_times)
    unsigned char* region = nullptr;   // [0,S) half A, [S,2S) half B
    uint64_t sweep_bytes = 0;
    uint64_t seed_dev = 0;             // seed_base | minor
    uint64_t seed_cur = 0;             // seed of the pattern half A holds (or will hold after the next fill)
    uint64_t nonce_cur = 0;            // ... and its nonce
    uint64_t nonce_next = 0;           // nonce the next probe takes
    bool filled = false;
    KernelPlan plan{};
    SweepScratch scratch{}, scratch_aux{}, scratch_pfx{};   // main stream / closed form / p2p prefix closed form
    // lane 0's buffers under their old names: the synchronous probe, the single sweeps and cro_probe_all use lane 0
    SweepOut*& d_out = lanes[0].d_out;
    SweepOut*& h_out = lanes[0].h_out;
    cro_probe_result*& d_result = lanes[0].d_result;
    cro_probe_result*& h_result = lanes[0].h_result;
    cro_probe_result* d_tmpl = nullptr;    // identity + options, staged by the host
    cro_probe_result* d_gather = nullptr;  // all-gather receive buffer (world entries)
    cro_probe_result* h_gather = nullptr;  // pinned, CRO_MAX_DEVICES entries
    cro_probe_result tmpl{};               // host copy of d_tmpl
    // NVLink latency: tables[j] is the permutation device j chases THROUGH this device's memory
    std::vector<unsigned long long*> d_chase_tables;
    std::vector<unsigned> chase_expect;    // where this device's chase into peer j must end (hops of the last build)
    unsigned chase_hops_built = 0;
    unsigned long long* d_chase_out = nullptr;
    unsigned long long* h_chase_out = nullptr;   // pinned, 2 * CRO_MAX_DEVICES
    std::vector<cudaEvent_t> ev_push_done, ev_reread_done;   // one per NVLink round
    cudaEvent_t ev_hbm_done = nullptr, ev_aux_done = nullptr, ev_chase_ready = nullptr;
    // asynchronous probes (ctx_probe_begin / ctx_probe_end): results drained off the stream but not yet collected
    struct Collected { cro_probe_result r; int rc; std::chrono::steady_clock::time_point at; };
    std::deque<Collected> done;
    unsigned sm_clock_mhz = 0, mem_clock_mhz = 0;
    uint32_t ecc_uncorrected = 0;      // NVML count cached at init / full-box probe / failed probe
    std::chrono::steady_clock::time_point ecc_at{};   // last NVML read by cro_probe_all
    cro_probe_result last{};           // the most recent collected result (cro_metrics_text)
    bool have_last = false;

    Device() = default;
    Device(const Device&) = delete;
    Device& operator=(const Device&) = delete;
    // Releases every CUDA object this device owns (probe.cu).  Runs for half-built devices too,
    // so a cro_probe_init that fails midway (OOM on the sweep region) leaks nothing.
    ~Device();
};

// Phases of the most recent cro_probe_all, host wall clock + device windows (bench "fullbox").
struct FullBoxTimes {
    uint64_t enqueue_ns = 0;       // host time to enqueue everything
    uint64_t wall_ns = 0;          // host wall clock of the whole call
    uint64_t hbm_ns = 0;           // max over devices of the HBM probe (device timers)
    uint64_t p2p_ns = 0;           // first NVLink kernel start .. last NVLink kernel end (device timers, max over devices)
    uint64_t chase_ns = 0;         // max chase duration
    uint64_t gather_ns = 0;        // all-gather, CUDA events on rank 0's stream
    uint32_t rounds = 0;
    uint32_t host_syncs = 0;       // stream synchronisations the call performed
    uint32_t gather = 0;           // CRO_GATHER_*
};

}  // namespace cro

struct cro_ctx {
    cro_opts opts{};
    std::vector<std::unique_ptr<cro::Device>> devs;   // minor-sorted
    std::atomic<uint64_t> launches{0};
    // gauges / counters behind cro_metrics_text (the operator's Prometheus registry, cmd/main.go:66,119-125)
    std::atomic<uint64_t> m_probes{0}, m_probe_failures{0}, m_fullbox{0}, m_helper_probes{0}, m_helper_failures{0};
    std::mutex err_mu;
    std::string last_error;
    std::mutex all_mu;                 // serialises cro_probe_all
    void* nccl_lib = nullptr;
    std::vector<void*> nccl_comms;     // ncclComm_t per device
    bool nccl_ready = false;
    bool peers_enabled = false;
    bool nvtx = true;
    std::string proc_root = "/proc";   // where the node's /proc is mounted (tests point it at a fake tree)
    bool proc_lists_mine = false;      // at init the registry listed one of this context's devices (ctx_create)
    // the node's inventory as of the last enumeration (inventory.hpp)
    std::mutex inv_mu;
    std::string inv_key;               // uuid/minor set the cached list was built from
    std::vector<cro_dev_info> inv;
    bool inv_valid = false;
    bool inv_refreshing = false;       // a background full re-read is under way
    std::thread inv_thread;
    std::chrono::steady_clock::time_point inv_full_at{};   // last time the `information` files were read
    std::chrono::steady_clock::time_point inv_nvml_at{};   // last NVML re-initialisation (rate limit when /proc is absent)
    std::atomic<uint64_t> inv_rescans{0};                  // times the inventory had to be rebuilt
    cro::FullBoxTimes fullbox{};
    // NCCL entry points, resolved once
    int (*ncclCommInitAll)(void**, int, const int*) = nullptr;
    int (*ncclGroupStart)() = nullptr;
    int (*ncclGroupEnd)() = nullptr;
    int (*ncclAllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    const char* (*ncclGetErrorString)(int) = nullptr;

    void set_error(const std::string& m) {
        std::lock_guard<std::mutex> g(err_mu);
        last_error = m;
    }
    // a context that dies during cro_probe_init hands its error text to the calling thread
    // (cro_last_error(NULL, ...)); defined in probe.cu
    ~cro_ctx();
};

namespace cro {

const std::string& last_init_error();   // calling thread's last failed ctx_create (or exception stopped at the C ABI)
void set_thread_error(const std::string& m) noexcept;
int ctx_create(const cro_opts* o, cro_ctx** out);
void ctx_destroy(cro_ctx* c);
int ctx_probe_device(cro_ctx* c, int idx, cro_probe_result* out);
int ctx_probe_all(cro_ctx* c, cro_probe_result* out, int cap, int* n);
int ctx_probe_begin(cro_ctx* c, int idx);
int ctx_probe_end(cro_ctx* c, int idx, cro_probe_result* out);
int ctx_probe_poll(cro_ctx* c, int idx);
int ctx_probe_wait(cro_ctx* c, int idx);
int ctx_probe_depth(cro_ctx* c, int idx);
std::string ctx_metrics_text(cro_ctx* c);
int ctx_sweep_times(cro_ctx* c, int idx, cro_sweep_time* out, int cap, int* n);
// Fresh inventory of the node merged with the context's own devices (inventory.hpp).
// force: re-read every `information` file even if the registry's listing looks unchanged (done by itself once a
// second, and by the callers whenever a UUID they were told about is NOT in the list they got).
int ctx_inventory(cro_ctx* c, std::vector<cro_dev_info>* out, bool force = false);
// Probe by UUID: in-process device, helper process for one attached after init, CRO_ERR_NO_DEVICE when not on the node.
int ctx_probe_uuid(cro_ctx* c, const char* uuid, cro_probe_result* out);
int ctx_p2p_detail(cro_ctx* c, int idx, int peer, cro_p2p_detail* out);

// single sweeps (each takes the device mutex)
int ctx_fill(cro_ctx* c, int idx, uint32_t iters, cro_sweep_result* out);
int ctx_read(cro_ctx* c, int idx, uint32_t variant, uint32_t iters, bool dst_half, cro_sweep_result* out);
int ctx_copy(cro_ctx* c, int idx, uint32_t variant, uint32_t iters, cro_sweep_result* out);
int ctx_expected(cro_ctx* c, int idx, cro_sweep_result* out);
int ctx_inject(cro_ctx* c, int idx, uint64_t word, uint64_t mask);
int ctx_read_words(cro_ctx* c, int idx, uint64_t first, uint64_t n, uint64_t* out);

uint32_t resolve_read_variant(uint32_t v, uint64_t bytes);
uint32_t resolve_copy_variant(uint32_t v);

// Host restatement of the latency permutation of one directed pair (Sattolo cycle over kChaseSlots slots,
// mt19937_64 seeded with minor_src * 8 + minor_dst; SURVEY.md §8d config 3): perm[i] = successor of slot i.
constexpr uint32_t kChaseSlots = 65536;
void chase_permutation(int minor_src, int minor_dst, std::vector<uint32_t>* perm);

}  // namespace cro
