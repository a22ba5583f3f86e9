// probe.cu — probe context: enumeration, resident sweep buffers, the probe as
// one CUDA graph with a device-written verdict, and the full-box probe
// (concurrent HBM probes, NVLink rounds chained by events, one NCCL all-gather).
//
// Reference slot: utils.RunNvidiaSmi (internal/utils/gpus.go:666-689) and
// utils.CheckGPUVisible (internal/utils/gpus.go:54-86) as called from
// handleAttachingState (internal/controller/composableresource_controller.go:259,275).
#include "probe.hpp"

#include <dlfcn.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <thread>

#include <nvtx3/nvToolsExt.h>

#include "env.hpp"
#include "identity.hpp"
#include "inventory.hpp"

namespace cro {

namespace {

constexpr uint64_t kDefaultSweep = 4ull << 30;
constexpr uint64_t kDefaultP2P = 1ull << 30;
constexpr uint64_t kDefaultSeedBase = 0x00C0FFEE00000000ull;
// 1024 hops: the mean hop latency — and every pair's own value — is the same to 0.1 % at 1 Ki, 4 Ki, 16 Ki and 64 Ki hops
// (8 GPUs: 1779.4 / 1780.0 / 1780.4 / 1780.6 ns; 2 GPUs: 1860.4 / 1862.7 / 1861.7 / 1861.6; profiles/r02_latency_vs_hops.md),
// while 64 Ki hops of ~1.8 us would be 122 ms, three times the rest of the full-box probe.  SURVEY.md §8d's 64 Ki is one
// cro_set_latency_hops / latency_hops away, and bench.py runs all four lengths every time.
constexpr uint32_t kDefaultHops = 1024;

#define CU_TRY(ctx, expr)                                                              \
    do {                                                                               \
        cudaError_t e__ = (expr);                                                      \
        if (e__ != cudaSuccess) {                                                      \
            (ctx)->set_error(std::string(#expr) + ": " + cudaGetErrorString(e__));     \
            return e__ == cudaErrorMemoryAllocation ? CRO_ERR_OOM : CRO_ERR_CUDA;      \
        }                                                                              \
    } while (0)

uint64_t ms_to_ns(float ms) { return (uint64_t)((double)ms * 1.0e6 + 0.5); }
uint64_t now_ns() {
    return (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// NVTX ranges around the host-side phases (SURVEY.md §5); nsys / ncu --nvtx pick them up, nothing else pays.
struct Range {
    bool on;
    Range(const cro_ctx* c, const char* name) : on(c->nvtx) { if (on) nvtxRangePushA(name); }
    ~Range() { if (on) nvtxRangePop(); }
};

Params imm_params(const Device* d) { return Params{ProbeParams{d->seed_cur, d->nonce_cur}, nullptr}; }
Params graph_params(const Lane& L) { return Params{ProbeParams{0, 0}, L.d_params}; }
uint64_t seed_of(const Device* d, uint64_t nonce) { return d->seed_dev + nonce * kNonceStride; }

int ensure_region(cro_ctx* c, Device* d) {
    if (d->region) return CRO_OK;
    CU_TRY(c, cudaSetDevice(d->ordinal));
    // A device that is already in use may not have 2*S free (the reference's own pre-check for that
    // is CheckNoGPULoads, internal/utils/gpus.go:88).  Degrade: halve S down to 64 MiB — still far
    // beyond the 126 MB L2 when doubled — and report the size actually swept in the result.
    const uint64_t asked = d->sweep_bytes;
    cudaError_t e = cudaErrorMemoryAllocation;
    for (uint64_t s = asked;; s = (s / 2) & ~(uint64_t)15) {
        e = cudaMalloc(&d->region, 2 * s);
        if (e == cudaSuccess) {
            if (s != d->sweep_bytes) {
                d->sweep_bytes = s;
                for (Lane& L : d->lanes)
                    if (L.graph_exec) { cudaGraphExecDestroy(L.graph_exec); L.graph_exec = nullptr; }
            }
            break;
        }
        cudaGetLastError();
        d->region = nullptr;
        if (e != cudaErrorMemoryAllocation || s <= (64ull << 20) || !(c->opts.flags & CRO_F_DEGRADE_ON_OOM)) {
            c->set_error("cudaMalloc of sweep region (" + std::to_string(2 * s) + " bytes, asked for " +
                         std::to_string(2 * asked) + ") failed: " + cudaGetErrorString(e));
            return CRO_ERR_OOM;
        }
    }
    d->filled = false;
    return CRO_OK;
}

int ensure_filled(cro_ctx* c, Device* d) {
    int rc = ensure_region(c, d);
    if (rc) return rc;
    if (d->filled) return CRO_OK;
    CU_TRY(c, launch_fill(d->plan, d->region, d->sweep_bytes, imm_params(d), d->scratch, nullptr, d->stream));
    c->launches++;
    d->filled = true;
    return CRO_OK;
}

// Waits for the stream, honouring opts.deadline_ms (kernels cannot be
// cancelled; on expiry the caller gets CRO_ERR_DEADLINE and the next call on
// this device synchronises first because it takes the same stream).
int wait_stream(cro_ctx* c, Device* d) {
    if (c->opts.deadline_ms <= 0) {
        CU_TRY(c, cudaStreamSynchronize(d->stream));
        return CRO_OK;
    }
    const auto until = std::chrono::steady_clock::now() + std::chrono::milliseconds(c->opts.deadline_ms);
    for (;;) {
        cudaError_t q = cudaStreamQuery(d->stream);
        if (q == cudaSuccess) return CRO_OK;
        if (q != cudaErrorNotReady) {
            c->set_error(std::string("cudaStreamQuery: ") + cudaGetErrorString(q));
            return CRO_ERR_CUDA;
        }
        if (std::chrono::steady_clock::now() > until) {
            c->set_error("probe deadline of " + std::to_string(c->opts.deadline_ms) + " ms exceeded");
            return CRO_ERR_DEADLINE;
        }
        std::this_thread::sleep_for(std::chrono::microseconds(50));
    }
}

void copy_cstr(char* dst, size_t cap, const std::string& s) {
    memset(dst, 0, cap);
    memcpy(dst, s.data(), std::min(cap - 1, s.size()));
}

int alloc_scratch(cro_ctx* c, SweepScratch* sc, int max_grid) {
    CU_TRY(c, cudaMalloc(&sc->partials, sizeof(ulonglong4) * (size_t)max_grid));
    CU_TRY(c, cudaMalloc(&sc->counter, sizeof(unsigned)));
    CU_TRY(c, cudaMalloc(&sc->tmin, sizeof(unsigned long long)));
    CU_TRY(c, cudaMalloc(&sc->tmax, sizeof(unsigned long long)));
    CU_TRY(c, cudaMalloc(&sc->tile_ctr, sizeof(unsigned long long)));
    CU_TRY(c, cudaMemset(sc->tile_ctr, 0, sizeof(unsigned long long)));
    CU_TRY(c, cudaMemset(sc->counter, 0, sizeof(unsigned)));
    CU_TRY(c, cudaMemset(sc->tmin, 0xFF, sizeof(unsigned long long)));
    CU_TRY(c, cudaMemset(sc->tmax, 0, sizeof(unsigned long long)));
    return CRO_OK;
}
void free_scratch(SweepScratch* sc) {
    cudaFree(sc->partials);
    cudaFree(sc->counter);
    cudaFree(sc->tmin);
    cudaFree(sc->tmax);
    cudaFree(sc->tile_ctr);
}

}  // namespace

uint32_t resolve_read_variant(uint32_t v, uint64_t bytes) {
    // AUTO: the TMA ring has the higher asymptote (7.47 vs 7.36 TB/s at 4 GiB) but ~5.5 us more constant cost per launch
    // (ring ramp and drain, profiles/r02_fixed_cost.md), so small sweeps go to plain 256-bit LDG.  Whole probes, median of
    // 30 (profiles/r02_auto_threshold.jsonl): 256 MiB 732 us with LDG.256 vs 755 with TMA, 512 MiB 1342 vs 1357, 1 GiB
    // 2594 vs 2551, 2 GiB 5133 vs 5104 — the crossover sits between 512 MiB and 1 GiB.
    if (v == CRO_READ_AUTO) {
        v = env::get("CRO_READ_VARIANT");
        if (v == CRO_READ_AUTO) v = bytes <= (512ull << 20) ? CRO_READ_LDG256 : CRO_READ_TMA;
    }
    return (v == READ_LDG || v == READ_TMA || v == READ_LDG256) ? v : (uint32_t)READ_TMA;
}
uint32_t resolve_copy_variant(uint32_t v) {
    if (v == CRO_COPY_AUTO) {
        v = env::get("CRO_COPY_VARIANT");
        if (v == CRO_COPY_AUTO) v = CRO_COPY_TMA_FUSED;
    }
    return (v == COPY_LDG || v == COPY_TMA || v == COPY_TMA_FUSED) ? v : (uint32_t)COPY_TMA_FUSED;
}

void chase_permutation(int minor_src, int minor_dst, std::vector<uint32_t>* perm) {
    perm->resize(kChaseSlots);
    for (uint32_t i = 0; i < kChaseSlots; ++i) (*perm)[i] = i;
    std::mt19937_64 rng((uint64_t)((long long)minor_src * 8 + (long long)minor_dst));
    for (uint32_t i = kChaseSlots - 1; i > 0; --i) {        // Sattolo: one cycle through every slot
        const uint32_t j = (uint32_t)(rng() % i);
        std::swap((*perm)[i], (*perm)[j]);
    }
}

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
// Caches the device's uncorrected volatile ECC count (0 when NVML is not the identity source or ECC is off).
static void refresh_ecc(cro_ctx* c, Device* d) {
    if ((c->opts.flags & CRO_F_NO_NVML) || d->info.identity_source != 1) return;
    unsigned long long ecc = 0;
    if (identity::NvmlEccUncorrected(std::string(d->info.gpu_uuid, strnlen(d->info.gpu_uuid, sizeof d->info.gpu_uuid)), &ecc))
        d->ecc_uncorrected = (uint32_t)std::min<unsigned long long>(ecc, 0xFFFFFFFFull);
}

// Stages the fields of the result that the device cannot know (identity strings, NVML readings, options)
// into the template the finalize kernel starts from.  Caller has the device current.
static int stage_template(cro_ctx* c, Device* d) {
    cro_probe_result& t = d->tmpl;
    memset(&t, 0, sizeof t);
    t.abi_version = CRO_ABI_VERSION;
    t.cuda_ordinal = d->ordinal;
    t.device_minor = d->info.device_minor;
    memcpy(t.gpu_uuid, d->info.gpu_uuid, sizeof t.gpu_uuid);
    memcpy(t.pci_bus_id, d->info.pci_bus_id, sizeof t.pci_bus_id);
    t.hbm_bytes_total = d->info.hbm_bytes_total;
    t.sweep_bytes = d->sweep_bytes;
    t.sm_count = d->info.sm_count;
    t.sm_clock_mhz = d->sm_clock_mhz;
    t.mem_clock_mhz = d->mem_clock_mhz;
    t.ecc_errors = d->ecc_uncorrected;
    t.rank = (uint8_t)(c->opts.rank_base + (uint32_t)d->index);
    t.world = (uint8_t)(c->opts.world_override ? c->opts.world_override : (uint32_t)c->devs.size());
    t.p2p_bytes = c->opts.p2p_bytes;
    if (c->peers_enabled)
        for (size_t j = 0; j < c->devs.size() && j < 8; ++j) {
            if ((int)j == d->index) continue;
            int can = 0;
            cudaDeviceCanAccessPeer(&can, d->ordinal, c->devs[j]->ordinal);
            t.p2p_access[j] = (uint8_t)can;
        }
    CU_TRY(c, cudaMemcpyAsync(d->d_tmpl, &t, sizeof t, cudaMemcpyHostToDevice, d->stream));
    CU_TRY(c, cudaStreamSynchronize(d->stream));    // `t` lives in pageable memory
    return CRO_OK;
}

int ctx_create(const cro_opts* o, cro_ctx** out) {
    if (!out) return CRO_ERR_INVALID_ARG;
    *out = nullptr;
    cro_opts opts;
    memset(&opts, 0, sizeof opts);
    if (o) opts = *o;
    else opts.abi_version = CRO_ABI_VERSION;
    if (opts.abi_version != CRO_ABI_VERSION) return CRO_ERR_ABI_MISMATCH;
    if (opts.sweep_bytes == 0) opts.sweep_bytes = kDefaultSweep;
    if (opts.sweep_bytes % 16 != 0 || opts.sweep_bytes < 16) return CRO_ERR_INVALID_ARG;
    if (opts.p2p_bytes == 0) opts.p2p_bytes = std::min(kDefaultP2P, opts.sweep_bytes);
    if (opts.p2p_bytes > opts.sweep_bytes || opts.p2p_bytes % 16 != 0) return CRO_ERR_INVALID_ARG;
    if (opts.seed_base == 0) opts.seed_base = kDefaultSeedBase;
    if (opts.read_sweeps == 0) opts.read_sweeps = 5;
    if (opts.copy_sweeps == 0) opts.copy_sweeps = 5;
    if (opts.read_sweeps > kMaxSweepsEach || opts.copy_sweeps > kMaxSweepsEach) return CRO_ERR_INVALID_ARG;
    if (opts.latency_hops == 0) opts.latency_hops = kDefaultHops;
    if (opts.n_devices < 0 || opts.n_devices > CRO_MAX_DEVICES) return CRO_ERR_INVALID_ARG;

    std::unique_ptr<cro_ctx> c(new cro_ctx);
    c->opts = opts;
    // CRO_TRACE_INIT=1: where the cold start goes, phase by phase, on stderr (the hot-plug helper pays all of it)
    const bool trace_init = getenv("CRO_TRACE_INIT") && getenv("CRO_TRACE_INIT")[0] == '1';
    uint64_t t_phase = now_ns();
    auto phase = [&](const char* name) {
        if (!trace_init) return;
        const uint64_t t = now_ns();
        fprintf(stderr, "cro_probe_init: %-28s %8.3f ms\n", name, (double)(t - t_phase) / 1e6);
        t_phase = t;
    };
    {
        // the CRO_* knobs, validated the way the reference validates its own environment
        // (internal/controller/composableresource_adapter.go:42-45)
        std::string why;
        if (!env::reload(&why)) {
            c->set_error(why);
            return CRO_ERR_INVALID_ARG;
        }
        c->nvtx = env::get("CRO_NVTX") != 0;
        if (const char* pr = getenv("CRO_PROC_ROOT"))
            if (*pr) c->proc_root = pr;
    }

    phase("options + environment");
    int n_cuda = 0;
    cudaError_t e = cudaGetDeviceCount(&n_cuda);
    phase("cuInit (cudaGetDeviceCount)");
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) {
        // No usable GPU.  A probe library without a GPU must say so loudly:
        // there is no CPU fallback on this path.
        cudaGetLastError();
        return CRO_ERR_NO_DEVICE;
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        return CRO_ERR_CUDA;
    }
    std::vector<int> ordinals;
    if (opts.n_devices > 0) {
        for (int i = 0; i < opts.n_devices; ++i) {
            if (opts.devices[i] < 0 || opts.devices[i] >= n_cuda) return CRO_ERR_INVALID_ARG;
            ordinals.push_back(opts.devices[i]);
        }
    } else {
        for (int i = 0; i < n_cuda && i < CRO_MAX_DEVICES; ++i) ordinals.push_back(i);
    }

    // Identity: /proc first (a directory walk, ~0.06 ms), NVML only when asked to (its first call costs
    // tens of ms and serialises across processes) — CRO_F_NO_NVML keeps it off the hot-plug path entirely.
    const std::vector<identity::ProcGpu> proc = identity::ScanProc(c->proc_root);
    std::vector<identity::NvmlGpu> nvml;
    bool have_nvml = false;
    if (!(opts.flags & CRO_F_NO_NVML)) have_nvml = identity::ScanNvml(&nvml, nullptr);

    phase("identity scan (/proc, NVML)");
    struct Keyed { std::unique_ptr<Device> d; long long key; };
    std::vector<Keyed> keyed;
    for (int ord : ordinals) {
        std::unique_ptr<Device> d(new Device);
        d->ordinal = ord;
        cudaDeviceProp prop;
        CU_TRY(c.get(), cudaGetDeviceProperties(&prop, ord));
        cro_dev_info& info = d->info;
        memset(&info, 0, sizeof info);
        info.cuda_ordinal = ord;
        info.device_minor = -1;
        const std::string uuid = identity::FormatGpuUuid(reinterpret_cast<const unsigned char*>(prop.uuid.bytes));
        copy_cstr(info.gpu_uuid, sizeof info.gpu_uuid, uuid);
        copy_cstr(info.pci_bus_id, sizeof info.pci_bus_id,
                  identity::FormatBusIdSmi((unsigned)prop.pciDomainID, (unsigned)prop.pciBusID,
                                           (unsigned)prop.pciDeviceID, 0));
        copy_cstr(info.name, sizeof info.name, prop.name);
        info.hbm_bytes_total = prop.totalGlobalMem;
        info.sm_count = (uint32_t)prop.multiProcessorCount;
        info.cc_major = (uint32_t)prop.major;
        info.cc_minor = (uint32_t)prop.minor;
        info.identity_source = 3;
        long long key = ((long long)prop.pciDomainID << 16) | ((long long)prop.pciBusID << 8) |
                        (long long)prop.pciDeviceID;
        bool matched = false;
        if (have_nvml) {
            for (size_t k = 0; k < nvml.size(); ++k) {
                if (nvml[k].uuid != uuid) continue;
                info.device_minor = nvml[k].minor;
                if (!nvml[k].bus_id.empty()) copy_cstr(info.pci_bus_id, sizeof info.pci_bus_id, nvml[k].bus_id);
                info.identity_source = 1;
                d->sm_clock_mhz = nvml[k].sm_clock_mhz;
                d->mem_clock_mhz = nvml[k].mem_clock_mhz;
                key = (long long)k;   // nvidia-smi lists in NVML index order
                matched = true;
                break;
            }
        }
        if (!matched) {
            for (const identity::ProcGpu& g : proc) {
                if (g.uuid != uuid) continue;
                info.device_minor = atoi(g.minor.c_str());
                info.identity_source = 2;
                break;
            }
        }
        for (const identity::ProcGpu& g : proc) c->proc_lists_mine = c->proc_lists_mine || g.uuid == uuid;
        keyed.push_back({std::move(d), key});
    }
    std::stable_sort(keyed.begin(), keyed.end(), [](const Keyed& a, const Keyed& b) { return a.key < b.key; });

    for (size_t i = 0; i < keyed.size(); ++i) {
        Device* d = keyed[i].d.get();
        d->index = (int)i;
        d->sweep_bytes = opts.sweep_bytes;
        d->seed_dev = opts.seed_base | (uint64_t)(d->info.device_minor >= 0 ? d->info.device_minor : d->ordinal);
        d->seed_cur = d->seed_dev;
        phase("device properties");
        CU_TRY(c.get(), cudaSetDevice(d->ordinal));
        CU_TRY(c.get(), cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
        phase("primary context + stream");
        CU_TRY(c.get(), cudaStreamCreateWithFlags(&d->aux, cudaStreamNonBlocking));
        CU_TRY(c.get(), cudaEventCreate(&d->ev0));
        CU_TRY(c.get(), cudaEventCreate(&d->ev1));
        for (cudaEvent_t* ev : {&d->ev_fork, &d->ev_join, &d->ev_hbm_done, &d->ev_aux_done, &d->ev_chase_ready})
            CU_TRY(c.get(), cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
        CU_TRY(c.get(), plan_kernels(d->ordinal, &d->plan));
        phase("kernel plan (module load)");
        const int max_grid = std::max({d->plan.fill.grid, d->plan.read_ldg.grid, d->plan.read_ldg256.grid,
                                       d->plan.read_tma.grid, d->plan.copy_fused.grid, d->plan.expect.grid, 1});
        int rc = alloc_scratch(c.get(), &d->scratch, max_grid);
        if (rc) return rc;
        if ((rc = alloc_scratch(c.get(), &d->scratch_aux, max_grid))) return rc;
        if ((rc = alloc_scratch(c.get(), &d->scratch_pfx, max_grid))) return rc;
        for (int k = 0; k < 2; ++k) {
            Lane& L = d->lanes[k];
            const size_t slots = k == 0 ? (size_t)kSlotCount : 64;
            CU_TRY(c.get(), cudaMalloc(&L.d_out, sizeof(SweepOut) * slots));
            CU_TRY(c.get(), cudaMemset(L.d_out, 0xFF, sizeof(SweepOut) * slots));   // no slot starts with a plausible stamp
            CU_TRY(c.get(), cudaMallocHost(&L.h_out, sizeof(SweepOut) * slots));
            CU_TRY(c.get(), cudaMalloc(&L.d_params, sizeof(ProbeParams)));
            CU_TRY(c.get(), cudaMallocHost(&L.h_params, sizeof(ProbeParams)));
            CU_TRY(c.get(), cudaMalloc(&L.d_result, sizeof(cro_probe_result)));
            CU_TRY(c.get(), cudaMallocHost(&L.h_result, sizeof(cro_probe_result)));
            CU_TRY(c.get(), cudaMemset(L.d_result, 0, sizeof(cro_probe_result)));
            CU_TRY(c.get(), cudaEventCreateWithFlags(&L.ev_done, cudaEventDisableTiming));
        }
        CU_TRY(c.get(), cudaMalloc(&d->d_tmpl, sizeof(cro_probe_result)));
        CU_TRY(c.get(), cudaMalloc(&d->d_gather, sizeof(cro_probe_result) * CRO_MAX_DEVICES));
        CU_TRY(c.get(), cudaMallocHost(&d->h_gather, sizeof(cro_probe_result) * CRO_MAX_DEVICES));
        CU_TRY(c.get(), cudaMalloc(&d->d_chase_out, 2 * CRO_MAX_DEVICES * sizeof(unsigned long long)));
        CU_TRY(c.get(), cudaMallocHost(&d->h_chase_out, 2 * CRO_MAX_DEVICES * sizeof(unsigned long long)));
        phase("buffers (device + pinned)");
        if (!(opts.flags & CRO_F_LAZY_ALLOC)) {
            if ((rc = ensure_region(c.get(), d))) return rc;
            phase("sweep region");
        }
        refresh_ecc(c.get(), d);
        c->devs.push_back(std::move(keyed[i].d));
    }
    for (auto& d : c->devs) {
        CU_TRY(c.get(), cudaSetDevice(d->ordinal));
        int rc = stage_template(c.get(), d.get());
        if (rc) return rc;
    }
    phase("identity template");
    *out = c.release();
    return CRO_OK;
}

thread_local std::string g_init_error;
const std::string& last_init_error() { return g_init_error; }
void set_thread_error(const std::string& m) noexcept {
    try { g_init_error = m; } catch (...) {}
}

}  // namespace cro
cro_ctx::~cro_ctx() {
    if (inv_thread.joinable()) inv_thread.join();     // a background inventory refresh still reads this context
    if (!last_error.empty()) cro::g_init_error = last_error;
}
namespace cro {

Device::~Device() {
    if (ordinal < 0) return;                      // never bound to a CUDA device: owns nothing
    cudaSetDevice(ordinal);
    if (stream) cudaStreamSynchronize(stream);
    if (aux) cudaStreamSynchronize(aux);
    cudaFree(region);                             // cudaFree(nullptr) is a no-op
    free_scratch(&scratch);
    free_scratch(&scratch_aux);
    free_scratch(&scratch_pfx);
    for (Lane& L : lanes) {
        cudaFree(L.d_out);
        if (L.h_out) cudaFreeHost(L.h_out);
        cudaFree(L.d_params);
        if (L.h_params) cudaFreeHost(L.h_params);
        cudaFree(L.d_result);
        if (L.h_result) cudaFreeHost(L.h_result);
        if (L.graph_exec) cudaGraphExecDestroy(L.graph_exec);
        for (cudaEvent_t e : L.evpool) cudaEventDestroy(e);
        if (L.ev_done) cudaEventDestroy(L.ev_done);
    }
    cudaFree(d_tmpl);
    cudaFree(d_gather);
    if (h_gather) cudaFreeHost(h_gather);
    for (unsigned long long* t : d_chase_tables) cudaFree(t);
    cudaFree(d_chase_out);
    if (h_chase_out) cudaFreeHost(h_chase_out);
    for (cudaEvent_t e : ev_push_done) cudaEventDestroy(e);
    for (cudaEvent_t e : ev_reread_done) cudaEventDestroy(e);
    for (cudaEvent_t e : {ev0, ev1, ev_fork, ev_join, ev_hbm_done, ev_aux_done, ev_chase_ready})
        if (e) cudaEventDestroy(e);
    if (aux) cudaStreamDestroy(aux);
    if (stream) cudaStreamDestroy(stream);
    cudaGetLastError();                           // a failed release must not poison the caller's next CUDA call
}

void ctx_destroy(cro_ctx* c) {
    if (!c) return;
    if (c->nccl_ready && c->nccl_lib) {
        auto destroy = (int (*)(void*))dlsym(c->nccl_lib, "ncclCommDestroy");
        if (destroy)
            for (void* comm : c->nccl_comms)
                if (comm) destroy(comm);
    }
    delete c;                                     // ~Device releases the per-device CUDA objects
}

static void drain_pending(cro_ctx* c, Device* d);

static Device* dev_at(cro_ctx* c, int idx) {
    if (!c || idx < 0 || idx >= (int)c->devs.size()) return nullptr;
    return c->devs[(size_t)idx].get();
}

// ---------------------------------------------------------------------------
// single sweeps (tests, tuning, bench context): immediate seed, scratch slots
// ---------------------------------------------------------------------------
static void slot_to_result(const SweepOut& s, cro_sweep_result* out) {
    out->checksum_xor = s.x;
    out->checksum_sum = s.s;
    out->checksum_wsum = s.w;
    out->timer_ns = s.t1 - s.t0;
}

int ctx_fill(cro_ctx* c, int idx, uint32_t iters, cro_sweep_result* out) {
    Device* d = dev_at(c, idx);
    if (!d || !out || iters == 0) return CRO_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(d->mu);
    drain_pending(c, d);
    CU_TRY(c, cudaSetDevice(d->ordinal));
    int rc = ensure_region(c, d);
    if (rc) return rc;
    CU_TRY(c, cudaEventRecord(d->ev0, d->stream));
    for (uint32_t i = 0; i < iters; ++i)
        CU_TRY(c, launch_fill(d->plan, d->region, d->sweep_bytes, imm_params(d), d->scratch, &d->d_out[kSlotScratch], d->stream));
    CU_TRY(c, cudaEventRecord(d->ev1, d->stream));
    c->launches += iters;
    d->filled = true;
    CU_TRY(c, cudaMemcpyAsync(&d->h_out[kSlotScratch], &d->d_out[kSlotScratch], sizeof(SweepOut), cudaMemcpyDeviceToHost, d->stream));
    if ((rc = wait_stream(c, d))) return rc;
    float ms = 0;
    CU_TRY(c, cudaEventElapsedTime(&ms, d->ev0, d->ev1));
    memset(out, 0, sizeof *out);
    out->bytes = d->sweep_bytes * iters;
    out->ns = ms_to_ns(ms);
    out->timer_ns = d->h_out[kSlotScratch].t1 - d->h_out[kSlotScratch].t0;
    out->launches = iters;
    return CRO_OK;
}

int ctx_read(cro_ctx* c, int idx, uint32_t variant, uint32_t iters, bool dst_half,
             cro_sweep_result* out) {
    Device* d = dev_at(c, idx);
    if (!d || !out || iters == 0) return CRO_ERR_INVALID_ARG;
    variant = resolve_read_variant(variant, d->sweep_bytes);
    std::lock_guard<std::mutex> g(d->mu);
    drain_pending(c, d);
    CU_TRY(c, cudaSetDevice(d->ordinal));
    int rc = ensure_filled(c, d);
    if (rc) return rc;
    const unsigned char* base = d->region + (dst_half ? d->sweep_bytes : 0);
    CU_TRY(c, cudaEventRecord(d->ev0, d->stream));
    for (uint32_t i = 0; i < iters; ++i)
        CU_TRY(c, launch_read(d->plan, variant, base, d->sweep_bytes, imm_params(d), d->scratch, &d->d_out[kSlotScratch], d->stream));
    CU_TRY(c, cudaEventRecord(d->ev1, d->stream));
    c->launches += iters;
    CU_TRY(c, cudaMemcpyAsync(&d->h_out[kSlotScratch], &d->d_out[kSlotScratch], sizeof(SweepOut), cudaMemcpyDeviceToHost,
                              d->stream));
    if ((rc = wait_stream(c, d))) return rc;
    float ms = 0;
    CU_TRY(c, cudaEventElapsedTime(&ms, d->ev0, d->ev1));
    memset(out, 0, sizeof *out);
    out->bytes = d->sweep_bytes * iters;
    out->ns = ms_to_ns(ms);
    slot_to_result(d->h_out[kSlotScratch], out);
    out->variant = variant;
    out->launches = iters;
    return CRO_OK;
}

int ctx_copy(cro_ctx* c, int idx, uint32_t variant, uint32_t iters, cro_sweep_result* out) {
    Device* d = dev_at(c, idx);
    if (!d || !out || iters == 0) return CRO_ERR_INVALID_ARG;
    variant = resolve_copy_variant(variant);
    std::lock_guard<std::mutex> g(d->mu);
    drain_pending(c, d);
    CU_TRY(c, cudaSetDevice(d->ordinal));
    int rc = ensure_filled(c, d);
    if (rc) return rc;
    CU_TRY(c, cudaMemsetAsync(&d->d_out[kSlotScratch], 0, sizeof(SweepOut), d->stream));
    CU_TRY(c, cudaEventRecord(d->ev0, d->stream));
    for (uint32_t i = 0; i < iters; ++i)
        CU_TRY(c, launch_copy(d->plan, variant, d->region + d->sweep_bytes, d->region, d->sweep_bytes, imm_params(d),
                              d->scratch, &d->d_out[kSlotScratch], d->stream));
    CU_TRY(c, cudaEventRecord(d->ev1, d->stream));
    c->launches += iters;
    CU_TRY(c, cudaMemcpyAsync(&d->h_out[kSlotScratch], &d->d_out[kSlotScratch], sizeof(SweepOut), cudaMemcpyDeviceToHost,
                              d->stream));
    if ((rc = wait_stream(c, d))) return rc;
    float ms = 0;
    CU_TRY(c, cudaEventElapsedTime(&ms, d->ev0, d->ev1));
    memset(out, 0, sizeof *out);
    out->bytes = 2 * d->sweep_bytes * iters;
    out->ns = ms_to_ns(ms);
    if (variant == COPY_TMA_FUSED) slot_to_result(d->h_out[kSlotScratch], out);   // checksum of the source as read
    out->variant = variant;
    out->launches = iters;
    return CRO_OK;
}

int ctx_expected(cro_ctx* c, int idx, cro_sweep_result* out) {
    Device* d = dev_at(c, idx);
    if (!d || !out) return CRO_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(d->mu);
    drain_pending(c, d);
    CU_TRY(c, cudaSetDevice(d->ordinal));
    CU_TRY(c, cudaEventRecord(d->ev0, d->stream));
    CU_TRY(c, launch_expected(d->plan, d->sweep_bytes, imm_params(d), d->scratch, &d->d_out[kSlotScratch], d->stream));
    c->launches++;
    CU_TRY(c, cudaEventRecord(d->ev1, d->stream));
    CU_TRY(c, cudaMemcpyAsync(&d->h_out[kSlotScratch], &d->d_out[kSlotScratch], sizeof(SweepOut), cudaMemcpyDeviceToHost,
                              d->stream));
    CU_TRY(c, cudaStreamSynchronize(d->stream));
    float ms = 0;
    CU_TRY(c, cudaEventElapsedTime(&ms, d->ev0, d->ev1));
    memset(out, 0, sizeof *out);
    out->bytes = 0;
    out->ns = ms_to_ns(ms);
    slot_to_result(d->h_out[kSlotScratch], out);
    out->launches = 1;
    return CRO_OK;
}

int ctx_inject(cro_ctx* c, int idx, uint64_t word, uint64_t mask) {
    Device* d = dev_at(c, idx);
    if (!d) return CRO_ERR_INVALID_ARG;
    if (word >= 2 * (d->sweep_bytes / 8)) return CRO_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(d->mu);
    drain_pending(c, d);
    CU_TRY(c, cudaSetDevice(d->ordinal));
    int rc = ensure_filled(c, d);
    if (rc) return rc;
    CU_TRY(c, launch_xor_word(d->region, word, mask, d->stream));
    c->launches++;
    CU_TRY(c, cudaStreamSynchronize(d->stream));
    return CRO_OK;
}

int ctx_read_words(cro_ctx* c, int idx, uint64_t first, uint64_t n, uint64_t* out) {
    Device* d = dev_at(c, idx);
    if (!d || !out) return CRO_ERR_INVALID_ARG;
    const uint64_t limit = 2 * (d->sweep_bytes / 8);
    if (n > limit || first > limit - n) return CRO_ERR_INVALID_ARG;    // no wrap: first + n may not overflow
    if (n == 0) return CRO_OK;
    std::lock_guard<std::mutex> g(d->mu);
    drain_pending(c, d);
    CU_TRY(c, cudaSetDevice(d->ordinal));
    int rc = ensure_filled(c, d);
    if (rc) return rc;
    CU_TRY(c, cudaMemcpyAsync(out, d->region + first * 8, n * 8, cudaMemcpyDeviceToHost, d->stream));
    CU_TRY(c, cudaStreamSynchronize(d->stream));
    return CRO_OK;
}

// ---------------------------------------------------------------------------
// full per-device probe
// ---------------------------------------------------------------------------
// Which half (0 = A, 1 = B) a sweep touches.  Copies run ping-pong — A->B, B->A, ... — so the checksum
// copy k+1 folds out of its source is the verification of what copy k wrote; the first read sweep reads the
// last copy's destination and the reads alternate from there.
static int copy_src_half(uint32_t k) { return (int)(k & 1u); }
static int read_half(uint32_t copies, uint32_t k) {
    if (copies == 0) return 0;
    const int last_dst = (int)(copies & 1u);           // C odd: B, C even: A
    return (k & 1u) ? 1 - last_dst : last_dst;
}

// Caller holds d->mu.  Enqueues one whole probe on the device's stream, using lane L's buffers, and returns without
// waiting: params refresh, fill, copy sweeps, read sweeps, the closed-form generator on the side stream, the finalize
// kernel that writes the result struct, and the copy-back of that struct.
static int probe_enqueue(cro_ctx* c, Device* d, Lane& L) {
    const cro_opts& o = c->opts;
    Range nv(c, "cro.probe.enqueue");
    CU_TRY(c, cudaSetDevice(d->ordinal));
    int rc = ensure_region(c, d);
    if (rc) return rc;
    const uint32_t rv = resolve_read_variant(o.read_variant, d->sweep_bytes);
    const uint32_t cv = resolve_copy_variant(o.copy_variant);
    const uint32_t R = o.read_sweeps;
    const uint32_t C = (o.flags & CRO_F_SKIP_COPY) ? 0 : o.copy_sweeps;
    if (d->tmpl.sweep_bytes != d->sweep_bytes) {      // ensure_region degraded S
        if ((rc = stage_template(c, d))) return rc;
    }

    // events: one before the fill, one after every sweep (pool lives with the lane)
    const size_t need = 2 + R + C;
    while (L.evpool.size() < need) {
        cudaEvent_t e;
        CU_TRY(c, cudaEventCreate(&e));
        L.evpool.push_back(e);
    }
    std::vector<cudaEvent_t>& ev = L.evpool;
    const bool overlap = env::get("CRO_EXPECT_OVERLAP") != 0;
    unsigned char* half[2] = {d->region, d->region + d->sweep_bytes};
    const Params gp = graph_params(L);

    size_t k = 0;
    // The whole probe as one sequence; `external` records the timing events as external event-record
    // nodes so that the same sequence can be stream-captured into a CUDA graph once and replayed.
    auto issue = [&](bool external) -> int {
        const unsigned flag = external ? cudaEventRecordExternal : cudaEventRecordDefault;
        k = 0;
        CU_TRY(c, cudaMemcpyAsync(L.d_params, L.h_params, sizeof(ProbeParams), cudaMemcpyHostToDevice, d->stream));
        CU_TRY(c, cudaEventRecordWithFlags(ev[k++], d->stream, flag));
        uint32_t sweep_no = 0;
        auto maybe_inject = [&]() -> int {      // CRO_F_TEST_INJECT: corrupt one word behind a chosen sweep
            if ((o.flags & CRO_F_TEST_INJECT) && o.test_inject_after == sweep_no && o.test_inject_word < 2 * (d->sweep_bytes / 8))
                CU_TRY(c, launch_xor_word(d->region, o.test_inject_word, o.test_inject_mask, d->stream));
            ++sweep_no;
            return CRO_OK;
        };
        CU_TRY(c, launch_fill(d->plan, half[0], d->sweep_bytes, gp, d->scratch, &L.d_out[kSlotFill], d->stream));
        CU_TRY(c, cudaEventRecordWithFlags(ev[k++], d->stream, flag));
        if (maybe_inject()) return CRO_ERR_CUDA;
        // the closed form: ALU only, so it runs beside the copy sweeps (which leave the ALUs idle)
        cudaStream_t es = overlap ? d->aux : d->stream;
        if (overlap) {
            CU_TRY(c, cudaEventRecord(d->ev_fork, d->stream));
            CU_TRY(c, cudaStreamWaitEvent(d->aux, d->ev_fork, 0));
        }
        CU_TRY(c, launch_expected(d->plan, d->sweep_bytes, gp, d->scratch_aux, &L.d_out[kSlotExpect], es));
        if (overlap) CU_TRY(c, cudaEventRecord(d->ev_join, d->aux));
        for (uint32_t i = 0; i < C; ++i) {
            const int s = copy_src_half(i);
            CU_TRY(c, launch_copy(d->plan, cv, half[1 - s], half[s], d->sweep_bytes, gp, d->scratch,
                                  &L.d_out[kSlotSweep0 + i], d->stream));
            CU_TRY(c, cudaEventRecordWithFlags(ev[k++], d->stream, flag));
            if (maybe_inject()) return CRO_ERR_CUDA;
        }
        for (uint32_t i = 0; i < R; ++i) {
            CU_TRY(c, launch_read(d->plan, rv, half[read_half(C, i)], d->sweep_bytes, gp, d->scratch,
                                  &L.d_out[kSlotSweep0 + C + i], d->stream));
            CU_TRY(c, cudaEventRecordWithFlags(ev[k++], d->stream, flag));
            if (maybe_inject()) return CRO_ERR_CUDA;
        }
        if (overlap) CU_TRY(c, cudaStreamWaitEvent(d->stream, d->ev_join, 0));
        FinalizeArgs fa{};
        fa.tmpl = d->d_tmpl;
        fa.out = L.d_result;
        fa.slots = L.d_out;
        fa.pp = L.d_params;
        fa.sweep_bytes = d->sweep_bytes;
        fa.read_sweeps = R;
        fa.copy_sweeps = C;
        fa.read_variant = rv;
        fa.copy_variant = C ? cv : 0;
        fa.fused = (cv == COPY_TMA_FUSED) ? 1u : 0u;
        CU_TRY(c, launch_finalize(fa, d->stream));
        CU_TRY(c, cudaMemcpyAsync(L.h_result, L.d_result, sizeof(cro_probe_result), cudaMemcpyDeviceToHost, d->stream));
        CU_TRY(c, cudaMemcpyAsync(L.h_out, L.d_out, sizeof(SweepOut) * 64, cudaMemcpyDeviceToHost, d->stream));
        return CRO_OK;
    };

    // this probe's seed: the host refreshes the 16 bytes the graph's first node copies to the device
    const uint64_t nonce = d->nonce_next++;
    L.h_params->seed = seed_of(d, nonce);
    L.h_params->nonce = nonce;
    d->seed_cur = L.h_params->seed;
    d->nonce_cur = nonce;

    // One graph launch instead of ~40 runtime calls per probe (matters when one host thread feeds 8 GPUs).
    // The graph is tied to the options it was captured with; any capture problem falls back to direct launches.
    const uint64_t graph_key = ((uint64_t)rv << 48) ^ ((uint64_t)cv << 40) ^ ((uint64_t)R << 24) ^ ((uint64_t)C << 8) ^
                               (overlap ? 1u : 0u) ^ (d->sweep_bytes << 1) ^
                               ((o.flags & CRO_F_TEST_INJECT) ? ((uint64_t)o.test_inject_after << 56) ^ (o.test_inject_word * 0x9E3779B97F4A7C15ull) ^ o.test_inject_mask : 0);
    if (env::get("CRO_USE_GRAPH") && !L.graph_failed) {
        if (L.graph_exec && L.graph_key != graph_key) {
            cudaGraphExecDestroy(L.graph_exec);
            L.graph_exec = nullptr;
        }
        if (!L.graph_exec) {
            Range nvc(c, "cro.probe.capture");
            // a probe still running on the stream does not matter: capture records, it does not execute — and it must
            // not wait either (one host thread feeds eight GPUs: a 10 ms wait here starves the other seven)
            cudaGraph_t graph = nullptr;
            bool ok = cudaStreamBeginCapture(d->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
            if (ok) {
                const int irc = issue(true);
                const cudaError_t ec = cudaStreamEndCapture(d->stream, &graph);
                ok = irc == CRO_OK && ec == cudaSuccess && graph != nullptr;
            }
            if (ok) ok = cudaGraphInstantiate(&L.graph_exec, graph, 0) == cudaSuccess;
            if (graph) cudaGraphDestroy(graph);
            if (!ok) {
                cudaGetLastError();
                L.graph_exec = nullptr;
                L.graph_failed = true;
            } else {
                L.graph_key = graph_key;
                L.graph_events = k;
            }
        }
    }
    if (L.graph_exec) {
        CU_TRY(c, cudaGraphLaunch(L.graph_exec, d->stream));
        k = L.graph_events;
    } else {
        int irc = issue(false);
        if (irc) return irc;
    }
    CU_TRY(c, cudaEventRecord(L.ev_done, d->stream));
    d->filled = true;
    c->launches += 3 + R + C;       // fill + closed form + sweeps + finalize
    L.events = k;
    L.reads = R;
    L.copies = C;
    L.timed = true;
    L.in_flight = true;
    L.since = std::chrono::steady_clock::now();
    return CRO_OK;
}

static std::string describe_failure(const Device* d, const cro_probe_result& r) {
    const std::string who = std::string(d->info.gpu_uuid, strnlen(d->info.gpu_uuid, sizeof d->info.gpu_uuid));
    const std::string idx = std::to_string((unsigned)r.fail_index);
    switch (r.fail_code) {
        case CRO_FAIL_EXPECT: return "closed-form checksum slot on " + who + " is stale: the generator kernel did not run";
        case CRO_FAIL_COPY_SRC:
            return "HBM copy sweep " + idx + " on " + who + " read something else than the pattern" +
                   (r.fail_index ? " (the destination of sweep " + std::to_string((unsigned)r.fail_index - 1) + " is corrupt)" : " (the fill is corrupt)");
        case CRO_FAIL_READ: return "HBM read sweep " + idx + " on " + who + " does not reproduce the pattern checksum";
        case CRO_FAIL_P2P_READ: return "NVLink read of peer " + idx + " from " + who + " does not reproduce the pattern checksum";
        case CRO_FAIL_P2P_PUSH: return "NVLink push between " + who + " and peer " + idx + " did not land the pattern checksum";
        case CRO_FAIL_P2P_CHASE: return "NVLink pointer chase from " + who + " through peer " + idx + " ended on the wrong slot";
        case CRO_FAIL_STALE: return "sweep slot " + idx + " on " + who + " carries another probe's stamp: a kernel of the probe did not run";
        default: return "probe of " + who + " failed";
    }
}

// Waits for a lane's probe, honouring opts.deadline_ms (see wait_stream).
static int wait_lane(cro_ctx* c, Lane& L) {
    if (c->opts.deadline_ms <= 0) {
        CU_TRY(c, cudaEventSynchronize(L.ev_done));
        return CRO_OK;
    }
    const auto until = std::chrono::steady_clock::now() + std::chrono::milliseconds(c->opts.deadline_ms);
    for (;;) {
        cudaError_t q = cudaEventQuery(L.ev_done);
        if (q == cudaSuccess) return CRO_OK;
        if (q != cudaErrorNotReady) {
            c->set_error(std::string("cudaEventQuery: ") + cudaGetErrorString(q));
            return CRO_ERR_CUDA;
        }
        if (std::chrono::steady_clock::now() > until) {
            c->set_error("probe deadline of " + std::to_string(c->opts.deadline_ms) + " ms exceeded");
            return CRO_ERR_DEADLINE;
        }
        std::this_thread::sleep_for(std::chrono::microseconds(50));
    }
}

// Caller holds d->mu.  Waits for the probe enqueued on lane L and hands out the struct the device wrote.
static int probe_finish(cro_ctx* c, Device* d, Lane& L, cro_probe_result* r) {
    CU_TRY(c, cudaSetDevice(d->ordinal));
    int rc = wait_lane(c, L);
    L.in_flight = false;
    d->last_lane = (int)(&L - d->lanes);
    if (rc) {
        memset(r, 0, sizeof *r);
        r->abi_version = CRO_ABI_VERSION;
        r->status = rc;
        return rc;
    }
    *r = *L.h_result;
    d->last = *r;
    d->have_last = true;
    c->m_probes++;
    if (r->status != CRO_OK) {
        c->m_probe_failures++;
        c->set_error(describe_failure(d, *r));
        // What the memory itself reported: uncorrected volatile ECC errors (nvmlDeviceGetTotalEccErrors).
        // NVML calls serialise across processes (measured: ~2 ms each with 4 ranks probing, enough to skew the
        // ranks' all-gather), so the warm probe reuses the count read at init / at the last full-box probe and
        // only a FAILED probe pays for a fresh read — which then also goes into the device-resident copies.
        const uint32_t before = d->ecc_uncorrected;
        refresh_ecc(c, d);
        if (d->ecc_uncorrected != before) {
            r->ecc_errors = d->ecc_uncorrected;
            d->tmpl.ecc_errors = d->ecc_uncorrected;
            *L.h_result = *r;
            CU_TRY(c, cudaMemcpyAsync(L.d_result, L.h_result, sizeof *r, cudaMemcpyHostToDevice, d->stream));
            CU_TRY(c, cudaMemcpyAsync(d->d_tmpl, &d->tmpl, sizeof d->tmpl, cudaMemcpyHostToDevice, d->stream));
            CU_TRY(c, cudaStreamSynchronize(d->stream));
        }
    }
    return r->status;
}

// Drains every probe still in flight on the device (oldest first) into d->done, so another operation may use the
// stream / the region.  Caller holds d->mu.
static void drain_pending(cro_ctx* c, Device* d) {
    while (d->lane_count > 0) {
        Lane& L = d->lanes[d->lane_head];
        Device::Collected col;
        col.rc = probe_finish(c, d, L, &col.r);
        col.at = std::chrono::steady_clock::now();
        d->done.push_back(col);
        d->lane_head ^= 1;
        --d->lane_count;
    }
}

int ctx_probe_device(cro_ctx* c, int idx, cro_probe_result* out) {
    Device* d = dev_at(c, idx);
    if (!d || !out) return CRO_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(d->mu);
    drain_pending(c, d);
    d->done.clear();                  // a synchronous probe supersedes uncollected asynchronous ones
    d->lane_head = 0;
    Lane& L = d->lanes[0];            // always lane 0: its result buffer is the all-gather send buffer
    int rc = probe_enqueue(c, d, L);
    if (rc) {
        memset(out, 0, sizeof *out);
        out->abi_version = CRO_ABI_VERSION;
        out->status = rc;
        return rc;
    }
    return probe_finish(c, d, L, out);
}

// Asynchronous form: begin enqueues a probe and returns; end waits for the OLDEST one and evaluates it.  Up to two
// probes per device may be in flight — the second one's kernels are already queued behind the first's, so the GPU
// does not idle while the host collects one result and starts the next.  Lets ONE host thread (the reference's single
// reconcile worker) keep every attached GPU busy.
int ctx_probe_begin(cro_ctx* c, int idx) {
    Device* d = dev_at(c, idx);
    if (!d) return CRO_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(d->mu);
    if (d->lane_count + (int)d->done.size() >= 2) return CRO_OK;   // two in flight (or waiting to be collected): no-op
    Lane& L = d->lanes[(d->lane_head + d->lane_count) & 1];
    if (L.in_flight) return CRO_OK;
    int rc = probe_enqueue(c, d, L);
    if (rc) return rc;
    ++d->lane_count;
    return CRO_OK;
}

// 1 when the oldest probe begun on this device has finished (or none is in flight), 0 while it runs.
int ctx_probe_poll(cro_ctx* c, int idx) {
    Device* d = dev_at(c, idx);
    if (!d) return 1;
    std::lock_guard<std::mutex> g(d->mu);
    if (!d->done.empty() || d->lane_count == 0) return 1;
    cudaSetDevice(d->ordinal);
    // anything but "still running" counts as finished: a failed stream must not keep a poller spinning —
    // cro_probe_end then reports the CUDA error
    return cudaEventQuery(d->lanes[d->lane_head].ev_done) == cudaErrorNotReady ? 0 : 1;
}

// Probes in flight or finished-but-uncollected on this device (0..2).
int ctx_probe_depth(cro_ctx* c, int idx) {
    Device* d = dev_at(c, idx);
    if (!d) return 0;
    std::lock_guard<std::mutex> g(d->mu);
    return d->lane_count + (int)d->done.size();
}

// Blocks until the oldest probe in flight on this device (if any) has finished; does not collect it.
int ctx_probe_wait(cro_ctx* c, int idx) {
    Device* d = dev_at(c, idx);
    if (!d) return CRO_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(d->mu);
    if (!d->done.empty() || d->lane_count == 0) return CRO_OK;
    CU_TRY(c, cudaSetDevice(d->ordinal));
    CU_TRY(c, cudaEventSynchronize(d->lanes[d->lane_head].ev_done));
    return CRO_OK;
}

int ctx_probe_end(cro_ctx* c, int idx, cro_probe_result* out) {
    Device* d = dev_at(c, idx);
    if (!d || !out) return CRO_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(d->mu);
    // a drained result nobody collected for more than a second says nothing about the device NOW
    while (!d->done.empty() && std::chrono::steady_clock::now() - d->done.front().at > std::chrono::seconds(1)) d->done.pop_front();
    if (d->done.empty()) {
        if (d->lane_count == 0) {      // nothing begun: behave like the synchronous call
            Lane& L0 = d->lanes[d->lane_head];
            int rc = probe_enqueue(c, d, L0);
            if (rc) return rc;
            ++d->lane_count;
        }
        Lane& L = d->lanes[d->lane_head];
        const int rc = probe_finish(c, d, L, out);
        d->lane_head ^= 1;
        --d->lane_count;
        return rc;
    }
    *out = d->done.front().r;
    const int rc = d->done.front().rc;
    d->done.pop_front();
    return rc;
}

// Prometheus text exposition of what the context has seen (SURVEY.md §5: the operator registers collectors with the
// controller-runtime metrics registry, cmd/main.go:66,119-125; a Go collector forwards these lines).
std::string ctx_metrics_text(cro_ctx* c) {
    std::string o;
    auto counter = [&](const char* name, const char* help, uint64_t v) {
        o += std::string("# HELP ") + name + " " + help + "\n# TYPE " + name + " counter\n" + name + " " + std::to_string(v) + "\n";
    };
    counter("cro_probe_total", "HBM probes collected by this context.", c->m_probes.load());
    counter("cro_probe_failures_total", "Probes whose device-side verdict was not ok.", c->m_probe_failures.load());
    counter("cro_fullbox_probe_total", "cro_probe_all calls (concurrent probes + NVLink rounds + all-gather).", c->m_fullbox.load());
    counter("cro_helper_probe_total", "Probes of devices attached after cuInit, run through the helper process.", c->m_helper_probes.load());
    counter("cro_helper_probe_failures_total", "Helper-process probes that failed or timed out.", c->m_helper_failures.load());
    counter("cro_inventory_rescans_total", "Times the node inventory was rebuilt from the driver registry.", c->inv_rescans.load());
    counter("cro_kernel_launches_total", "CUDA kernels launched by this context.", c->launches.load());
    struct G { const char* name; const char* help; };
    const G gauges[] = {{"cro_probe_status", "Status of the device's last probe (0 ok, <0 a CRO_ERR_* code)."},
                        {"cro_probe_hbm_read_bytes_per_second", "Best read sweep of the last probe."},
                        {"cro_probe_hbm_copy_bytes_per_second", "Best copy sweep of the last probe (read + written bytes)."},
                        {"cro_probe_hbm_fill_bytes_per_second", "Fill sweep of the last probe."},
                        {"cro_probe_copies_verified", "Copy sweeps of the last probe whose destination was re-read and matched."},
                        {"cro_probe_ecc_uncorrected", "Uncorrected volatile ECC errors as last read from NVML."},
                        {"cro_probe_nonce", "Probes run on the device by this context."}};
    for (const G& g : gauges) {
        o += std::string("# HELP ") + g.name + " " + g.help + "\n# TYPE " + g.name + " gauge\n";
        for (auto& dp : c->devs) {
            Device* d = dp.get();
            std::lock_guard<std::mutex> lk(d->mu);
            if (!d->have_last) continue;
            const cro_probe_result& r = d->last;
            const std::string uuid(r.gpu_uuid, strnlen(r.gpu_uuid, sizeof r.gpu_uuid));
            auto rate = [](uint64_t bytes, uint64_t ns) -> long long { return ns ? (long long)((unsigned __int128)bytes * 1000000000ull / ns) : 0; };
            long long v = 0;
            const std::string n = g.name;
            if (n == "cro_probe_status") v = r.status;
            else if (n == "cro_probe_hbm_read_bytes_per_second") v = rate(r.sweep_bytes, r.read_best_ns);
            else if (n == "cro_probe_hbm_copy_bytes_per_second") v = rate(2 * r.sweep_bytes, r.copy_best_ns);
            else if (n == "cro_probe_hbm_fill_bytes_per_second") v = rate(r.sweep_bytes, r.fill_ns);
            else if (n == "cro_probe_copies_verified") v = r.copy_verified;
            else if (n == "cro_probe_ecc_uncorrected") v = r.ecc_errors;
            else v = r.nonce;
            o += n + "{gpu_uuid=\"" + uuid + "\",minor=\"" + std::to_string(r.device_minor) + "\"} " + std::to_string(v) + "\n";
        }
    }
    return o;
}

// CUDA-event and %globaltimer times of the sweeps of the device's last collected probe.
int ctx_sweep_times(cro_ctx* c, int idx, cro_sweep_time* out, int cap, int* n_out) {
    Device* d = dev_at(c, idx);
    if (!d || !n_out) return CRO_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(d->mu);
    drain_pending(c, d);
    Lane& L = d->lanes[d->last_lane];
    const int n = L.timed ? (int)(1 + L.copies + L.reads) : 0;
    *n_out = n;
    if (n == 0) return CRO_OK;
    if (!out || cap < n) return CRO_ERR_BUFFER_SMALL;
    CU_TRY(c, cudaSetDevice(d->ordinal));
    for (int i = 0; i < n; ++i) {
        float ms = 0;
        CU_TRY(c, cudaEventElapsedTime(&ms, L.evpool[(size_t)i], L.evpool[(size_t)i + 1]));
        cro_sweep_time& t = out[i];
        memset(&t, 0, sizeof t);
        const SweepOut& s = L.h_out[i == 0 ? kSlotFill : kSlotSweep0 + i - 1];
        t.kind = i == 0 ? 0u : (i <= (int)L.copies ? 1u : 2u);
        t.index = i == 0 ? 0u : (t.kind == 1 ? (uint32_t)(i - 1) : (uint32_t)(i - 1 - (int)L.copies));
        t.bytes = t.kind == 1 ? 2 * d->sweep_bytes : d->sweep_bytes;
        t.event_ns = ms_to_ns(ms);
        t.timer_ns = s.t1 - s.t0;
    }
    return CRO_OK;
}

// ---------------------------------------------------------------------------
// the node's inventory, fresh on every query (inventory.hpp)
// ---------------------------------------------------------------------------
// The slow part of an inventory refresh: reads the registry's `information` files (each read goes through the
// driver) and, when the node holds other devices than this context, re-initialises NVML for nvidia-smi's ordering.
// Touches nothing of the context but its options, so it can run on a side thread.
static std::vector<cro_dev_info> build_inventory(const cro_ctx* c, const std::vector<cro_dev_info>& mine, bool have_proc,
                                                 bool* scanned_nvml) {
    const bool nvml_ok = !(c->opts.flags & CRO_F_NO_NVML);
    std::vector<identity::ProcGpu> proc;
    if (have_proc) proc = identity::ScanProc(c->proc_root);
    std::vector<inventory::Seen> seen;
    bool have_scan = have_proc;
    if (have_proc) {
        seen = inventory::FromProc(proc);
        // the common case — the node holds exactly the devices this context manages — needs nothing more
        bool same = seen.size() == mine.size();
        for (const auto& s : seen) {
            bool found = false;
            for (const auto& m : mine) found = found || s.uuid == std::string(m.gpu_uuid, strnlen(m.gpu_uuid, sizeof m.gpu_uuid));
            same = same && found;
        }
        if (same) have_scan = false;          // Merge then keeps the context's own (nvidia-smi) order
    }
    if (have_scan || !have_proc) {
        std::vector<identity::NvmlGpu> nv;
        if (nvml_ok && identity::ScanNvml(&nv, nullptr)) {   // init + shutdown: NVML sees hot-plugged devices only after a re-init
            *scanned_nvml = true;
            std::vector<inventory::Seen> ordered;
            for (const auto& g2 : nv) {                        // nvidia-smi lists in NVML index order
                bool on_node = !have_proc;
                for (const auto& s : seen) on_node = on_node || s.uuid == g2.uuid;
                if (!on_node) continue;
                inventory::Seen s;
                s.uuid = g2.uuid; s.bus_id = g2.bus_id; s.minor = g2.minor; s.source = 1;
                ordered.push_back(s);
            }
            for (const auto& s : seen) {                       // on the bus but not (yet) known to NVML: keep, at the end
                bool in = false;
                for (const auto& o2 : ordered) in = in || o2.uuid == s.uuid;
                if (!in) ordered.push_back(s);
            }
            seen = ordered;
            have_scan = true;
        }
    }
    return inventory::Merge(mine, have_scan, seen);
}

int ctx_inventory(cro_ctx* c, std::vector<cro_dev_info>* out, bool force) {
    if (!c || !out) return CRO_ERR_INVALID_ARG;
    std::vector<cro_dev_info> mine;
    for (auto& d : c->devs) mine.push_back(d->info);
    std::unique_lock<std::mutex> g(c->inv_mu);
    const bool nvml_ok = !(c->opts.flags & CRO_F_NO_NVML);
    // Every call looks at the node: the registry's directory listing (readdir + stat, ~10 us, no driver lock).  The
    // `information` files are read again
    //   * at once, when that listing differs from the last one or the caller insists (it was told about a UUID the
    //     list lacks);
    //   * in the BACKGROUND every 30 s — the reference's own requeue period (composableresource_controller.go:223,285)
    //     — because each such read goes through the driver's locks (100+ ms for a full box while nvidia-smi polls) and
    //     a reconcile must not pay for a refresh that will almost always confirm what is known.
    // A registry that listed none of the devices CUDA had just opened describes some other view of the node (a container
    // may mount it empty): it is not consulted, and the inventory goes by NVML as on a host without one.
    std::string key = c->proc_lists_mine ? identity::ProcRegistryListing(c->proc_root) : std::string();
    const bool have_proc = !key.empty();
    if (!have_proc) key = "-";
    const auto now = std::chrono::steady_clock::now();
    const bool nvml_due = !have_proc && nvml_ok && now - c->inv_nvml_at > std::chrono::seconds(1);
    if (c->inv_valid && key == c->inv_key && !nvml_due && !force) {
        if (have_proc && now - c->inv_full_at > std::chrono::seconds(30) && !c->inv_refreshing) {
            c->inv_refreshing = true;
            c->inv_full_at = now;
            c->inv_rescans++;
            if (c->inv_thread.joinable()) c->inv_thread.join();     // the previous refresh ended long ago
            c->inv_thread = std::thread([c, mine, key]() {
                bool nv = false;
                std::vector<cro_dev_info> fresh;
                try { fresh = build_inventory(c, mine, true, &nv); } catch (...) { fresh.clear(); nv = false; }
                std::lock_guard<std::mutex> lk(c->inv_mu);
                if (c->inv_key == key && (!fresh.empty() || c->inv.empty())) c->inv = fresh;   // a newer listing wins
                if (nv) c->inv_nvml_at = std::chrono::steady_clock::now();
                c->inv_refreshing = false;
            });
        }
        *out = c->inv;
        return CRO_OK;
    }
    c->inv_rescans++;
    c->inv_full_at = now;
    bool nv = false;
    c->inv = build_inventory(c, mine, have_proc, &nv);
    if (nv) c->inv_nvml_at = now;
    c->inv_key = key;
    c->inv_valid = true;
    *out = c->inv;
    return CRO_OK;
}

int ctx_probe_uuid(cro_ctx* c, const char* uuid, cro_probe_result* out) {
    if (!uuid || !out) return CRO_ERR_INVALID_ARG;
    const std::string want = uuid;
    uint64_t sweep = 1ull << 30;              // helper default: 1 GiB already sweeps at ~7 TB/s and starts ~4x sooner
    if (!c) env::reload(nullptr);            // no context ever validated the environment for this caller
    int deadline = (int)env::get("CRO_HELPER_TIMEOUT_MS");
    if (c) {
        std::vector<cro_dev_info> inv;
        int rc = ctx_inventory(c, &inv);
        if (rc) return rc;
        const cro_dev_info* hit = nullptr;
        for (int attempt = 0; attempt < 2 && !hit; ++attempt) {
            // told about a UUID the cached list lacks: look again, properly, before saying "not on this node"
            if (attempt == 1 && (rc = ctx_inventory(c, &inv, true))) return rc;
            for (const auto& d : inv)
                if (want == std::string(d.gpu_uuid, strnlen(d.gpu_uuid, sizeof d.gpu_uuid))) hit = &d;
        }
        if (!hit) {
            c->set_error("device '" + want + "' is not on this node");
            return CRO_ERR_NO_DEVICE;
        }
        if (hit->flags & CRO_DEV_IN_PROCESS) return ctx_probe_device(c, hit->dev_index, out);
        sweep = std::min<uint64_t>(c->opts.sweep_bytes, sweep);
        if (c->opts.deadline_ms > 0) deadline = c->opts.deadline_ms;
    }
    std::string err;
    if (c && c->nvtx) nvtxRangePushA("cro.probe.helper");
    const int rc = inventory::RunHelper("", want, sweep, deadline, out, &err);
    if (c && c->nvtx) nvtxRangePop();
    if (c) {
        c->m_helper_probes++;
        if (rc != CRO_OK) c->m_helper_failures++;
    }
    if (rc != CRO_OK && !err.empty()) {
        if (c) c->set_error(err);
        else set_thread_error(err);
    }
    return rc;
}

// ---------------------------------------------------------------------------
// multi-device: concurrent probes, NVLink rounds, one all-gather
// ---------------------------------------------------------------------------
namespace {

// Round-robin 1-factorisation of K_n (n even): n-1 rounds of n/2 disjoint pairs.
std::vector<std::vector<std::pair<int, int>>> one_factorisation(int n) {
    std::vector<std::vector<std::pair<int, int>>> rounds;
    if (n < 2) return rounds;
    const int m = (n % 2 == 0) ? n : n + 1;  // odd n: vertex m-1 is a bye
    for (int r = 0; r < m - 1; ++r) {
        std::vector<std::pair<int, int>> pairs;
        auto add = [&](int a, int b) { if (a < n && b < n) pairs.push_back({a, b}); };
        add(m - 1, r);
        for (int k = 1; k < m / 2; ++k) add((r + k) % (m - 1), (r - k + (m - 1)) % (m - 1));
        rounds.push_back(pairs);
    }
    return rounds;
}

int enable_peers(cro_ctx* c) {
    if (c->peers_enabled) return CRO_OK;
    const int n = (int)c->devs.size();
    for (int a = 0; a < n; ++a) {
        CU_TRY(c, cudaSetDevice(c->devs[a]->ordinal));
        for (int b = 0; b < n; ++b) {
            if (a == b) continue;
            int can = 0;
            CU_TRY(c, cudaDeviceCanAccessPeer(&can, c->devs[a]->ordinal, c->devs[b]->ordinal));
            if (!can) continue;
            cudaError_t e = cudaDeviceEnablePeerAccess(c->devs[b]->ordinal, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
                c->set_error(std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
                cudaGetLastError();
                return CRO_ERR_P2P;
            }
            cudaGetLastError();
        }
    }
    c->peers_enabled = true;
    for (int a = 0; a < n; ++a) {     // p2p_access goes into every device's identity template
        CU_TRY(c, cudaSetDevice(c->devs[a]->ordinal));
        int rc = stage_template(c, c->devs[(size_t)a].get());
        if (rc) return rc;
    }
    return CRO_OK;
}

// Latency permutations: device b holds, for every other device a, the Sattolo cycle a will chase through b's
// memory (slot i lives at table[i*16], one per 128-byte line), and a remembers where `hops` steps must end.
int ensure_chase(cro_ctx* c, uint32_t hops) {
    const int n = (int)c->devs.size();
    bool built = true;
    for (auto& d : c->devs) built = built && (int)d->d_chase_tables.size() == n && d->chase_hops_built == hops;
    if (built) return CRO_OK;
    Range nv(c, "cro.chase.build");
    std::vector<uint32_t> perm;
    std::vector<unsigned long long> wide(kChaseSlots);
    for (int b = 0; b < n; ++b) {
        Device* owner = c->devs[(size_t)b].get();
        CU_TRY(c, cudaSetDevice(owner->ordinal));
        if ((int)owner->d_chase_tables.size() != n) owner->d_chase_tables.assign((size_t)n, nullptr);
        for (int a = 0; a < n; ++a) {
            if (a == b) continue;
            Device* chaser = c->devs[(size_t)a].get();
            const int ma = chaser->info.device_minor >= 0 ? chaser->info.device_minor : chaser->ordinal;
            const int mb = owner->info.device_minor >= 0 ? owner->info.device_minor : owner->ordinal;
            chase_permutation(ma, mb, &perm);
            if (!owner->d_chase_tables[(size_t)a]) {
                CU_TRY(c, cudaMalloc(&owner->d_chase_tables[(size_t)a], (size_t)kChaseSlots * 128));
                CU_TRY(c, cudaMemset(owner->d_chase_tables[(size_t)a], 0, (size_t)kChaseSlots * 128));
                for (uint32_t i = 0; i < kChaseSlots; ++i) wide[i] = perm[i];
                // scatter: 8 bytes into the head of every 128-byte line
                CU_TRY(c, cudaMemcpy2D(owner->d_chase_tables[(size_t)a], 128, wide.data(), 8, 8, kChaseSlots, cudaMemcpyHostToDevice));
            }
            if ((int)chaser->chase_expect.size() != n) chaser->chase_expect.assign((size_t)n, 0u);
            uint32_t at = 0;
            for (uint32_t h = 0; h < hops; ++h) at = perm[at];
            chaser->chase_expect[(size_t)b] = at;
        }
    }
    for (auto& d : c->devs) d->chase_hops_built = hops;
    return CRO_OK;
}

int load_nccl(cro_ctx* c) {
    if (c->ncclAllGather) return CRO_OK;
    if (!c->nccl_lib) {
        const char* path = getenv("CRO_NCCL_PATH");
        if (path && strcmp(path, "off") == 0) {          // the host does not want NCCL in its process
            c->set_error("NCCL switched off (CRO_NCCL_PATH=off): host-side gather");
            return CRO_ERR_NCCL;
        }
        // 1. whatever NCCL the host process already carries (a torch host brings its own, newer than the system's:
        //    loading the system copy first would make the host's later import fail on a missing symbol)
        c->nccl_lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_LOCAL);
        // 2. an explicit path, 3. the system library — never RTLD_GLOBAL: our copy must not answer anyone else's symbols
        if (!c->nccl_lib) {
            const char* extra = getenv("CRO_NCCL_PATH");
            if (extra && *extra) c->nccl_lib = dlopen(extra, RTLD_NOW | RTLD_LOCAL);
        }
        if (!c->nccl_lib) c->nccl_lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
        if (!c->nccl_lib) c->nccl_lib = dlopen("libnccl.so", RTLD_NOW | RTLD_LOCAL);
        if (!c->nccl_lib) {
            c->set_error("libnccl.so.2 not found (set CRO_NCCL_PATH)");
            return CRO_ERR_NCCL;
        }
    }
    c->ncclCommInitAll = (int (*)(void**, int, const int*))dlsym(c->nccl_lib, "ncclCommInitAll");
    c->ncclGroupStart = (int (*)())dlsym(c->nccl_lib, "ncclGroupStart");
    c->ncclGroupEnd = (int (*)())dlsym(c->nccl_lib, "ncclGroupEnd");
    c->ncclGetErrorString = (const char* (*)(int))dlsym(c->nccl_lib, "ncclGetErrorString");
    auto ag = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(c->nccl_lib, "ncclAllGather");
    if (!c->ncclCommInitAll || !c->ncclGroupStart || !c->ncclGroupEnd || !ag) {
        c->set_error("libnccl lacks a required symbol");
        return CRO_ERR_NCCL;
    }
    c->ncclAllGather = ag;
    return CRO_OK;
}

}  // namespace

// One call = the full-box probe (BASELINE config 3).  Everything is ENQUEUED first — per-device probe graphs,
// the NVLink rounds chained across devices by events, the device-side verdicts, the all-gather, the copy-back —
// and only then does the host wait, once per device.
int ctx_probe_all(cro_ctx* c, cro_probe_result* out, int cap, int* n_out) {
    if (!c || !out || !n_out) return CRO_ERR_INVALID_ARG;
    const int n = (int)c->devs.size();
    *n_out = n;
    if (cap < n) return CRO_ERR_BUFFER_SMALL;
    if (n == 0) return CRO_OK;
    std::lock_guard<std::mutex> all(c->all_mu);
    const cro_opts& o = c->opts;
    Range nv_all(c, "cro.probe_all");
    const uint64_t t_call = now_ns();
    c->fullbox = FullBoxTimes{};
    uint32_t host_syncs = 0;

    std::vector<std::unique_lock<std::mutex>> locks;
    for (int i = 0; i < n; ++i) locks.emplace_back(c->devs[(size_t)i]->mu);
    for (int i = 0; i < n; ++i) {
        Device* d = c->devs[(size_t)i].get();
        drain_pending(c, d);
        d->done.clear();
        d->lane_head = 0;
    }
    const bool p2p = n > 1 && !(o.flags & CRO_F_SKIP_P2P);
    const bool push = p2p && !(o.flags & CRO_F_SKIP_P2P_WRITE);
    bool use_nccl = n > 1 && !(o.flags & CRO_F_SKIP_NCCL);
    bool nccl_degraded = false;
    int rc;
    // one-time setup (peer mappings, latency tables, communicators) happens BEFORE anything is enqueued
    if (p2p) {
        if ((rc = enable_peers(c))) return rc;
        if ((rc = ensure_chase(c, o.latency_hops))) return rc;
    }
    if (use_nccl && load_nccl(c) != CRO_OK) {
        // no usable libnccl in reach: the structs still come back, per device over pinned memory ("replicas only",
        // SURVEY.md §8e) — the call says so (cro_fullbox_time.gather, last error) instead of failing the attach
        use_nccl = false;
        nccl_degraded = true;
    }
    if (use_nccl) {
        if (!c->nccl_ready) {
            Range nv(c, "cro.nccl.init");
            std::vector<int> ords;
            for (auto& d : c->devs) ords.push_back(d->ordinal);
            c->nccl_comms.assign((size_t)n, nullptr);
            int r = c->ncclCommInitAll(c->nccl_comms.data(), n, ords.data());
            if (r != 0) {
                c->set_error(std::string("ncclCommInitAll: ") + (c->ncclGetErrorString ? c->ncclGetErrorString(r) : "error"));
                return CRO_ERR_NCCL;
            }
            c->nccl_ready = true;
        }
    }
    const auto rounds = p2p ? one_factorisation(n) : std::vector<std::vector<std::pair<int, int>>>();
    for (int i = 0; i < n && p2p; ++i) {
        Device* d = c->devs[(size_t)i].get();
        CU_TRY(c, cudaSetDevice(d->ordinal));
        while (d->ev_push_done.size() < rounds.size()) {
            cudaEvent_t e1, e2;
            CU_TRY(c, cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
            CU_TRY(c, cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
            d->ev_push_done.push_back(e1);
            d->ev_reread_done.push_back(e2);
        }
    }

    // ---- phase 1: every device's HBM probe, one graph launch each ---------------------------------------
    {
        Range nv(c, "cro.probe_all.hbm");
        for (int i = 0; i < n; ++i) {
            Device* d = c->devs[(size_t)i].get();
            if ((rc = probe_enqueue(c, d, d->lanes[0]))) return rc;
            if (p2p) {
                // what this device's first p2p_bytes must fold to, for the peers that will read them
                CU_TRY(c, launch_expected(d->plan, std::min<uint64_t>(o.p2p_bytes, d->sweep_bytes), imm_params(d), d->scratch_pfx,
                                          &d->d_out[kSlotPrefix], d->aux));
                c->launches++;
                CU_TRY(c, cudaEventRecord(d->ev_aux_done, d->aux));
                CU_TRY(c, cudaStreamWaitEvent(d->stream, d->ev_aux_done, 0));
                CU_TRY(c, cudaEventRecord(d->ev_hbm_done, d->stream));
            }
        }
    }

    // ---- phase 2: NVLink rounds, 1-factorised so each GPU is in exactly one pair per round ----------------
    // Per round and device (partner p):  [wait p's HBM phase, p's previous re-read]  READ p's half A over the
    // link -> PUSH my prefix into p's half B -> [wait p's push]  RE-READ my own half B locally.  Both directions
    // of a pair run at once; nothing waits on the host.
    const bool unidir = env::get("CRO_P2P_UNIDIR") != 0;
    const unsigned rvp = env::get("CRO_P2P_READ_VARIANT"), wvp = env::get("CRO_P2P_WRITE_VARIANT");
    auto pair_ok = [&](int a, int b) { return a < 8 && b < 8 && c->devs[(size_t)a]->tmpl.p2p_access[b]; };
    auto push_bytes = [&](const Device* a, const Device* b) {
        return std::min<uint64_t>(std::min<uint64_t>(o.p2p_bytes, a->sweep_bytes), b->sweep_bytes);
    };
    if (p2p) {
        Range nv(c, "cro.probe_all.nvlink");
        for (size_t r = 0; r < rounds.size(); ++r) {
            std::vector<std::pair<int, int>> directed;
            for (const auto& p : rounds[r]) {
                directed.push_back({p.first, p.second});
                // CRO_P2P_UNIDIR=1 (measurement only, tools/p2p_variants.py): one direction per pair, to see what the
                // link gives when its other half is idle; the reverse direction's result slots stay zero
                if (!unidir) directed.push_back({p.second, p.first});
            }
            for (const auto& pr : directed) {                       // stage A: read + push
                Device* a = c->devs[(size_t)pr.first].get();
                Device* b = c->devs[(size_t)pr.second].get();
                if (!pair_ok(pr.first, pr.second)) continue;
                CU_TRY(c, cudaSetDevice(a->ordinal));
                CU_TRY(c, cudaStreamWaitEvent(a->stream, b->ev_hbm_done, 0));
                if (r > 0) CU_TRY(c, cudaStreamWaitEvent(a->stream, b->ev_reread_done[r - 1], 0));
                // TMA bulk copies straight out of the peer's HBM (cp.async.bulk on the peer-mapped address) into
                // this GPU's shared memory, checksummed as they land
                CU_TRY(c, launch_read(a->plan, rvp, b->region, std::min<uint64_t>(o.p2p_bytes, b->sweep_bytes), imm_params(a),
                                      a->scratch, &a->d_out[kSlotP2P0 + 3 * pr.second], a->stream));
                c->launches++;
                if (push) {
                    // posted NVLink writes: a streams its own prefix through shared memory (bulk load from local
                    // HBM, bulk store to the peer-mapped address, folded on the way) into half B of b's region
                    CU_TRY(c, launch_copy(a->plan, wvp, b->region + b->sweep_bytes, a->region, push_bytes(a, b), imm_params(a),
                                          a->scratch, &a->d_out[kSlotP2P0 + 3 * pr.second + 1], a->stream));
                    c->launches++;
                }
                CU_TRY(c, cudaEventRecord(a->ev_push_done[r], a->stream));
            }
            for (const auto& pr : directed) {                       // stage B: the receiver checks what landed
                Device* a = c->devs[(size_t)pr.first].get();          // pusher
                Device* b = c->devs[(size_t)pr.second].get();         // receiver
                if (!pair_ok(pr.first, pr.second)) continue;
                CU_TRY(c, cudaSetDevice(b->ordinal));
                if (push) {
                    CU_TRY(c, cudaStreamWaitEvent(b->stream, a->ev_push_done[r], 0));
                    CU_TRY(c, launch_read(b->plan, resolve_read_variant(CRO_READ_AUTO, push_bytes(a, b)), b->region + b->sweep_bytes,
                                          push_bytes(a, b), imm_params(b), b->scratch, &b->d_out[kSlotP2P0 + 3 * pr.first + 2], b->stream));
                    c->launches++;
                }
                CU_TRY(c, cudaEventRecord(b->ev_reread_done[r], b->stream));
            }
            if (unidir)   // the idle direction's devices still have to publish their round events
                for (const auto& p : rounds[r]) {
                    Device* b = c->devs[(size_t)p.second].get();
                    CU_TRY(c, cudaSetDevice(b->ordinal));
                    CU_TRY(c, cudaEventRecord(b->ev_push_done[r], b->stream));
                    Device* a = c->devs[(size_t)p.first].get();
                    CU_TRY(c, cudaSetDevice(a->ordinal));
                    CU_TRY(c, cudaEventRecord(a->ev_reread_done[r], a->stream));
                }
        }
        // latency: every device chases all its peers at once (one warp per peer, one load in flight each),
        // after EVERY device has finished its bandwidth legs so the links are quiet
        for (int i = 0; i < n; ++i) {
            Device* d = c->devs[(size_t)i].get();
            CU_TRY(c, cudaSetDevice(d->ordinal));
            CU_TRY(c, cudaEventRecord(d->ev_chase_ready, d->stream));
        }
        for (int i = 0; i < n; ++i) {
            Device* d = c->devs[(size_t)i].get();
            CU_TRY(c, cudaSetDevice(d->ordinal));
            ChaseArgs ca{};
            ca.n = (unsigned)n;
            ca.hops = o.latency_hops;
            for (int j = 0; j < n; ++j) {
                if (j == i || !pair_ok(i, j)) continue;
                CU_TRY(c, cudaStreamWaitEvent(d->stream, c->devs[(size_t)j]->ev_chase_ready, 0));
                ca.table[j] = c->devs[(size_t)j]->d_chase_tables[(size_t)i];
            }
            CU_TRY(c, cudaMemsetAsync(d->d_chase_out, 0, 2 * CRO_MAX_DEVICES * sizeof(unsigned long long), d->stream));
            CU_TRY(c, launch_chase(ca, d->d_chase_out, d->stream));
            c->launches++;
            P2PFinalizeArgs pa{};
            pa.out = d->d_result;
            pa.slots = d->d_out;
            pa.chase_out = d->d_chase_out;
            pa.n = (unsigned)n;
            pa.self = (unsigned)i;
            pa.hops = o.latency_hops;
            pa.have_push = (push && !unidir) ? 1u : 0u;
            pa.push_folded = wvp == COPY_TMA_FUSED ? 1u : 0u;   // the plain copies land bytes but fold nothing: only the receiver checks
            pa.p2p_bytes = o.p2p_bytes;
            pa.stamp = d->nonce_cur;
            for (int j = 0; j < n; ++j) {
                if (j == i || !pair_ok(i, j)) continue;
                pa.peer_slots[j] = c->devs[(size_t)j]->d_out;
                pa.peer_stamp[j] = c->devs[(size_t)j]->nonce_cur;
                pa.chase_expect[j] = d->chase_expect[(size_t)j];
            }
            if (unidir)     // measurement mode: only the pairs' first devices read; check nothing that did not run
                for (const auto& rd : rounds)
                    for (const auto& p : rd)
                        if (p.second == i) pa.peer_slots[p.first] = nullptr;
            CU_TRY(c, launch_p2p_finalize(pa, d->stream));
            c->launches++;
            CU_TRY(c, cudaMemcpyAsync(d->h_chase_out, d->d_chase_out, 2 * CRO_MAX_DEVICES * sizeof(unsigned long long), cudaMemcpyDeviceToHost, d->stream));
            CU_TRY(c, cudaMemcpyAsync(d->h_out, d->d_out, sizeof(SweepOut) * kSlotCount, cudaMemcpyDeviceToHost, d->stream));
        }
    }

    // ---- phase 3: ONE all-gather of the 512-byte structs, enqueued behind the verdict kernels ---------------
    if (use_nccl) {
        Range nv(c, "cro.probe_all.allgather");
        CU_TRY(c, cudaSetDevice(c->devs[0]->ordinal));
        CU_TRY(c, cudaEventRecord(c->devs[0]->ev0, c->devs[0]->stream));
        int r = c->ncclGroupStart();
        for (int i = 0; r == 0 && i < n; ++i) {
            Device* d = c->devs[(size_t)i].get();
            r = c->ncclAllGather(d->d_result, d->d_gather, sizeof(cro_probe_result), /*ncclUint8*/ 1,
                                 c->nccl_comms[(size_t)i], d->stream);
        }
        int r2 = c->ncclGroupEnd();
        if (r != 0 || r2 != 0) {
            c->set_error(std::string("ncclAllGather: ") + (c->ncclGetErrorString ? c->ncclGetErrorString(r ? r : r2) : "error"));
            return CRO_ERR_NCCL;
        }
        CU_TRY(c, cudaSetDevice(c->devs[0]->ordinal));
        CU_TRY(c, cudaEventRecord(c->devs[0]->ev1, c->devs[0]->stream));
        for (int i = 0; i < n; ++i) {
            Device* d = c->devs[(size_t)i].get();
            CU_TRY(c, cudaSetDevice(d->ordinal));
            CU_TRY(c, cudaMemcpyAsync(d->h_gather, d->d_gather, sizeof(cro_probe_result) * (size_t)n, cudaMemcpyDeviceToHost, d->stream));
        }
    } else {
        for (int i = 0; i < n; ++i) {
            Device* d = c->devs[(size_t)i].get();
            CU_TRY(c, cudaSetDevice(d->ordinal));
            CU_TRY(c, cudaMemcpyAsync(d->h_result, d->d_result, sizeof(cro_probe_result), cudaMemcpyDeviceToHost, d->stream));
        }
    }
    c->fullbox.enqueue_ns = now_ns() - t_call;

    // While the GPUs work: a fresh ECC read per device (NVML, 3–5 ms each — on the critical path it would cost the box
    // more than the NVLink rounds of one pair; and eight of them can outlast the 36 ms the GPUs need, so a device is
    // asked at most once a second).  The structs being gathered right now carry the count staged before this call; a
    // count that moved is staged for the next probe, and a FAILING probe re-reads it at once anyway.
    std::vector<int> restage;
    if (n > 1) {
        const auto t_now = std::chrono::steady_clock::now();
        for (int i = 0; i < n; ++i) {
            Device* d = c->devs[(size_t)i].get();
            if (t_now - d->ecc_at < std::chrono::seconds(1)) continue;
            d->ecc_at = t_now;
            refresh_ecc(c, d);
            if (d->tmpl.ecc_errors != d->ecc_uncorrected) restage.push_back(i);
        }
    }

    // ---- the only host waits: one per device ------------------------------------------------------------------
    {
        Range nv(c, "cro.probe_all.wait");
        for (int i = 0; i < n; ++i) {
            Device* d = c->devs[(size_t)i].get();
            CU_TRY(c, cudaSetDevice(d->ordinal));
            if ((rc = wait_stream(c, d))) return rc;
            ++host_syncs;
        }
    }
    for (int i = 0; i < n; ++i) {
        c->devs[(size_t)i]->lanes[0].in_flight = false;
        c->devs[(size_t)i]->last_lane = 0;
    }
    int worst = CRO_OK;
    if (use_nccl) {
        for (int i = 1; i < n; ++i)
            if (memcmp(c->devs[0]->h_gather, c->devs[(size_t)i]->h_gather, sizeof(cro_probe_result) * (size_t)n) != 0) {
                c->set_error("all-gather result differs between rank 0 and rank " + std::to_string(i));
                return CRO_ERR_NCCL;
            }
        memcpy(out, c->devs[0]->h_gather, sizeof(cro_probe_result) * (size_t)n);
        float ms = 0;
        CU_TRY(c, cudaSetDevice(c->devs[0]->ordinal));
        if (cudaEventElapsedTime(&ms, c->devs[0]->ev0, c->devs[0]->ev1) == cudaSuccess) c->fullbox.gather_ns = ms_to_ns(ms);
    } else {
        for (int i = 0; i < n; ++i) out[i] = *c->devs[(size_t)i]->h_result;
    }
    c->m_fullbox++;
    for (int i = 0; i < n; ++i) {
        Device* d = c->devs[(size_t)i].get();
        *d->h_result = out[i];
        d->last = out[i];
        d->have_last = true;
        c->m_probes++;
        if (out[i].status != CRO_OK) c->m_probe_failures++;
        if (out[i].status != CRO_OK) {
            worst = out[i].status;
            c->set_error(describe_failure(d, out[i]));
        }
        c->fullbox.hbm_ns = std::max<uint64_t>(c->fullbox.hbm_ns, out[i].total_ns);
        if (p2p) {
            unsigned long long lo = ~0ull, hi = 0;
            for (int j = 0; j < n; ++j) {
                if (j == i) continue;
                for (int k = 0; k < 3; ++k) {
                    const SweepOut& s = d->h_out[kSlotP2P0 + 3 * j + k];
                    if (s.stamp != d->nonce_cur) continue;
                    lo = std::min(lo, s.t0);
                    hi = std::max(hi, s.t1);
                }
                c->fullbox.chase_ns = std::max<uint64_t>(c->fullbox.chase_ns, d->h_chase_out[2 * j + 1]);
            }
            if (hi > lo) c->fullbox.p2p_ns = std::max<uint64_t>(c->fullbox.p2p_ns, hi - lo);
        }
    }
    for (int i : restage) {
        Device* d = c->devs[(size_t)i].get();
        CU_TRY(c, cudaSetDevice(d->ordinal));
        if ((rc = stage_template(c, d))) return rc;
    }
    c->fullbox.rounds = (uint32_t)rounds.size();
    c->fullbox.host_syncs = host_syncs;
    c->fullbox.gather = use_nccl ? CRO_GATHER_NCCL : nccl_degraded ? CRO_GATHER_DEGRADED : CRO_GATHER_HOST;
    c->fullbox.wall_ns = now_ns() - t_call;
    return worst;
}

int ctx_p2p_detail(cro_ctx* c, int idx, int peer, cro_p2p_detail* out) {
    Device* d = dev_at(c, idx);
    Device* p = dev_at(c, peer);
    if (!d || !p || !out || idx == peer) return CRO_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> all(c->all_mu);
    memset(out, 0, sizeof *out);
    const SweepOut& rd = d->h_out[kSlotP2P0 + 3 * peer];
    const SweepOut& ps = d->h_out[kSlotP2P0 + 3 * peer + 1];
    const SweepOut& landed = p->h_out[kSlotP2P0 + 3 * idx + 2];   // the peer's re-read of what this device pushed
    const SweepOut& want = p->h_out[kSlotPrefix];
    if (rd.stamp == d->nonce_cur) {
        out->read_ns = rd.t1 - rd.t0;
        out->read_xor = rd.x; out->read_sum = rd.s; out->read_wsum = rd.w;
    }
    if (ps.stamp == d->nonce_cur) out->push_ns = ps.t1 - ps.t0;
    if (landed.stamp == p->nonce_cur) {
        out->reread_ns = landed.t1 - landed.t0;
        out->landed_xor = landed.x; out->landed_sum = landed.s; out->landed_wsum = landed.w;
    }
    if (want.stamp == p->nonce_cur) { out->expect_xor = want.x; out->expect_sum = want.s; out->expect_wsum = want.w; }
    out->chase_end = (uint32_t)d->h_chase_out[2 * peer];
    out->chase_ns = d->h_chase_out[2 * peer + 1];
    out->chase_expect = (size_t)peer < d->chase_expect.size() ? d->chase_expect[(size_t)peer] : 0;
    out->hops = c->opts.latency_hops;
    out->access = idx < 8 && peer < 8 ? d->tmpl.p2p_access[peer] : 0;
    return CRO_OK;
}

}  // namespace cro
