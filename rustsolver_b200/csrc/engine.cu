// Host engine behind the C ABI (include/b200cfr.h): owns device memory, the per-round launch
// descriptors, the CUDA graph of one iteration and (when board-sharded) the NCCL communicator.
//
// Replaces MCCFRTrainer::{init, train} (src/solver/cfr.rs:159-297) and the InfosetTable
// (src/solver/infoset.rs:6-49).  No CPU fallback: without a CUDA device rs_create fails.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/b200cfr.h"
#include <cmath>

#include "abstraction_kernels.h"
#include "histogram_kernel.h"
#include "indexer_kernel.h"
#include "kernels.cuh"
#include "plan.h"
#include "street_kernel.cuh"

namespace rs {

thread_local std::string g_last_error;

static int set_err(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

// ---- NCCL through dlopen: the library loads on CPU-only hosts and single-GPU runs never touch it ----
namespace nccl {
typedef struct {
    char internal[128];
} UniqueId;
typedef void* Comm;
typedef int (*GetUniqueId_t)(UniqueId*);
typedef int (*CommInitRank_t)(Comm*, int, UniqueId, int);
typedef int (*AllReduce_t)(const void*, void*, size_t, int, int, Comm, cudaStream_t);
typedef int (*CommDestroy_t)(Comm);
typedef const char* (*GetErrorString_t)(int);
struct Api {
    void* lib = nullptr;
    GetUniqueId_t GetUniqueId = nullptr;
    CommInitRank_t CommInitRank = nullptr;
    AllReduce_t AllReduce = nullptr;
    CommDestroy_t CommDestroy = nullptr;
    GetErrorString_t GetErrorString = nullptr;
};
static Api g_api;
constexpr int kFloat32 = 7;  // ncclFloat32
constexpr int kSum = 0;      // ncclSum

static bool load(std::string* err) {
    if (g_api.lib) return true;
    const char* env = getenv("RS_NCCL_LIB");
    const char* names[] = {env, "libnccl.so.2", "libnccl.so"};
    void* lib = nullptr;
    for (const char* n : names) {
        if (!n || !*n) continue;
        lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (lib) break;
    }
    if (!lib) {
        *err = "cannot dlopen libnccl.so.2 (set RS_NCCL_LIB to its path)";
        return false;
    }
    g_api.lib = lib;
    g_api.GetUniqueId = (GetUniqueId_t)dlsym(lib, "ncclGetUniqueId");
    g_api.CommInitRank = (CommInitRank_t)dlsym(lib, "ncclCommInitRank");
    g_api.AllReduce = (AllReduce_t)dlsym(lib, "ncclAllReduce");
    g_api.CommDestroy = (CommDestroy_t)dlsym(lib, "ncclCommDestroy");
    g_api.GetErrorString = (GetErrorString_t)dlsym(lib, "ncclGetErrorString");
    if (!g_api.GetUniqueId || !g_api.CommInitRank || !g_api.AllReduce || !g_api.CommDestroy) {
        *err = "libnccl is missing expected symbols";
        g_api = Api();
        return false;
    }
    return true;
}
}  // namespace nccl

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return set_err(RS_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));      \
    } while (0)

// plan.h: BatchIndexFn backed by the device indexer
static bool device_batch_index(const HandIndexer& ix, const uint8_t* cards, size_t n, uint64_t* out, std::string* err) {
    return gpu_index_hands(ix, ix.rounds() - 1, cards, n, out, nullptr, err);
}

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    ~DevBuf() {
        if (p) cudaFree(p);
    }
    cudaError_t alloc(size_t count) {
        n = count;
        if (count == 0) count = 1;
        return cudaMalloc(&p, count * sizeof(T));
    }
    cudaError_t upload(const T* src, size_t count) {
        cudaError_t e = alloc(count);
        if (e != cudaSuccess || count == 0) return e;
        return cudaMemcpy(p, src, count * sizeof(T), cudaMemcpyHostToDevice);
    }
    cudaError_t upload(const std::vector<T>& v) { return upload(v.data(), v.size()); }
    cudaError_t zero() { return cudaMemset(p, 0, (n ? n : 1) * sizeof(T)); }
};

struct RoundDev {
    // per player q, board-local hand order (plan.h: LocalTables)
    DevBuf<uint16_t> row_of_pos[2], row_start[2], row_pos[2], cl_pos[2], parent_pos[2], child_pos[2], slot_of_pos[2];
    DevBuf<HandRec> hrec[2];
    DevBuf<uint32_t> n_rows[2], n_rows_pad[2], n_live[2];
    DevBuf<uint64_t> board_off[2];
    DevBuf<float> regrets[2], ssum[2];
    DevBuf<float> chance_scale;
    DevBuf<int32_t> parent_board;
    // transients of one traversal (shared by both traversers, sized for the larger)
    DevBuf<float> rbuf, cbuf, gathered;
    DevBuf<float> sbuf[2];  // street-root values in parent-board order, one pool per traverser (unwritten entries must stay 0)
    uint32_t n_leaves = 0, n_boards = 0;
};

// a traversal's task list with ticket numbering materialised for a given number of instances per round
struct TaskSet {
    DevBuf<NodeTask> tasks;
    DevBuf<TaskSrc> srcs;
    DevBuf<uint32_t> tix;  // instance slot -> node-task index
    DevBuf<uint32_t> order;  // ticket -> instance slot (empty: identity), see TaskArgs::order
    uint32_t n_tickets = 0, phase_cut = 0, n_tasks = 0;
    uint32_t street_lo = 0, street_hi = 0;  // tickets of the final round's node tasks (replaced by the street kernel)
    uint32_t street_inst = 0;               // instances (boards or sampled run-outs) of the final round
    // Tickets are emitted street by street (plan.cpp: TaskGen::run): [down r0][down r1][down r2][up r2][gather][up r1]...
    // A run is a maximal ticket range whose tasks need the same block size (Engine::round_threads); a traversal is
    // launched run by run, so the rounds with fewer live hands (the river: 1081 of 1176 / 1326) run at the smaller
    // block with one more resident CTA per SM.
    struct Run {
        uint32_t t0, t1;
        int threads;
    };
    std::vector<Run> runs;
    uint32_t xch_lo = 0, xch_hi = 0;  // tickets of the gathers that exchange their sums between the ranks (none: lo == hi)
    struct Section {  // the down or up tasks of one round: where its algorithmic table bytes are accounted
        uint32_t first;
        uint32_t round_k;
        bool up;
    };
    std::vector<Section> sections;
};

// device copy of one traverser's final-street programs (street.h)
struct StreetDev {
    DevBuf<SwSeg> segs;
    DevBuf<SwDown> downs;
    DevBuf<SwUp> ups;
    DevBuf<SwTerm> terms;
    DevBuf<uint32_t> prog, prog_off, l_steps, c_steps, hinfo;
    uint32_t n_segs = 0;
};

struct Engine {
    Plan plan;
    int device = 0;
    int threads = 512;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t graph_exec = nullptr;
    bool use_graph = true;
    nccl::Comm comm = nullptr;
    bool isolated = false;  // RS_FLAG_SHARD_ISOLATED: a shard without peers, no exchange of any kind

    RoundDev rd[3];
    DevBuf<float> scratch;  // strategy read-outs
    DevBuf<float> root_weights[2];
    TaskSet full[2];                                        // every board of every round (rs_iterate)
    std::map<int, std::unique_ptr<TaskSet[]>> sampled_sets;  // by number of sampled paths (rs_iterate_sampled)
    DevBuf<int32_t> sample_board[3];
    int sample_cap = 0;
    DevBuf<uint32_t> flags;
    DevBuf<TaskCtl> ctl;
    DevBuf<unsigned long long> timing;
    // in-kernel exchange of the chance-node partial sums (board-sharded engines): one allocation per rank,
    // [flags: 2 * vectors u32, padded to 256 B][data: 2 * vectors * Hpad floats], vectors = leaves * parent boards * world
    DevBuf<unsigned char> xch;
    size_t xch_flag_bytes = 0, xch_vectors = 0;
    void* xch_peer_base[RS_MAX_PEERS] = {nullptr};
    bool fused_exchange = false;
    float prune_threshold = -INFINITY;  // rs_set_prune_threshold
    // rs_set_opponent_sampling: every CFR traversal draws one action per opponent hand and node (kernels.cuh: xs_uniform)
    int xs_mode = 0;
    uint64_t xs_seed = 0, xs_count = 0;  // traversals since the mode was set: the key of a traversal is splitmix64(seed + count)
    // bounded waits (kernels.cuh: host_abort / wait_timeout_ns)
    uint32_t* abort_host = nullptr;   // mapped pinned word the host raises (rs_abort)
    uint32_t* abort_dev = nullptr;    // its device alias
    uint64_t wait_timeout_ms = 30000; // rs_set_wait_timeout_ms
    bool aborted = false;             // a traversal gave up: the tables are partly updated, the engine refuses further work
    int check_abort(const char* what);
    int maybe_discount();
    // rs_set_update_rule: the rule and t of the last iteration run under it.  VANILLA launches the plain CFR builds and
    // writes no factors, so the default path is exactly what it was without the rule.
    rs_update_rule rule = {RS_RULE_VANILLA, 1.5f, 0.f, 2.f};
    uint64_t rule_t = 0;
    bool rule_on() const { return rule.kind != RS_RULE_VANILLA; }
    int advance_rule();
    uint64_t last_discount_period = 0;
    // fused final-street kernel (street_kernel.cu); off: the final round runs as node tasks like the others
    bool street_on = false;
    StreetDev street[2];
    DevBuf<float> st_scratch;
    size_t st_stride = 0, st_smem = 0;
    int st_XP = 0, st_rows = 0, st_vy_rows = 0, st_vm_rows = 0, st_slots = 0, st_threads = 0, st_blocks_per_sm = 1, st_qs = 1, st_qm = 1;
    int slots = 1;
    size_t smem_bytes = 0;  // dynamic shared memory of the wide task-kernel build
    size_t smem_small = 0;  // of the 288-thread build
    int blocks_per_sm = 1, n_sms = 148;
    int round_threads[3] = {0, 0, 0};  // compute threads the tasks of round k need: live hands / 4, a warp multiple
    int bps_small = 0;                 // resident CTAs per SM of the 288-thread specialisation (0: no round fits it)
    // a piece of `tickets` instances at `thr` compute threads: the wide specialisation unless a third CTA per SM gets work
    bool wide_for(int thr, uint64_t tickets) const {
        return thr > 288 || bps_small == 0 || getenv("RS_WIDE_ONLY") || (tickets <= uint64_t(n_sms) * blocks_per_sm && !getenv("RS_SMALL_ONLY"));
    }
    // profiling: when non-null, enqueue_traversal brackets every launch with an event pair
    std::vector<rs_kernel_time>* prof = nullptr;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;

    uint64_t iterations = 0;
    double device_ms = 0;
    uint64_t launches = 0;
    uint64_t launches_per_iter = 0;
    uint64_t table_bytes = 0;
    uint64_t updates_global = 0;
    uint64_t discount_interval = 0, discount_cap = 0;

    void close_peers() {
        for (int r = 0; r < RS_MAX_PEERS; ++r) {
            if (xch_peer_base[r] && r != plan.rank) cudaIpcCloseMemHandle(xch_peer_base[r]);
            xch_peer_base[r] = nullptr;
        }
    }

    ~Engine() {
        close_peers();
        if (graph_exec) cudaGraphExecDestroy(graph_exec);
        if (graph) cudaGraphDestroy(graph);
        if (comm && nccl::g_api.CommDestroy) nccl::g_api.CommDestroy(comm);
        if (abort_host) cudaFreeHost(abort_host);
        if (root_stage) cudaFreeHost(root_stage);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (stream) cudaStreamDestroy(stream);
    }

    int init(const rs_config* cfg);
    void fill_args(TaskArgs* a, int trav, const TaskSet& set) const;
    int materialize(int trav, const uint32_t counts[3], TaskSet* out);
    int enqueue_sampled(int n_paths, int n_paths_global, uint64_t* count);
    // n_paths >= 0: sampled iteration on this rank's n_paths run-outs (of n_paths_global over all ranks)
    int enqueue_traversal(int trav, int mode, uint64_t* count, const TaskSet* set = nullptr, int n_paths = -1, int n_paths_global = 0);
    int init_street();
    int enqueue_street(int trav, int mode, const TaskSet& set, int n_paths);
    int enqueue_iteration(uint64_t* count);
    int iterate(uint64_t n);
    int root_sum(int player, double* out);
    int root_values(int player, std::vector<float>* out);
    int root_values_into(int player, float* dst);
    DevBuf<float> root_out;
    float* root_stage = nullptr;
    size_t root_stage_n = 0;
    int prof_begin();
    int prof_end(uint32_t kind, uint32_t k, int trav, uint32_t grid, uint64_t table_bytes, uint64_t vector_bytes);
};

template <class T>
static std::vector<T> slice(const std::vector<T>& v, size_t lo, size_t hi, size_t stride) {
    if (v.empty()) return {};
    return std::vector<T>(v.begin() + lo * stride, v.begin() + hi * stride);
}

int Engine::init(const rs_config* cfg) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return set_err(RS_ERR_CUDA, std::string("no CUDA device available (the engine has no CPU fallback): ") +
                                        (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    device = cfg->device;
    if (device < 0 || device >= ndev) return set_err(RS_ERR_INVALID, "device ordinal out of range");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return set_err(RS_ERR_UNSUPPORTED, "kernels are built for sm_100a only; found an older device");
    if (cfg->threads_per_block)
        return set_err(RS_ERR_INVALID, "threads_per_block is derived from the range size (4 hands per thread) and cannot be set");
    if (cfg->flags & ~uint32_t(RS_FLAG_ALL)) return set_err(RS_ERR_INVALID, "unknown bits in rs_config.flags");
    use_graph = !(cfg->flags & RS_FLAG_NO_GRAPH);
    isolated = (cfg->flags & RS_FLAG_SHARD_ISOLATED) != 0;
    discount_interval = cfg->discount_interval;
    discount_cap = cfg->discount_cap;
    CU(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    CU(cudaEventCreate(&ev0));
    CU(cudaEventCreate(&ev1));

    const Plan& P = plan;
    for (int q = 0; q < 2; ++q) {
        std::vector<float> ones(P.H[q], 1.0f);
        CU(root_weights[q].upload(ones));
    }
    const int HP[2] = {int((P.H[0] + 3) & ~3u), int((P.H[1] + 3) & ~3u)};
    const size_t maxHP = size_t(std::max(HP[0], HP[1]));
    const bool street_wanted = P.street[0].eligible && P.street[1].eligible;
    threads = int(((maxHP / 4) + 31) / 32 * 32);
    if (threads > MAX_TASK_THREADS) return set_err(RS_ERR_UNSUPPORTED, "range larger than 1326 hands");
    // Per-round block size.  Live hands come first in the board-local order, so a round whose boards hold c public cards
    // never touches a position past min(H, C(52 - c, 2)): its tasks run with that many quads of threads.  The bound only
    // depends on the number of public cards, so every rank of a sharded engine cuts its launches at the same places.
    for (uint32_t k = 0; k < P.n_rounds; ++k) {
        round_threads[k] = threads;
        if (!P.board_mask[k].empty() && !getenv("RS_UNIFORM_BLOCK")) {
            const int left = 52 - __builtin_popcountll(P.board_mask[k][0]);
            const size_t live_max = std::min<size_t>(maxHP, size_t(left) * size_t(left - 1) / 2);
            round_threads[k] = std::min(threads, int((((live_max + 3) / 4) + 31) / 32 * 32));
        }
    }
    n_sms = prop.multiProcessorCount;
    if (street_wanted) {  // sets street_on when the fused street kernel fits
        int rc = init_street();
        if (rc != RS_OK) return rc;
    }
    for (uint32_t k = 0; k < P.n_rounds; ++k) {
        RoundDev& R = rd[k];
        const uint32_t lo = P.local_lo[k], hi = P.local_hi[k], nb = hi - lo;
        R.n_boards = nb;
        R.n_leaves = (k + 1 < P.n_rounds) ? uint32_t(P.segs[k + 1].size()) : 0;
        for (int q = 0; q < 2; ++q) {
            const RoundPlayerTables& T = P.tabs[k][q];
            const LocalTables& L = P.loc[k][q];
            const size_t hp = L.Hpad;
            CU(R.row_of_pos[q].upload(slice(L.row_of_pos, lo, hi, hp)));
            CU(R.row_start[q].upload(slice(L.row_start, lo, hi, hp + 4)));
            CU(R.row_pos[q].upload(slice(L.row_pos, lo, hi, hp)));
            CU(R.cl_pos[q].upload(slice(L.cl_pos, lo, hi, 2 * hp)));
            CU(R.slot_of_pos[q].upload(slice(L.slot_of_pos, lo, hi, hp)));
            {
                // four word planes per board: [board][word][pos] (see stage_recs)
                std::vector<HandRec> aos = slice(L.hrec, lo, hi, hp);
                std::vector<HandRec> soa(aos.size());
                const uint32_t* src = reinterpret_cast<const uint32_t*>(aos.data());
                uint32_t* dst = reinterpret_cast<uint32_t*>(soa.data());
                for (size_t b = 0; b < size_t(nb); ++b)
                    for (size_t i = 0; i < hp; ++i)
                        for (int wd = 0; wd < 4; ++wd) dst[(b * 4 + wd) * hp + i] = src[(b * hp + i) * 4 + wd];
                CU(R.hrec[q].upload(soa));
            }
            if (k > 0) {
                CU(R.parent_pos[q].upload(slice(L.parent_pos, lo, hi, hp)));
                CU(R.child_pos[q].upload(slice(L.child_pos, lo, hi, size_t(P.loc[k - 1][q].Hpad))));
            }
            CU(R.n_rows[q].upload(slice(T.n_rows, lo, hi, 1)));
            CU(R.n_rows_pad[q].upload(slice(L.n_rows_pad, lo, hi, 1)));
            CU(R.n_live[q].upload(slice(L.n_live, lo, hi, 1)));
            CU(R.board_off[q].upload(slice(T.board_off, lo, hi, 1)));
            const size_t cells = size_t(T.board_off[P.n_boards[k]]);
            CU(R.regrets[q].alloc(cells));
            CU(R.ssum[q].alloc(cells));
            CU(R.regrets[q].zero());
            CU(R.ssum[q].zero());
            table_bytes += 2 * cells * sizeof(float);
        }
        CU(R.chance_scale.upload(slice(P.chance_scale[k], lo, hi, 1)));
        std::vector<int32_t> pb(nb, -1);
        if (k > 0)
            for (uint32_t b = 0; b < nb; ++b) pb[b] = P.board_parent[k][lo + b] - int32_t(P.local_lo[k - 1]);
        CU(R.parent_board.upload(pb));
        // the fused street kernel keeps the final round's vectors in its own per-CTA scratch; only the root round's
        // value buffers are read from outside (rs_root_values)
        const bool fused_round = street_on && k + 1 == P.n_rounds;
        const size_t n_r = fused_round ? 0 : std::max(P.tl[0].n_rbuf[k], P.tl[1].n_rbuf[k]);
        const size_t n_c = (fused_round && k > 0) ? 0 : std::max(P.tl[0].n_cbuf[k], P.tl[1].n_cbuf[k]);
        CU(R.rbuf.alloc(n_r * nb * maxHP));
        CU(R.cbuf.alloc(n_c * nb * maxHP));
        CU(R.gathered.alloc(size_t(R.n_leaves) * nb * maxHP));
        for (int p = 0; p < 2; ++p) {
            CU(R.sbuf[p].alloc(size_t(P.tl[p].n_sbuf[k]) * nb * maxHP));
            CU(R.sbuf[p].zero());
        }
        CU(R.rbuf.zero());
        CU(R.cbuf.zero());
        CU(R.gathered.zero());
    }
    uint32_t max_tickets = 0;
    for (int p = 0; p < 2; ++p) {
        uint32_t counts[3] = {0, 0, 0};
        for (uint32_t k = 0; k < P.n_rounds; ++k) counts[k] = rd[k].n_boards;
        int rc = materialize(p, counts, &full[p]);
        if (rc != RS_OK) return rc;
        max_tickets = std::max(max_tickets, full[p].n_tickets);
        slots = std::max(slots, int(std::max(P.tl[p].max_terminal, 1 + P.tl[p].max_children)));
    }
    CU(timing.alloc(96));
    CU(timing.zero());
    CU(flags.alloc(max_tickets));
    CU(flags.zero());
    {
        TaskCtl c0{};
        c0.ticket = 0;
        c0.exited = 0;
        c0.xch_seq = 1;
        c0.epoch = 1;  // flags start at 0 = "never completed"
        c0.rule[0] = c0.rule[1] = c0.rule[2] = 1.f;
        c0.rule[3] = -INFINITY;
        CU(ctl.upload(&c0, 1));
        CU(cudaHostAlloc(reinterpret_cast<void**>(&abort_host), sizeof(uint32_t), cudaHostAllocMapped));
        *abort_host = 0;
        CU(cudaHostGetDevicePointer(reinterpret_cast<void**>(&abort_dev), abort_host, 0));
    }
    size_t smem_need = std::max(task_kernel_smem_bytes(true, slots, HP[0], HP[1]), task_kernel_smem_bytes(true, slots, HP[1], HP[0]));
    int max_optin = 0;
    CU(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    if (smem_need > size_t(max_optin))
        return set_err(RS_ERR_UNSUPPORTED, "node too wide for one CTA's shared memory: need " +
                                               std::to_string(smem_need) + " B, device allows " + std::to_string(max_optin));
    smem_bytes = smem_need;
    CU(configure_task_kernels(smem_need, threads, true, &blocks_per_sm));  // the wide specialisation, used by every engine
    if (blocks_per_sm < 1) return set_err(RS_ERR_UNSUPPORTED, "task kernel does not fit on an SM");
    for (uint32_t k = 0; k < P.n_rounds; ++k)
        if (round_threads[k] <= 288 && bps_small == 0) {
            smem_small = std::max(task_kernel_smem_bytes(false, slots, HP[0], HP[1]), task_kernel_smem_bytes(false, slots, HP[1], HP[0]));
            CU(configure_task_kernels(smem_small, 288, false, &bps_small));
            if (bps_small < 1) return set_err(RS_ERR_UNSUPPORTED, "task kernel does not fit on an SM");
        }
    n_sms = prop.multiProcessorCount;
    CU(scratch.alloc(size_t(1326) * MAX_ACTIONS));

    updates_global = P.updates_per_iter_local;
    if (P.world > 1 && !isolated) {
        std::string err;
        if (!nccl::load(&err)) return set_err(RS_ERR_NCCL, err);
        nccl::UniqueId id;
        static_assert(sizeof(id) == RS_NCCL_ID_BYTES, "nccl id size");
        memcpy(&id, cfg->nccl_id, sizeof(id));
        int rc = nccl::g_api.CommInitRank(&comm, P.world, id, P.rank);
        if (rc != 0)
            return set_err(RS_ERR_NCCL, std::string("ncclCommInitRank: ") +
                                            (nccl::g_api.GetErrorString ? nccl::g_api.GetErrorString(rc) : "error"));
        // global update count: all-reduce the local count once (as two floats of 24 bits each is lossy; use double via 2 x u32 halves)
        DevBuf<float> tmp;
        CU(tmp.alloc(4));
        uint64_t u = P.updates_per_iter_local;
        // replicated (unsharded) rounds are counted once: subtract on ranks > 0
        if (P.rank > 0)
            for (uint32_t k = 0; k < P.shard_round; ++k)
                for (int q = 0; q < 2; ++q) u -= P.tabs[k][q].board_off[P.n_boards[k]];
        float parts[4] = {float(u & 0xFFFFF), float((u >> 20) & 0xFFFFF), float((u >> 40) & 0xFFFFF), 0.f};
        CU(cudaMemcpy(tmp.p, parts, sizeof(parts), cudaMemcpyHostToDevice));
        rc = nccl::g_api.AllReduce(tmp.p, tmp.p, 4, nccl::kFloat32, nccl::kSum, comm, stream);
        if (rc != 0) return set_err(RS_ERR_NCCL, "ncclAllReduce failed");
        CU(cudaStreamSynchronize(stream));
        CU(cudaMemcpy(parts, tmp.p, sizeof(parts), cudaMemcpyDeviceToHost));
        updates_global = uint64_t(parts[0]) + (uint64_t(parts[1]) << 20) + (uint64_t(parts[2]) << 40);
    }
    if (P.world > 1 && P.shard_round >= 1 && !isolated) {
        const RoundDev& Par = rd[P.shard_round - 1];
        xch_vectors = size_t(Par.n_leaves) * Par.n_boards * size_t(P.world);
        xch_flag_bytes = (2 * xch_vectors * sizeof(uint32_t) + 255) & ~size_t(255);
        CU(xch.alloc(xch_flag_bytes + 2 * xch_vectors * maxHP * sizeof(float)));
        CU(xch.zero());
    }
    CU(cudaDeviceSynchronize());
    return RS_OK;
}


// Upload the final-street programs and size the per-CTA scratch of the fused street kernel.
int Engine::init_street() {
    const Plan& P = plan;
    uint32_t max_rows = 1, max_slots = 1, max_q_sd = 1, max_q_mo = 1;
    for (int p = 0; p < 2; ++p) {
        const StreetPlan& S = P.street[p];
        StreetDev& D = street[p];
        CU(D.segs.upload(S.segs));
        CU(D.downs.upload(S.downs));
        CU(D.ups.upload(S.ups));
        CU(D.terms.upload(S.terms));
        CU(D.prog.upload(S.prog));
        CU(D.prog_off.upload(S.prog_off));
        CU(D.l_steps.upload(S.l_steps));
        CU(D.c_steps.upload(S.c_steps));
        CU(D.hinfo.upload(S.hinfo));
        D.n_segs = uint32_t(S.segs.size());
        max_rows = std::max(max_rows, S.max_rows);
        max_slots = std::max(max_slots, S.max_slots);
        max_q_sd = std::max(max_q_sd, S.max_q_sd);
        max_q_mo = std::max(max_q_mo, S.max_q_mo);
    }
    const int HP[2] = {int((P.H[0] + 3) & ~3u), int((P.H[1] + 3) & ~3u)};
    const int HPmax = std::max(HP[0], HP[1]);
    st_XP = (HPmax + 31) & ~31;
    st_rows = int(max_rows);
    st_vy_rows = 4 * int(max_q_sd);
    st_vm_rows = 4 * int(max_q_sd + max_q_mo);
    st_slots = int(max_slots);
    st_stride = size_t(st_rows) * st_XP + size_t(st_vy_rows + st_vm_rows + st_slots) * HPmax;
    st_threads = threads;  // 4 hands per thread in one pass of the D and U phases
    if (const char* e = getenv("RS_STREET_THREADS")) st_threads = std::max(64, std::min(352, atoi(e) / 32 * 32));
    // quads staged per round: as many as fit the shared-memory budget of one CTA (3 CTAs per SM by default)
    size_t budget = 72 * 1024;
    if (const char* e = getenv("RS_STREET_SMEM_KB")) budget = size_t(std::max(16, atoi(e))) * 1024;
    st_qs = st_qm = 1;
    const int max_q = st_threads / 32;  // one warp per quad reduces the totals
    while (st_qs < int(max_q_sd) && st_qs < max_q && street_smem_bytes(st_qs + 1, st_qm, HPmax, HPmax) <= budget) ++st_qs;
    while (st_qm < int(max_q_mo) && st_qm < max_q && street_smem_bytes(st_qs, st_qm + 1, HPmax, HPmax) <= budget) ++st_qm;
    st_smem = street_smem_bytes(st_qs, st_qm, HPmax, HPmax);
    int max_optin = 0;
    CU(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    if (st_smem > size_t(max_optin)) return RS_OK;  // does not fit one CTA: stay on the task kernel
    CU(configure_street_kernels(st_smem, st_threads, &st_blocks_per_sm));
    if (st_blocks_per_sm < 1) return RS_OK;
    if (const char* e = getenv("RS_STREET_BLOCKS")) st_blocks_per_sm = std::max(1, std::min(st_blocks_per_sm, atoi(e)));
    CU(st_scratch.alloc(st_stride * size_t(n_sms) * st_blocks_per_sm));
    CU(st_scratch.zero());
    street_on = true;
    return RS_OK;
}

int Engine::enqueue_street(int trav, int mode, const TaskSet& set, int n_paths) {
    const Plan& P = plan;
    const uint32_t k = P.n_rounds - 1;
    const RoundDev& R = rd[k];
    const StreetDev& D = street[trav];
    StreetArgs a;
    memset(&a, 0, sizeof(a));
    for (int q = 0; q < 2; ++q) {
        DevRoundPlayer& d = a.rp[q];
        d.row_of_pos = R.row_of_pos[q].p;
        d.row_start = R.row_start[q].p;
        d.row_pos = R.row_pos[q].p;
        d.cl_pos = R.cl_pos[q].p;
        d.parent_pos = R.parent_pos[q].p;
        d.child_pos = R.child_pos[q].p;
        d.slot_of_pos = R.slot_of_pos[q].p;
        d.hrec = R.hrec[q].p;
        d.n_rows = R.n_rows[q].p;
        d.n_rows_pad = R.n_rows_pad[q].p;
        d.n_live = R.n_live[q].p;
        d.board_off = R.board_off[q].p;
        d.regrets = R.regrets[q].p;
        d.ssum = R.ssum[q].p;
        d.identity = 1;
    }
    a.chance_scale = R.chance_scale.p;
    a.parent_board = R.parent_board.p;
    a.parent_rbuf = k > 0 ? rd[k - 1].rbuf.p : nullptr;
    a.parent_n_boards = k > 0 ? int(rd[k - 1].n_boards) : 0;
    a.n_boards = int(R.n_boards);
    a.root_weights = root_weights[1 - trav].p;
    a.out_buf = k > 0 ? R.sbuf[trav].p : R.cbuf.p;
    a.out_scatter = k > 0 ? 1 : 0;
    a.n_segs = int(D.n_segs);
    a.segs = D.segs.p;
    a.downs = D.downs.p;
    a.ups = D.ups.p;
    a.terms = D.terms.p;
    a.prog = D.prog.p;
    a.prog_off = D.prog_off.p;
    a.l_steps = D.l_steps.p;
    a.c_steps = D.c_steps.p;
    a.hinfo = D.hinfo.p;
    a.scratch = st_scratch.p;
    a.scratch_stride = st_stride;
    a.XP = st_XP;
    a.max_rows = st_rows;
    a.vy_rows = st_vy_rows;
    a.vm_rows = st_vm_rows;
    a.max_slots = st_slots;
    a.qs = st_qs;
    a.qm = st_qm;
    a.trav = trav;
    a.HpP = int((P.H[trav] + 3) & ~3u);
    a.HoP = int((P.H[1 - trav] + 3) & ~3u);
    a.n_units = set.street_inst * D.n_segs;
    a.sample_board = (n_paths >= 0 && k > 0) ? sample_board[k].p : nullptr;
    a.prune_threshold = prune_threshold;
    const int grid = int(std::min<uint64_t>(a.n_units, uint64_t(n_sms) * st_blocks_per_sm));
    CU(launch_street_kernel(a, mode, grid, st_threads, st_smem, stream));
    return RS_OK;
}

int Engine::materialize(int trav, const uint32_t counts[3], TaskSet* out) {
    MaterializedTasks mt;
    materialize_tasks(plan, trav, counts, &mt);  // slot numbering + dependencies as first slots (plan.cpp, shared with the CPU checks)
    std::vector<NodeTask>& t = mt.tasks;
    std::vector<TaskSrc>& sr = mt.srcs;
    const uint32_t first = mt.n_tickets;
    out->phase_cut = mt.phase_cut;
    out->n_tickets = first;
    out->n_tasks = uint32_t(t.size());
    out->street_lo = out->street_hi = 0;
    out->street_inst = counts[plan.n_rounds - 1];
    if (street_on) {
        // the node tasks of the final round form one contiguous ticket range: down tasks of the last street are
        // emitted last, its up tasks first (plan.cpp: TaskGen::run)
        bool seen = false, closed = false;
        for (const NodeTask& x : t) {
            const bool fin = uint32_t(x.round_k) + 1 == plan.n_rounds;
            if (fin && closed) return set_err(RS_ERR_INVALID, "internal: final-round tasks are not contiguous");
            if (fin && !seen) {
                seen = true;
                out->street_lo = x.first;
            }
            if (fin) out->street_hi = x.first + x.count;
            if (!fin && seen) closed = true;
        }
    }
    out->runs.clear();
    out->sections.clear();
    out->xch_lo = out->xch_hi = 0;
    for (const NodeTask& x : t) {
        if (x.count == 0) continue;
        if (x.kind == TK_GATHER && plan.world > 1 && plan.shard_round >= 1 && uint32_t(x.round_k) + 1 == plan.shard_round) {
            if (out->xch_hi == out->xch_lo) out->xch_lo = x.first;
            out->xch_hi = x.first + x.count;
        }
        const int thr = round_threads[x.round_k];
        if (out->runs.empty() || out->runs.back().threads != thr) out->runs.push_back({x.first, x.first + x.count, thr});
        else out->runs.back().t1 = x.first + x.count;
        const bool up = x.kind == TK_UP_TRAV, down = x.kind == TK_DOWN;
        if (up || down) {
            bool seen = false;
            for (const TaskSet::Section& sc : out->sections) seen |= (sc.round_k == x.round_k && sc.up == up);
            if (!seen) out->sections.push_back({x.first, uint32_t(x.round_k), up});
        }
    }
    std::vector<uint32_t> tix(first);
    for (size_t j = 0; j < t.size(); ++j)
        for (uint32_t i = 0; i < t[j].count; ++i) tix[t[j].first + i] = uint32_t(j);
    CU(out->tasks.upload(t));
    CU(out->srcs.upload(sr));
    CU(out->tix.upload(tix));
    // Execution order of the final round when it is large (config 4: 2 352 river boards, ~10 GB of reach / value vectors
    // per traversal).  Task-major slots touch every board once per node task, so a board's index tables (hand records,
    // card lists, position maps: ~50 KB per player) come back from DRAM for every one of the ~500 tasks that run on it
    // (measured: DRAM traffic 2.4x the algorithmic bytes).  Instead the round is walked parent board by parent board:
    // inside one parent's group of child boards the slots stay task-major (every depth level of the group is still a
    // few thousand independent instances, enough for every CTA), the group's index tables stay in L2 for all its
    // tasks, and a reach vector is read back one level later instead of 2 352 boards later.  Producers still precede
    // consumers.  (Walking a group street segment by street segment keeps even more in L2 but starves the in-order
    // ticket dispenser: measured 3.4x slower.)
    if (!getenv("RS_TASK_MAJOR")) {
        std::vector<uint32_t> ord;
        std::string oerr;
        if (!build_execution_order(plan, trav, mt, counts, getenv("RS_BOARD_MAJOR") != nullptr, &ord, &oerr)) return set_err(RS_ERR_INVALID, oerr);
        if (!ord.empty()) CU(out->order.upload(ord));
    }
    return RS_OK;
}

void Engine::fill_args(TaskArgs* a, int trav, const TaskSet& set) const {
    const Plan& P = plan;
    memset(a, 0, sizeof(*a));
    for (int q = 0; q < 2; ++q) {
        a->H[q] = int(P.H[q]);
        a->Hpad[q] = int((P.H[q] + 3) & ~3u);
        a->root_weights[q] = root_weights[q].p;
    }
    for (uint32_t k = 0; k < P.n_rounds; ++k) {
        const RoundDev& R = rd[k];
        RoundArgs& ra = a->rounds[k];
        for (int q = 0; q < 2; ++q) {
            DevRoundPlayer& d = ra.rp[q];
            d.row_of_pos = R.row_of_pos[q].p;
            d.row_start = R.row_start[q].p;
            d.row_pos = R.row_pos[q].p;
            d.cl_pos = R.cl_pos[q].p;
            d.parent_pos = R.parent_pos[q].p;
            d.child_pos = R.child_pos[q].p;
            d.slot_of_pos = R.slot_of_pos[q].p;
            d.hrec = R.hrec[q].p;
            d.n_rows = R.n_rows[q].p;
            d.n_rows_pad = R.n_rows_pad[q].p;
            d.n_live = R.n_live[q].p;
            d.board_off = R.board_off[q].p;
            d.regrets = R.regrets[q].p;
            d.ssum = R.ssum[q].p;
            d.identity = P.loc[k][q].identity ? 1 : 0;
        }
        ra.chance_scale = R.chance_scale.p;
        ra.parent_board = R.parent_board.p;
        ra.rbuf = R.rbuf.p;
        ra.cbuf = R.cbuf.p;
        ra.sbuf = R.sbuf[trav].p;
        ra.gathered = R.gathered.p;
        ra.n_boards = int(R.n_boards);
        ra.board_base = int(P.local_lo[k]);
        if (k + 1 < P.n_rounds) {
            const bool sharded_next = (P.world > 1 && k + 1 == P.shard_round);
            ra.per_parent = sharded_next ? 0 : int(P.deal_count[k + 1]);
            ra.n_boards_next = int(rd[k + 1].n_boards);
        }
    }
    a->tasks = set.tasks.p;
    a->srcs = set.srcs.p;
    a->task_of_ticket = set.tix.p;
    a->order = set.order.n ? set.order.p : nullptr;
    a->n_tasks = set.n_tasks;
    a->flags = flags.p;
    a->ctl = ctl.p;
    a->trav = trav;
    a->HpP = a->Hpad[trav];
    a->HoP = a->Hpad[1 - trav];
    a->Hx = std::max(a->HpP, a->HoP);
    if (fused_exchange) {
        a->xch_world = P.world;
        a->xch_rank = P.rank;
        a->xch_round = int(P.shard_round);
        a->xch_leaves = int(rd[P.shard_round - 1].n_leaves);
        for (int r = 0; r < P.world; ++r) {
            a->xflag_peer[r] = reinterpret_cast<uint32_t*>(xch_peer_base[r]);
            a->xch_peer[r] = reinterpret_cast<float*>(static_cast<unsigned char*>(xch_peer_base[r]) + xch_flag_bytes);
        }
    }
    a->slots = slots;
    a->prune_threshold = prune_threshold;
    a->host_abort = abort_dev;
    a->wait_timeout_ns = wait_timeout_ms * 1000000ull;
    a->timing = timing.p;
}

int Engine::prof_begin() {
    if (!prof) return RS_OK;
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    prof_events.emplace_back(a, b);
    CU(cudaEventRecord(a, stream));
    return RS_OK;
}

int Engine::prof_end(uint32_t kind, uint32_t phase, int trav, uint32_t grid, uint64_t tb, uint64_t vb) {
    if (!prof) return RS_OK;
    CU(cudaEventRecord(prof_events.back().second, stream));
    rs_kernel_time t;
    memset(&t, 0, sizeof(t));
    t.kind = kind;
    t.phase = phase;
    t.traverser = uint32_t(trav);
    t.grid = grid;
    t.table_bytes = tb;
    t.vector_bytes = vb;
    prof->push_back(t);
    return RS_OK;
}

int Engine::enqueue_traversal(int trav, int mode, uint64_t* count, const TaskSet* set, int n_paths, int n_paths_global) {
    const Plan& P = plan;
    const TaskList& tl = P.tl[trav];
    if (!set) set = &full[trav];
    TaskArgs a;
    fill_args(&a, trav, *set);
    if (n_paths >= 0) {
        a.n_paths = n_paths;
        for (uint32_t k = 1; k < P.n_rounds; ++k) {
            a.sample_board[k] = sample_board[k].p;
            a.gather_scale[k - 1] = float(P.deal_count[k]) / float(k == 1 ? n_paths_global : 1);
        }
    }
    if (mode == KM_CFR && xs_mode) {
        // sampled opponent actions: a fresh key per traversal (a kernel argument, so these launches are never graph replays)
        uint64_t z = xs_seed + 0x9E3779B97F4A7C15ull * (++xs_count);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        a.xs_key = z ^ (z >> 31);
        a.xs_mode = xs_mode;
        mode = KM_CFR_XS;
    }
    if (rule_on() && (mode == KM_CFR || mode == KM_CFR_XS)) mode = mode == KM_CFR ? KM_CFR_DR : KM_CFR_XS_DR;
    int rc;
    // Launch schedule.  Without the street kernel a traversal is one launch of the task kernel (with the in-kernel
    // exchange) or two around the NCCL all-reduce.  With it the final round's tickets [street_lo, street_hi) are
    // replaced by one launch of the fused street kernel between the down pass of the rounds above and their up pass.
    struct Step {
        int kind;  // 0 task kernel [t0, t1), 1 street kernel, 2 all-reduce
        uint32_t t0, t1, phase;
    };
    std::vector<Step> steps;
    const bool use_street = street_on && set->street_hi > set->street_lo;
    uint32_t at = 0;
    if (use_street) {
        if (set->street_lo > 0) steps.push_back({0, 0, set->street_lo, 0});
        steps.push_back({1, 0, 0, 0});
        at = set->street_hi;
    }
    const bool split = !fused_exchange && !isolated && set->phase_cut < set->n_tickets;
    const uint32_t cut = split ? std::max(set->phase_cut, at) : set->n_tickets;
    if (cut > at) steps.push_back({0, at, cut, use_street ? 1u : 0u});
    if (split) {
        steps.push_back({2, 0, 0, 0});
        steps.push_back({0, cut, set->n_tickets, 2});
    }
    uint64_t vec = 0;
    for (uint32_t k = 0; k < P.n_rounds; ++k)
        vec += (uint64_t(tl.n_rbuf[k]) * P.H[1 - trav] + uint64_t(tl.n_cbuf[k]) * P.H[trav]) * rd[k].n_boards * 8;  // written once, read once
    for (const Step& sp : steps) {
        if ((rc = prof_begin()) != RS_OK) return rc;
        if (sp.kind == 0) {
            // one launch per run of equal block size inside [t0, t1); the longest piece keeps the step's phase label and
            // the others report as phase + 8 (bench.py's roofline reads phase 0).  Table bytes go to the piece that holds
            // the first ticket of a round's down (opponent regrets read) or up (own tables read + written) tasks.
            struct Piece {
                uint32_t t0, t1;
                int threads;
            };
            std::vector<Piece> pieces;
            for (const TaskSet::Run& r : set->runs) {
                const uint32_t lo = std::max(sp.t0, r.t0), hi = std::min(sp.t1, r.t1);
                if (lo < hi) pieces.push_back({lo, hi, r.threads});
            }
            size_t longest = 0;
            for (size_t i = 1; i < pieces.size(); ++i)
                if (pieces[i].t1 - pieces[i].t0 > pieces[longest].t1 - pieces[longest].t0) longest = i;
            for (size_t i = 0; i < pieces.size(); ++i) {
                if (i > 0 && (rc = prof_begin()) != RS_OK) return rc;
                a.t0 = pieces[i].t0;
                a.t1 = pieces[i].t1;
                a.xch_bump = (fused_exchange && set->xch_lo < set->xch_hi && a.t0 <= set->xch_lo && set->xch_lo < a.t1) ? 1 : 0;
                const int thr = pieces[i].threads;
                const bool wide = wide_for(thr, a.t1 - a.t0);
                const int grid = int(std::min<uint64_t>(uint64_t(a.t1 - a.t0), uint64_t(n_sms) * (wide ? blocks_per_sm : bps_small)));
                CU(launch_task_kernel(a, mode, grid, thr, wide, wide ? smem_bytes : smem_small, stream));
                uint64_t bytes = 0;
                for (const TaskSet::Section& sc : set->sections)
                    if (sc.first >= a.t0 && sc.first < a.t1) {
                        const uint64_t own = P.tabs[sc.round_k][trav].board_off[P.n_boards[sc.round_k]];
                        const uint64_t opp = P.tabs[sc.round_k][1 - trav].board_off[P.n_boards[sc.round_k]];
                        bytes += sc.up ? own * 16 : opp * 4;
                    }
                if ((rc = prof_end(RS_KERNEL_TRAVERSAL, sp.phase + (i == longest ? 0u : 8u), trav, uint32_t(grid), bytes, i == longest ? vec : 0)) != RS_OK)
                    return rc;
                if (i + 1 < pieces.size()) ++*count;
            }
        } else if (sp.kind == 1) {
            if ((rc = enqueue_street(trav, mode, *set, n_paths)) != RS_OK) return rc;
            const uint32_t k = P.n_rounds - 1;
            const uint64_t own = P.tabs[k][trav].board_off[P.n_boards[k]], opp = P.tabs[k][1 - trav].board_off[P.n_boards[k]];
            const uint32_t grid = uint32_t(std::min<uint64_t>(uint64_t(set->street_inst) * street[trav].n_segs, uint64_t(n_sms) * st_blocks_per_sm));
            if ((rc = prof_end(RS_KERNEL_STREET, 0, trav, grid, own * 16 + opp * 4, 0)) != RS_OK) return rc;
        } else {
            // the one exchange step of the path: counterfactual values at the shared chance nodes
            RoundDev& Par = rd[P.shard_round - 1];
            const size_t n = size_t(Par.n_leaves) * Par.n_boards * ((P.H[trav] + 3) & ~3u);
            int nrc = nccl::g_api.AllReduce(Par.gathered.p, Par.gathered.p, n, nccl::kFloat32, nccl::kSum, comm, stream);
            if (nrc != 0) return set_err(RS_ERR_NCCL, "ncclAllReduce failed");
            if ((rc = prof_end(RS_KERNEL_ALLREDUCE, 0, trav, 0, 0, n * 4)) != RS_OK) return rc;
        }
        ++*count;
    }
    return RS_OK;
}

// one iteration on sampled run-outs: sample_board[] already holds the board ids
int Engine::enqueue_sampled(int n_paths, int n_paths_global, uint64_t* count) {
    auto it = sampled_sets.find(n_paths);
    if (it == sampled_sets.end()) {
        std::unique_ptr<TaskSet[]> sets(new TaskSet[2]);
        for (int p = 0; p < 2; ++p) {
            uint32_t counts[3] = {rd[0].n_boards, uint32_t(n_paths), uint32_t(n_paths)};
            int rc = materialize(p, counts, &sets[p]);
            if (rc != RS_OK) return rc;
        }
        it = sampled_sets.emplace(n_paths, std::move(sets)).first;
    }
    for (int p = 0; p < 2; ++p) {
        int rc = enqueue_traversal(p, KM_CFR, count, &it->second[p], n_paths, n_paths_global);
        if (rc != RS_OK) return rc;
    }
    return RS_OK;
}

int Engine::enqueue_iteration(uint64_t* count) {
    // players alternate, player 0 first; player 1 sees player 0's fresh regrets (cfr.rs:216-224)
    for (int p = 0; p < 2; ++p) {
        int rc = enqueue_traversal(p, KM_CFR, count);
        if (rc != RS_OK) return rc;
    }
    return RS_OK;
}

int Engine::iterate(uint64_t n) {
    CU(cudaSetDevice(device));
    if (n == 0) return RS_OK;
    if (aborted) return set_err(RS_ERR_CUDA, "an earlier traversal was aborted: the tables are partly updated, create a new engine");
    const bool use_graph = this->use_graph && !xs_mode;  // the traversal key of the sampling mode changes with every launch
    if (use_graph && !graph_exec) {
        uint64_t cnt = 0;
        CU(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
        int rc = enqueue_iteration(&cnt);
        cudaError_t e = cudaStreamEndCapture(stream, &graph);
        if (rc != RS_OK) return rc;
        if (e != cudaSuccess) return set_err(RS_ERR_CUDA, std::string("graph capture: ") + cudaGetErrorString(e));
        CU(cudaGraphInstantiate(&graph_exec, graph, 0));
        launches_per_iter = cnt;
    }
    CU(cudaEventRecord(ev0, stream));
    for (uint64_t i = 0; i < n; ++i) {
        {
            int rc = advance_rule();
            if (rc != RS_OK) return rc;
        }
        if (use_graph) {
            CU(cudaGraphLaunch(graph_exec, stream));
            launches += launches_per_iter;
        } else {
            uint64_t cnt = 0;
            int rc = enqueue_iteration(&cnt);
            if (rc != RS_OK) return rc;
            launches += cnt;
            launches_per_iter = cnt;
        }
        ++iterations;
        {
            int rc = maybe_discount();
            if (rc != RS_OK) return rc;
        }
    }
    CU(cudaEventRecord(ev1, stream));
    CU(cudaStreamSynchronize(stream));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, ev0, ev1));
    device_ms += ms;
    return check_abort("rs_iterate");
}

// Factors {fp, fn, fs, floor} of iteration t under rule r (b200cfr.h: rs_set_update_rule): those of iteration t - 1, all 1
// for t = 1; computed in double and rounded to fp32.  x^a / (x^a + 1) is evaluated as 1 / (1 + x^-a), which stays finite
// where x^a overflows.
static void update_rule_factors(const rs_update_rule& r, uint64_t t, float f[4]) {
    f[0] = f[1] = f[2] = 1.f;
    f[3] = r.kind == RS_RULE_CFR_PLUS ? 0.f : -INFINITY;
    if (t <= 1) return;
    const double s = double(t - 1);
    if (r.kind == RS_RULE_DCFR || r.kind == RS_RULE_LCFR) {
        const bool lin = r.kind == RS_RULE_LCFR;
        const double a = lin ? 1.0 : double(r.alpha), b = lin ? 1.0 : double(r.beta), g = lin ? 1.0 : double(r.gamma);
        f[0] = float(1.0 / (1.0 + std::pow(s, -a)));
        f[1] = float(1.0 / (1.0 + std::pow(s, -b)));
        f[2] = float(std::pow(s / double(t), g));
    } else if (r.kind == RS_RULE_CFR_PLUS) {
        f[2] = float(s / double(t));
    }
}

// before every rs_iterate iteration: the factors of the next t go to TaskCtl::rule on the stream (outside the graph)
int Engine::advance_rule() {
    if (!rule_on()) return RS_OK;
    float f[4];
    update_rule_factors(rule, ++rule_t, f);
    CU(launch_set_rule(ctl.p, f, stream));
    ++launches;
    return RS_OK;
}

// monitor thread of train() (cfr.rs:243-262): when the iteration count crosses into a new period p = t / DISCOUNT_INTERVAL
// (and t has not passed the cap) every table is scaled by d = p / (p + 1).  Shared by rs_iterate and rs_iterate_sampled.
int Engine::maybe_discount() {
    if (!discount_interval) return RS_OK;
    const uint64_t period = iterations / discount_interval;
    if (period == last_discount_period) return RS_OK;
    last_discount_period = period;
    if (discount_cap && iterations > discount_cap) return RS_OK;
    const float pf = float(period);
    const float d = pf / (pf + 1.0f);
    for (uint32_t k = 0; k < plan.n_rounds; ++k)
        for (int q = 0; q < 2; ++q) {
            CU(launch_scale(rd[k].regrets[q].p, rd[k].regrets[q].n, d, stream));
            CU(launch_scale(rd[k].ssum[q].p, rd[k].ssum[q].n, d, stream));
            launches += 2;
        }
    return RS_OK;
}

// After a synchronised launch sequence: did a waiter inside the kernel give up (rs_abort, or a wait longer than the bound:
// a peer rank that never launched, a rank-asymmetric call of a collective entry point)?  Only engines that can wait on
// something outside their own stream pay for the read-back: the in-kernel exchange, or a raised abort word.
int Engine::check_abort(const char* what) {
    if (!fused_exchange && !(abort_host && *abort_host)) return RS_OK;
    TaskCtl c;
    CU(cudaMemcpy(&c, ctl.p, sizeof(c), cudaMemcpyDeviceToHost));
    if (!c.abort) return RS_OK;
    aborted = true;
    return set_err(RS_ERR_CUDA, std::string(what) + ": the traversal kernel gave up waiting (" +
                                    ((abort_host && *abort_host) ? "rs_abort was called" : "a wait exceeded the bound of " + std::to_string(wait_timeout_ms) +
                                                                                               " ms: a peer rank did not launch the same traversal") +
                                    "); the tables are partly updated, create a new engine");
}

// root counterfactual values of `player` by hand slot, [root boards][H]
// root counterfactual values by hand slot straight into `dst` (n_boards * H floats): the permutation from the board-local
// order runs on the device, the copy goes through a pinned staging buffer
int Engine::root_values_into(int player, float* dst) {
    const Plan& P = plan;
    const RoundDev& R = rd[0];
    const uint32_t hp = (P.H[player] + 3) & ~3u, H = P.H[player];
    const size_t n = size_t(R.n_boards) * H;
    if (root_out.n < n) CU(root_out.alloc(n));
    if (root_stage_n < n) {
        if (root_stage) cudaFreeHost(root_stage);
        root_stage = nullptr;
        CU(cudaHostAlloc(reinterpret_cast<void**>(&root_stage), n * sizeof(float), cudaHostAllocDefault));
        root_stage_n = n;
    }
    CU(cudaMemsetAsync(root_out.p, 0, n * sizeof(float), stream));
    CU(launch_unpermute(R.cbuf.p + size_t(P.tl[player].root_cbuf) * R.n_boards * hp, R.slot_of_pos[player].p, R.n_live[player].p, root_out.p,
                        R.n_boards, hp, H, stream));
    CU(cudaMemcpyAsync(root_stage, root_out.p, n * sizeof(float), cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    memcpy(dst, root_stage, n * sizeof(float));
    return RS_OK;
}

int Engine::root_values(int player, std::vector<float>* out) {
    out->assign(size_t(rd[0].n_boards) * plan.H[player], 0.f);
    return root_values_into(player, out->data());
}

int Engine::root_sum(int player, double* out) {
    std::vector<float> v;
    int rc = root_values(player, &v);
    if (rc != RS_OK) return rc;
    double s = 0;
    for (float x : v) s += x;
    *out = s;
    return RS_OK;
}

}  // namespace rs

// =================================================================================================
// C ABI
// =================================================================================================
using namespace rs;

struct rs_engine {
    Engine e;
};
struct rs_plan {
    Plan p;
};

extern "C" {

const char* rs_last_error(void) { return g_last_error.c_str(); }
int rs_version(void) { return 100; }

int rs_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int rs_nccl_unique_id(uint8_t* out) {
    if (!out) return set_err(RS_ERR_INVALID, "null output");
    std::string err;
    if (!nccl::load(&err)) return set_err(RS_ERR_NCCL, err);
    nccl::UniqueId id;
    int rc = nccl::g_api.GetUniqueId(&id);
    if (rc != 0) return set_err(RS_ERR_NCCL, "ncclGetUniqueId failed");
    memcpy(out, &id, RS_NCCL_ID_BYTES);
    return RS_OK;
}

static int abstraction_args_ok(const void* a, const void* b, uint32_t dim, uint32_t dist_kind) {
    if (!a || !b) return set_err(RS_ERR_INVALID, "null argument");
    if (dim == 0 || dim > ABS_MAX_BINS) return set_err(RS_ERR_INVALID, "histograms have 1..128 bins");
    if (dist_kind != RS_DIST_EMD_1D && dist_kind != RS_DIST_L2) return set_err(RS_ERR_INVALID, "unknown distance");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return set_err(RS_ERR_CUDA, "no CUDA device available (no CPU fallback)");
    return RS_OK;
}

int rs_kmeans_assign(const float* points, size_t n, uint32_t dim, const float* centers, uint32_t k, uint32_t dist_kind,
                     uint32_t* cluster, float* min_dist, double* inertia, float* kernel_ms) {
    int rc = abstraction_args_ok(points, centers, dim, dist_kind);
    if (rc != RS_OK) return rc;
    if (!cluster) return set_err(RS_ERR_INVALID, "null argument");
    if (k == 0) return set_err(RS_ERR_INVALID, "no centres");
    std::string err;
    if (!gpu_kmeans_assign(points, n, dim, centers, k, dist_kind, cluster, min_dist, inertia, kernel_ms, &err)) return set_err(RS_ERR_CUDA, err);
    return RS_OK;
}

int rs_kmeans_fit_regular(const float* points, size_t n, uint32_t dim, float* centers, uint32_t k, uint32_t dist_kind, uint32_t rounds,
                          uint32_t* cluster, float* inertia) {
    int rc = abstraction_args_ok(points, centers, dim, dist_kind);
    if (rc != RS_OK) return rc;
    if (!cluster) return set_err(RS_ERR_INVALID, "null argument");
    if (k < 2) return set_err(RS_ERR_INVALID, "fit_regular needs at least two centres (kmeans.rs:547-548 reads center_movement[1])");
    std::string err;
    if (!gpu_kmeans_fit_regular(points, n, dim, centers, k, dist_kind, rounds, cluster, inertia, &err)) return set_err(RS_ERR_CUDA, err);
    return RS_OK;
}

int rs_kmeans_fit_growbatch(const float* points, size_t n, uint32_t dim, float* centers, uint32_t k, uint32_t dist_kind, uint32_t initial_batch_size,
                            uint64_t seed, uint32_t* batch_index_out, uint32_t* cluster_out, float* stats_out) {
    int rc = abstraction_args_ok(points, centers, dim, dist_kind);
    if (rc != RS_OK) return rc;
    if (k < 2) return set_err(RS_ERR_INVALID, "fit_growbatch needs at least two centres (kmeans.rs:423-424 reads center_movements[1])");
    if (initial_batch_size == 0 || size_t(initial_batch_size) > n)
        return set_err(RS_ERR_INVALID, "need 1 <= initial_batch_size <= n (the reference indexes shuffled_data[0 .. batch))");
    std::string err;
    if (!gpu_kmeans_fit_growbatch(points, n, dim, centers, k, dist_kind, initial_batch_size, seed, batch_index_out, cluster_out, stats_out, &err))
        return set_err(RS_ERR_CUDA, err);
    return RS_OK;
}

int rs_generate_histograms(uint32_t round, uint64_t first_index, size_t count, uint32_t samples, uint32_t bins, uint64_t seed, float* out,
                           uint8_t* cards_out, float* kernel_ms) {
    if (!out) return set_err(RS_ERR_INVALID, "null argument");
    if (round > 3) return set_err(RS_ERR_INVALID, "round must be 0 (preflop) .. 3 (river)");
    if (samples == 0 || bins == 0 || bins > HIST_MAX_BINS) return set_err(RS_ERR_INVALID, "need samples >= 1 and 1 <= bins <= 128");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return set_err(RS_ERR_CUDA, "no CUDA device available (no CPU fallback)");
    // EHS::new()'s indexers (ehs.rs:26-31): [2] for the preflop, [2, 3 / 4 / 5] afterwards; hands of the LAST round
    static const uint8_t board_cards[4] = {0, 3, 4, 5};
    HandIndexer ix;
    const bool ok = round == 0 ? ix.init(1, {2}) : ix.init(2, {2, board_cards[round]});
    if (!ok) return set_err(RS_ERR_INVALID, "hand indexer init failed");
    const int ir = round == 0 ? 0 : 1;
    const uint64_t size = ix.size(ir);
    if (first_index > size || count > size - first_index) return set_err(RS_ERR_INVALID, "index range exceeds the round size " + std::to_string(size));
    const uint32_t n_known = 2 + board_cards[round];
    std::vector<uint8_t> cards(count * 7, 0);
    for (size_t i = 0; i < count; ++i)
        if (!ix.get_hand(ir, first_index + i, &cards[i * 7])) return set_err(RS_ERR_INVALID, "hand un-index failed");
    if (cards_out) memcpy(cards_out, cards.data(), cards.size());
    std::string err;
    if (!gpu_generate_histograms(cards.data(), n_known, first_index, count, samples, bins, seed, out, kernel_ms, &err)) return set_err(RS_ERR_CUDA, err);
    return RS_OK;
}

int rs_histogram_distances(const float* p, const float* q, size_t n, uint32_t dim, uint32_t dist_kind, float* out) {
    int rc = abstraction_args_ok(p, q, dim, dist_kind);
    if (rc != RS_OK) return rc;
    if (!out) return set_err(RS_ERR_INVALID, "null argument");
    std::string err;
    if (!gpu_pair_dist(p, q, false, n, dim, dist_kind, out, nullptr, &err)) return set_err(RS_ERR_CUDA, err);
    return RS_OK;
}

int rs_kmeans_update_min_dists(const float* points, size_t n, uint32_t dim, const float* new_center, uint32_t dist_kind, float* min_dists) {
    int rc = abstraction_args_ok(points, new_center, dim, dist_kind);
    if (rc != RS_OK) return rc;
    if (!min_dists) return set_err(RS_ERR_INVALID, "null argument");
    std::string err;
    if (!gpu_pair_dist(points, new_center, true, n, dim, dist_kind, nullptr, min_dists, &err)) return set_err(RS_ERR_CUDA, err);
    return RS_OK;
}

int rs_kmeans_init_pp(const float* points, size_t n, uint32_t dim, uint32_t k, uint32_t dist_kind, uint64_t seed, uint32_t* chosen_out,
                      float* centers_out) {
    int rc = abstraction_args_ok(points, points, dim, dist_kind);
    if (rc != RS_OK) return rc;
    if (!chosen_out || k == 0 || n == 0 || k > n) return set_err(RS_ERR_INVALID, "need 1 <= k <= n and an output buffer");
    std::string err;
    if (!gpu_kmeans_init_pp(points, n, dim, k, dist_kind, seed, chosen_out, &err)) return set_err(RS_ERR_CUDA, err);
    if (centers_out)
        for (uint32_t c = 0; c < k; ++c) memcpy(centers_out + size_t(c) * dim, points + size_t(chosen_out[c]) * dim, dim * sizeof(float));
    return RS_OK;
}

int rs_kmeans_init_random(const float* points, size_t n, uint32_t dim, uint32_t k, uint32_t n_restarts, uint32_t dist_kind, uint64_t seed,
                          uint32_t* chosen_out, float* centers_out) {
    int rc = abstraction_args_ok(points, points, dim, dist_kind);
    if (rc != RS_OK) return rc;
    if (!chosen_out || k < 2 || n == 0 || k > n || n_restarts == 0) return set_err(RS_ERR_INVALID, "need 2 <= k <= n, n_restarts >= 1 and an output buffer");
    std::string err;
    if (!gpu_kmeans_init_random(points, n, dim, k, n_restarts, dist_kind, seed, chosen_out, &err)) return set_err(RS_ERR_CUDA, err);
    if (centers_out)
        for (uint32_t c = 0; c < k; ++c) memcpy(centers_out + size_t(c) * dim, points + size_t(chosen_out[c]) * dim, dim * sizeof(float));
    return RS_OK;
}

int rs_gpu_index_hands(uint32_t n_board_cards, const uint8_t* cards, size_t n, uint64_t* out, float* kernel_ms) {
    if (!cards || !out) return set_err(RS_ERR_INVALID, "null argument");
    if (n_board_cards < 3 || n_board_cards > 5) return set_err(RS_ERR_INVALID, "n_board_cards must be 3, 4 or 5");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return set_err(RS_ERR_CUDA, "no CUDA device available (no CPU fallback)");
    HandIndexer ix;
    if (!ix.init(2, {2, uint8_t(n_board_cards)})) return set_err(RS_ERR_INVALID, "hand indexer init failed");
    std::string err;
    if (!gpu_index_hands(ix, 1, cards, n, out, kernel_ms, &err)) return set_err(RS_ERR_CUDA, err);
    return RS_OK;
}

int rs_abort(rs_engine* e) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    if (e->e.abort_host) *e->e.abort_host = 1u;  // plain store to mapped pinned memory: safe from any host thread while a kernel runs
    return RS_OK;
}

int rs_set_wait_timeout_ms(rs_engine* e, uint64_t ms) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    Engine& E = e->e;
    E.wait_timeout_ms = ms;
    // the bound is a kernel argument baked into the captured iteration graph: capture again on the next call
    CU(cudaSetDevice(E.device));
    CU(cudaStreamSynchronize(E.stream));
    if (E.graph_exec) {
        cudaGraphExecDestroy(E.graph_exec);
        E.graph_exec = nullptr;
    }
    if (E.graph) {
        cudaGraphDestroy(E.graph);
        E.graph = nullptr;
    }
    return RS_OK;
}

int rs_set_opponent_sampling(rs_engine* e, uint32_t mode, uint64_t seed) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    if (mode > 2) return set_err(RS_ERR_INVALID, "mode must be RS_OPP_FULL (0), RS_OPP_SAMPLE (1) or RS_OPP_SAMPLE_TIMES_SIGMA (2)");
    Engine& E = e->e;
    if (mode && E.street_on) return set_err(RS_ERR_UNSUPPORTED, "sampled opponent actions are not available with RS_FLAG_STREET_KERNEL");
    CU(cudaSetDevice(E.device));
    CU(cudaStreamSynchronize(E.stream));
    E.xs_mode = int(mode);
    E.xs_seed = seed;
    E.xs_count = 0;
    return RS_OK;
}

int rs_set_prune_threshold(rs_engine* e, float threshold) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    if (threshold != threshold) return set_err(RS_ERR_INVALID, "threshold is NaN (use -INFINITY to switch pruning off)");
    Engine& E = e->e;
    E.prune_threshold = threshold;
    // the threshold is a kernel argument baked into the captured iteration graph: capture again on the next call
    CU(cudaSetDevice(E.device));
    CU(cudaStreamSynchronize(E.stream));
    if (E.graph_exec) {
        cudaGraphExecDestroy(E.graph_exec);
        E.graph_exec = nullptr;
    }
    if (E.graph) {
        cudaGraphDestroy(E.graph);
        E.graph = nullptr;
    }
    return RS_OK;
}

int rs_exchange_export(rs_engine* e, uint8_t* out) {
    if (!e || !out) return set_err(RS_ERR_INVALID, "null argument");
    Engine& E = e->e;
    if (!E.xch.p || E.xch_vectors == 0) return set_err(RS_ERR_INVALID, "engine is not board-sharded: nothing to exchange");
    CU(cudaSetDevice(E.device));
    cudaIpcMemHandle_t h;
    static_assert(sizeof(h) == RS_EXCHANGE_HANDLE_BYTES, "IPC handle size");
    CU(cudaIpcGetMemHandle(&h, E.xch.p));
    memcpy(out, &h, sizeof(h));
    return RS_OK;
}

int rs_exchange_import(rs_engine* e, const uint8_t* handles, uint32_t n_ranks) {
    if (!e || !handles) return set_err(RS_ERR_INVALID, "null argument");
    Engine& E = e->e;
    if (!E.xch.p || E.xch_vectors == 0) return set_err(RS_ERR_INVALID, "engine is not board-sharded: nothing to exchange");
    if (int(n_ranks) != E.plan.world || n_ranks > uint32_t(RS_MAX_PEERS))
        return set_err(RS_ERR_INVALID, "rs_exchange_import needs one handle per rank (at most 8 ranks)");
    if (E.fused_exchange) return set_err(RS_ERR_INVALID, "exchange buffers already imported");
    CU(cudaSetDevice(E.device));
    CU(cudaStreamSynchronize(E.stream));
    for (uint32_t r = 0; r < n_ranks; ++r) {
        if (int(r) == E.plan.rank) {
            E.xch_peer_base[r] = E.xch.p;
            continue;
        }
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + size_t(r) * RS_EXCHANGE_HANDLE_BYTES, sizeof(h));
        void* p = nullptr;
        const cudaError_t ce = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (ce != cudaSuccess) {  // all or nothing: unmap what was mapped, the engine keeps the NCCL path
            cudaGetLastError();
            E.close_peers();
            return set_err(RS_ERR_CUDA, std::string("cudaIpcOpenMemHandle (rank ") + std::to_string(r) + "): " + cudaGetErrorString(ce));
        }
        E.xch_peer_base[r] = p;
    }
    E.fused_exchange = true;
    // the iteration graph was captured with the two-launch + all-reduce schedule: capture again on the next call
    if (E.graph_exec) {
        cudaGraphExecDestroy(E.graph_exec);
        E.graph_exec = nullptr;
    }
    if (E.graph) {
        cudaGraphDestroy(E.graph);
        E.graph = nullptr;
    }
    return RS_OK;
}

int rs_exchange_disable(rs_engine* e) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    Engine& E = e->e;
    CU(cudaSetDevice(E.device));
    CU(cudaStreamSynchronize(E.stream));
    E.close_peers();
    if (E.fused_exchange) {  // back to two launches + ncclAllReduce: the captured graph has to go
        E.fused_exchange = false;
        if (E.graph_exec) {
            cudaGraphExecDestroy(E.graph_exec);
            E.graph_exec = nullptr;
        }
        if (E.graph) {
            cudaGraphDestroy(E.graph);
            E.graph = nullptr;
        }
    }
    return RS_OK;
}

int rs_plan_create(const rs_tree* tree, const rs_ranges* ranges, const rs_abstraction* abs, const rs_config* cfg,
                   const uint64_t* board_masks, uint32_t n_subgames, rs_plan** out) {
    if (!out) return set_err(RS_ERR_INVALID, "null output");
    *out = nullptr;
    if (!cfg) return set_err(RS_ERR_INVALID, "null config");
    std::unique_ptr<rs_plan> h(new (std::nothrow) rs_plan());
    if (!h) return set_err(RS_ERR_INVALID, "out of memory");
    std::string err;
    uint64_t one = cfg->board_mask;
    try {
        if (!compile_plan(tree, ranges, abs, cfg, board_masks ? board_masks : &one, board_masks ? n_subgames : 1, &h->p, &err))
            return set_err(RS_ERR_INVALID, err);
    } catch (const std::exception& ex) {
        return set_err(RS_ERR_INVALID, std::string("plan compile failed: ") + ex.what());
    }
    *out = h.release();
    return RS_OK;
}

void rs_plan_destroy(rs_plan* p) { delete p; }

static int create_impl(const rs_tree* tree, const rs_ranges* ranges, const rs_abstraction* abs, const rs_config* cfg,
                       const uint64_t* board_masks, uint32_t n_sub, rs_engine** out) {
    if (!out) return set_err(RS_ERR_INVALID, "null output");
    *out = nullptr;
    if (!cfg) return set_err(RS_ERR_INVALID, "null config");
    std::unique_ptr<rs_engine> h(new (std::nothrow) rs_engine());
    if (!h) return set_err(RS_ERR_INVALID, "out of memory");
    std::string err;
    try {
        // card tables: the canonical hand indices come from the device indexer (bit-identical to the host one)
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) == cudaSuccess && cfg && cfg->device >= 0 && cfg->device < ndev) cudaSetDevice(cfg->device);
        if (!compile_plan(tree, ranges, abs, cfg, board_masks, n_sub, &h->e.plan, &err, ndev > 0 ? &device_batch_index : nullptr))
            return set_err(RS_ERR_INVALID, err);
        int rc = h->e.init(cfg);
        if (rc != RS_OK) return rc;
    } catch (const std::exception& ex) {
        return set_err(RS_ERR_INVALID, std::string("engine creation failed: ") + ex.what());
    }
    *out = h.release();
    return RS_OK;
}

int rs_create(const rs_tree* tree, const rs_ranges* ranges, const rs_abstraction* abs, const rs_config* cfg,
              rs_engine** out) {
    if (!cfg) return set_err(RS_ERR_INVALID, "null config");
    uint64_t one = cfg->board_mask;
    return create_impl(tree, ranges, abs, cfg, &one, 1, out);
}

int rs_create_batch(const rs_tree* tree, const rs_ranges* ranges, const rs_abstraction* abs, const rs_config* cfg,
                    const uint64_t* board_masks, uint32_t n_subgames, rs_engine** out) {
    if (!board_masks || n_subgames == 0) return set_err(RS_ERR_INVALID, "need at least one subgame board");
    return create_impl(tree, ranges, abs, cfg, board_masks, n_subgames, out);
}

void rs_destroy(rs_engine* e) {
    if (!e) return;
    cudaSetDevice(e->e.device);
    delete e;
}

int rs_iterate(rs_engine* e, uint64_t n_iters) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    return e->e.iterate(n_iters);
}

int rs_iterate_sampled(rs_engine* e, const uint8_t* dealt, uint32_t n_paths) {
    if (!e || !dealt) return set_err(RS_ERR_INVALID, "null argument");
    Engine& E = e->e;
    const Plan& P = E.plan;
    if (E.aborted) return set_err(RS_ERR_CUDA, "an earlier traversal was aborted: create a new engine");
    if (P.n_rounds < 2) return set_err(RS_ERR_INVALID, "a single-street tree has no chance node to sample");
    if (P.n_sub != 1) return set_err(RS_ERR_UNSUPPORTED, "sampled iterations need one root board");
    // a row of a board that is not sampled would miss the factors of this iteration (rs_set_update_rule)
    if (E.rule_on()) return set_err(RS_ERR_UNSUPPORTED, "rs_iterate_sampled needs RS_RULE_VANILLA: the update rules discount rows lazily");
    if (n_paths == 0 || n_paths > P.n_boards[1]) return set_err(RS_ERR_INVALID, "n_paths must be in 1..#first-street deals");
    const uint32_t L = P.n_rounds - 1;  // cards per path
    // Board-sharded engines: every rank is handed the SAME paths (the call is collective) and keeps those whose first
    // dealt card falls into its own slice of the first dealt-card level; the importance weight uses the global count.
    std::vector<int32_t> ids[3];
    std::vector<uint8_t> seen(52, 0);
    for (uint32_t s = 0; s < n_paths; ++s) {
        uint32_t id = 0;
        uint64_t mask = P.board_mask[0][0];
        int32_t path_ids[3] = {0, 0, 0};
        for (uint32_t k = 1; k <= L; ++k) {
            const int c = dealt[s * L + (k - 1)];
            if (c >= 52 || (mask & (1ull << c))) return set_err(RS_ERR_INVALID, "sampled card already on the board");
            if (k == 1) {
                if (seen[c]) return set_err(RS_ERR_INVALID, "sampled paths must start with distinct cards");
                seen[c] = 1;
            }
            id = id * P.deal_count[k] + uint32_t(__builtin_popcountll(~mask & ((1ull << c) - 1)));
            mask |= 1ull << c;
            path_ids[k] = int32_t(id);
        }
        if (uint32_t(path_ids[1]) < P.local_lo[1] || uint32_t(path_ids[1]) >= P.local_hi[1]) continue;  // another rank's
        for (uint32_t k = 1; k <= L; ++k) ids[k].push_back(path_ids[k] - int32_t(P.local_lo[k]));
    }
    const uint32_t n_local = uint32_t(ids[1].size());
    CU(cudaSetDevice(E.device));
    if (int(n_local) > E.sample_cap || E.sample_cap == 0) {
        for (uint32_t k = 1; k <= L; ++k) CU(E.sample_board[k].alloc(std::max<uint32_t>(n_local, 1)));
        E.sample_cap = int(std::max<uint32_t>(n_local, 1));
    }
    if (n_local)
        for (uint32_t k = 1; k <= L; ++k)
            CU(cudaMemcpyAsync(E.sample_board[k].p, ids[k].data(), n_local * sizeof(int32_t), cudaMemcpyHostToDevice, E.stream));
    CU(cudaEventRecord(E.ev0, E.stream));
    uint64_t cnt = 0;
    int rc = E.enqueue_sampled(int(n_local), int(n_paths), &cnt);
    if (rc != RS_OK) return rc;
    CU(cudaEventRecord(E.ev1, E.stream));
    CU(cudaStreamSynchronize(E.stream));  // ids[] are host temporaries
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, E.ev0, E.ev1));
    E.device_ms += ms;
    E.launches += cnt;
    E.iterations += 1;
    if ((rc = E.maybe_discount()) != RS_OK) return rc;
    return E.check_abort("rs_iterate_sampled");
}

/* generate_hand's board part (cfr.rs:100-122), see b200cfr.h */
int rs_sample_runouts(uint64_t seed, uint64_t board_mask, uint32_t n_cards, uint32_t n_paths, int distinct_first, uint8_t* dealt_out) {
    if (!dealt_out) return set_err(RS_ERR_INVALID, "null argument");
    const int n_board = __builtin_popcountll(board_mask);
    if (n_cards == 0 || n_board + int(n_cards) > 52) return set_err(RS_ERR_INVALID, "n_cards out of range");
    if (distinct_first && n_paths > uint32_t(52 - n_board)) return set_err(RS_ERR_INVALID, "more paths than distinct first cards");
    uint64_t state = seed;
    auto next = [&]() {  // splitmix64
        state += 0x9E3779B97F4A7C15ull;
        uint64_t z = state;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    };
    const uint64_t zone = (~0ull / 52ull) * 52ull;  // Uniform::from(0..52): reject the top of the range, exactly uniform
    auto card = [&]() {
        for (;;) {
            const uint64_t z = next();
            if (z < zone) return int(z % 52ull);
        }
    };
    uint64_t firsts = 0;
    for (uint32_t s = 0; s < n_paths; ++s) {
        uint64_t used = board_mask;
        for (uint32_t i = 0; i < n_cards;) {
            const int c = card();
            if (used & (1ull << c)) continue;                           // cfr.rs:115-121: draw again
            if (i == 0 && distinct_first && (firsts & (1ull << c))) continue;
            if (i == 0) firsts |= 1ull << c;
            used |= 1ull << c;
            dealt_out[size_t(s) * n_cards + i] = uint8_t(c);
            ++i;
        }
    }
    return RS_OK;
}

int rs_discount(rs_engine* e, float d) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    Engine& E = e->e;
    CU(cudaSetDevice(E.device));
    for (uint32_t k = 0; k < E.plan.n_rounds; ++k)
        for (int q = 0; q < 2; ++q) {
            CU(launch_scale(E.rd[k].regrets[q].p, E.rd[k].regrets[q].n, d, E.stream));
            CU(launch_scale(E.rd[k].ssum[q].p, E.rd[k].ssum[q].n, d, E.stream));
        }
    CU(cudaStreamSynchronize(E.stream));
    return RS_OK;
}

int rs_set_update_rule(rs_engine* e, const rs_update_rule* rule) {
    if (!rule) return set_err(RS_ERR_INVALID, "null rule");
    if (rule->kind > RS_RULE_CFR_PLUS)
        return set_err(RS_ERR_INVALID, "kind must be RS_RULE_VANILLA (0), RS_RULE_DCFR (1), RS_RULE_LCFR (2) or RS_RULE_CFR_PLUS (3)");
    if (!std::isfinite(rule->alpha) || !std::isfinite(rule->beta) || !std::isfinite(rule->gamma))
        return set_err(RS_ERR_INVALID, "alpha, beta and gamma must be finite");
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    Engine& E = e->e;
    if (rule->kind != RS_RULE_VANILLA && E.street_on)
        return set_err(RS_ERR_UNSUPPORTED, "update rules other than RS_RULE_VANILLA are not available with RS_FLAG_STREET_KERNEL");
    CU(cudaSetDevice(E.device));
    CU(cudaStreamSynchronize(E.stream));
    const bool was_on = E.rule_on();
    E.rule = *rule;
    E.rule_t = 0;
    // the captured iteration graph launches the builds of the old rule: capture again when that changes
    if (was_on != E.rule_on()) {
        if (E.graph_exec) {
            cudaGraphExecDestroy(E.graph_exec);
            E.graph_exec = nullptr;
        }
        if (E.graph) {
            cudaGraphDestroy(E.graph);
            E.graph = nullptr;
        }
    }
    return RS_OK;
}

int rs_get_update_rule(rs_engine* e, rs_update_rule* out, uint64_t* t_out) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    if (out) *out = e->e.rule;
    if (t_out) *t_out = e->e.rule_t;
    return RS_OK;
}

int rs_reset(rs_engine* e) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    Engine& E = e->e;
    CU(cudaSetDevice(E.device));
    for (uint32_t k = 0; k < E.plan.n_rounds; ++k)
        for (int q = 0; q < 2; ++q) {
            CU(E.rd[k].regrets[q].zero());
            CU(E.rd[k].ssum[q].zero());
        }
    E.iterations = 0;
    E.device_ms = 0;
    E.launches = 0;
    E.rule_t = 0;
    return RS_OK;
}

// locate slab (an_index, board_id): returns table pointers + shape
static int locate(const Plan& P, uint32_t an_index, uint32_t board_id, uint32_t* k_out, int* q_out, uint64_t* off,
                  uint32_t* n_rows, uint32_t* n_act) {
    if (an_index >= P.an_to_pnode.size() || P.an_to_pnode[an_index] < 0) return set_err(RS_ERR_INVALID, "unknown ActionNode.index");
    const PNode& n = P.nodes[P.an_to_pnode[an_index]];
    const uint32_t k = n.round_k;
    const int q = n.player;
    if (board_id >= P.n_boards[k]) return set_err(RS_ERR_INVALID, "board_id out of range for the node's round");
    if (board_id < P.local_lo[k] || board_id >= P.local_hi[k]) return set_err(RS_ERR_INVALID, "board is owned by another rank");
    const RoundPlayerTables& T = P.tabs[k][q];
    *k_out = k;
    *q_out = q;
    *n_rows = T.n_rows[board_id];
    *n_act = uint32_t(n.children.size());
    *off = T.board_off[board_id] + uint64_t(P.loc[k][q].n_rows_pad[board_id]) * n.cum_a;
    return RS_OK;
}

int rs_plan_infoset_offset(const rs_plan* p, uint32_t an_index, uint32_t board_id, uint64_t* offset_out,
                           uint32_t* n_rows_out, uint32_t* n_actions_out) {
    if (!p) return set_err(RS_ERR_INVALID, "null plan");
    uint32_t k, nr, na;
    int q;
    uint64_t off;
    int rc = locate(p->p, an_index, board_id, &k, &q, &off, &nr, &na);
    if (rc != RS_OK) return rc;
    if (offset_out) *offset_out = off;
    if (n_rows_out) *n_rows_out = nr;
    if (n_actions_out) *n_actions_out = na;
    return RS_OK;
}

int rs_read_infoset(rs_engine* e, uint32_t an_index, uint32_t board_id, float* regrets, float* strategy_sum,
                    size_t cap_floats, uint32_t* n_rows_out, uint32_t* n_actions_out) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    Engine& E = e->e;
    uint32_t k, nr, na;
    int q;
    uint64_t off;
    int rc = locate(E.plan, an_index, board_id, &k, &q, &off, &nr, &na);
    if (rc != RS_OK) return rc;
    if (n_rows_out) *n_rows_out = nr;
    if (n_actions_out) *n_actions_out = na;
    const size_t n = size_t(nr) * na;
    if ((regrets || strategy_sum) && cap_floats < n) return set_err(RS_ERR_CAPACITY, "output buffer too small");
    CU(cudaSetDevice(E.device));
    if (regrets) CU(cudaMemcpy(regrets, E.rd[k].regrets[q].p + off, n * sizeof(float), cudaMemcpyDeviceToHost));
    if (strategy_sum) CU(cudaMemcpy(strategy_sum, E.rd[k].ssum[q].p + off, n * sizeof(float), cudaMemcpyDeviceToHost));
    return RS_OK;
}

int rs_write_infoset(rs_engine* e, uint32_t an_index, uint32_t board_id, const float* regrets, const float* strategy_sum,
                     size_t n_floats) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    Engine& E = e->e;
    uint32_t k, nr, na;
    int q;
    uint64_t off;
    int rc = locate(E.plan, an_index, board_id, &k, &q, &off, &nr, &na);
    if (rc != RS_OK) return rc;
    const size_t n = size_t(nr) * na;
    if (n_floats != n) return set_err(RS_ERR_INVALID, "slab size mismatch");
    CU(cudaSetDevice(E.device));
    if (regrets) CU(cudaMemcpy(E.rd[k].regrets[q].p + off, regrets, n * sizeof(float), cudaMemcpyHostToDevice));
    if (strategy_sum) CU(cudaMemcpy(E.rd[k].ssum[q].p + off, strategy_sum, n * sizeof(float), cudaMemcpyHostToDevice));
    return RS_OK;
}

static int strategy_impl(rs_engine* e, uint32_t an_index, uint32_t board_id, float* out, size_t cap, uint32_t* n_rows_out,
                         uint32_t* n_actions_out, bool average) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    Engine& E = e->e;
    uint32_t k, nr, na;
    int q;
    uint64_t off;
    int rc = locate(E.plan, an_index, board_id, &k, &q, &off, &nr, &na);
    if (rc != RS_OK) return rc;
    if (n_rows_out) *n_rows_out = nr;
    if (n_actions_out) *n_actions_out = na;
    const size_t n = size_t(nr) * na;
    if (!out) return RS_OK;
    if (cap < n) return set_err(RS_ERR_CAPACITY, "output buffer too small");
    CU(cudaSetDevice(E.device));
    const float* src = (average ? E.rd[k].ssum[q].p : E.rd[k].regrets[q].p) + off;
    CU(launch_normalize(src, E.scratch.p, nr, na, E.stream));
    CU(cudaStreamSynchronize(E.stream));
    CU(cudaMemcpy(out, E.scratch.p, n * sizeof(float), cudaMemcpyDeviceToHost));
    return RS_OK;
}

int rs_average_strategy(rs_engine* e, uint32_t an_index, uint32_t board_id, float* out, size_t cap_floats,
                        uint32_t* n_rows_out, uint32_t* n_actions_out) {
    return strategy_impl(e, an_index, board_id, out, cap_floats, n_rows_out, n_actions_out, true);
}
int rs_current_strategy(rs_engine* e, uint32_t an_index, uint32_t board_id, float* out, size_t cap_floats,
                        uint32_t* n_rows_out, uint32_t* n_actions_out) {
    return strategy_impl(e, an_index, board_id, out, cap_floats, n_rows_out, n_actions_out, false);
}

// Headerless little-endian dump of the average strategy, the style of the reference's abstraction files
// (gen_abstraction/main.rs:372-380 packs u32 after u32, card_abstraction.rs:227-229 reads them back): for every action
// node in ActionNode.index order, for every board of the node's round this rank owns in board-id order, the slab
// [row][n_actions] of fp32 probabilities (Infoset::get_final_strategy, infoset.rs:104-123).
int rs_dump_average_strategy(rs_engine* e, const char* path, uint64_t* n_floats_out) {
    if (!e || !path) return set_err(RS_ERR_INVALID, "null argument");
    Engine& E = e->e;
    const Plan& P = E.plan;
    FILE* f = fopen(path, "wb");
    if (!f) return set_err(RS_ERR_INVALID, std::string("cannot open ") + path);
    uint64_t total = 0;
    std::vector<float> buf;
    int rc = RS_OK;
    for (uint32_t an = 0; an < P.an_to_pnode.size() && rc == RS_OK; ++an) {
        if (P.an_to_pnode[an] < 0) continue;
        const uint32_t k = P.nodes[P.an_to_pnode[an]].round_k;
        for (uint32_t b = P.local_lo[k]; b < P.local_hi[k]; ++b) {
            uint32_t nr = 0, na = 0;
            if ((rc = strategy_impl(e, an, b, nullptr, 0, &nr, &na, true)) != RS_OK) break;
            buf.resize(size_t(nr) * na);
            if (buf.empty()) continue;
            if ((rc = strategy_impl(e, an, b, buf.data(), buf.size(), &nr, &na, true)) != RS_OK) break;
            if (fwrite(buf.data(), sizeof(float), buf.size(), f) != buf.size()) {
                rc = set_err(RS_ERR_INVALID, std::string("short write to ") + path);
                break;
            }
            total += buf.size();
        }
    }
    fclose(f);
    if (rc == RS_OK && n_floats_out) *n_floats_out = total;
    return rc;
}

static int board_id_impl(const Plan& P, uint32_t round_idx, const uint8_t* dealt, uint32_t n_dealt, uint32_t* out) {
    if (round_idx >= P.n_rounds) return set_err(RS_ERR_INVALID, "round_idx out of range");
    if (n_dealt != round_idx) return set_err(RS_ERR_INVALID, "need exactly round_idx dealt cards");
    if (P.n_sub != 1) return set_err(RS_ERR_UNSUPPORTED, "board lookup by dealt cards needs a single root board; batch boards are their own ids");
    uint32_t id = 0;
    uint64_t mask = P.board_mask[0][0];
    for (uint32_t k = 1; k <= round_idx; ++k) {
        const int c = dealt[k - 1];
        if (c >= 52 || (mask & (1ull << c))) return set_err(RS_ERR_INVALID, "dealt card already on the board");
        const uint32_t idx = uint32_t(__builtin_popcountll(~mask & ((1ull << c) - 1)));
        id = id * P.deal_count[k] + idx;
        mask |= 1ull << c;
    }
    *out = id;
    return RS_OK;
}

int rs_plan_board_id(const rs_plan* p, uint32_t round_idx, const uint8_t* dealt, uint32_t n_dealt, uint32_t* board_id_out) {
    if (!p || !board_id_out) return set_err(RS_ERR_INVALID, "null argument");
    return board_id_impl(p->p, round_idx, dealt, n_dealt, board_id_out);
}
int rs_board_id(rs_engine* e, uint32_t round_idx, const uint8_t* dealt, uint32_t n_dealt, uint32_t* board_id_out) {
    if (!e || !board_id_out) return set_err(RS_ERR_INVALID, "null argument");
    return board_id_impl(e->e.plan, round_idx, dealt, n_dealt, board_id_out);
}

static int card_table_impl(const Plan& P, uint32_t round_idx, uint32_t player, uint32_t board_id, uint16_t* rows_out,
                           size_t cap, uint32_t* n_rows_out) {
    if (round_idx >= P.n_rounds || player > 1) return set_err(RS_ERR_INVALID, "round/player out of range");
    if (board_id >= P.n_boards[round_idx]) return set_err(RS_ERR_INVALID, "board_id out of range");
    if (board_id < P.local_lo[round_idx] || board_id >= P.local_hi[round_idx])
        return set_err(RS_ERR_INVALID, "board is owned by another rank");
    const RoundPlayerTables& T = P.tabs[round_idx][player];
    const uint32_t H = P.H[player];
    if (n_rows_out) *n_rows_out = T.n_rows[board_id];
    if (rows_out) {
        if (cap < H) return set_err(RS_ERR_CAPACITY, "output buffer too small");
        memcpy(rows_out, &T.row_of_hand[size_t(board_id) * H], H * sizeof(uint16_t));
    }
    return RS_OK;
}
int rs_plan_card_table(const rs_plan* p, uint32_t round_idx, uint32_t player, uint32_t board_id, uint16_t* rows_out,
                       size_t cap, uint32_t* n_rows_out) {
    if (!p) return set_err(RS_ERR_INVALID, "null plan");
    return card_table_impl(p->p, round_idx, player, board_id, rows_out, cap, n_rows_out);
}
int rs_card_table(rs_engine* e, uint32_t round_idx, uint32_t player, uint32_t board_id, uint16_t* rows_out, size_t cap,
                  uint32_t* n_rows_out) {
    if (!e) return set_err(RS_ERR_INVALID, "null engine");
    return card_table_impl(e->e.plan, round_idx, player, board_id, rows_out, cap, n_rows_out);
}

int rs_plan_showdown_order(const rs_plan* p, uint32_t player, uint32_t board_id, uint16_t* order_out, uint32_t* class_out,
                           size_t cap, uint32_t* n_live_out) {
    if (!p || player > 1) return set_err(RS_ERR_INVALID, "bad argument");
    const Plan& P = p->p;
    const uint32_t k = P.n_rounds - 1;
    const ShowdownTables& S = P.sd[player];
    if (S.n_live.empty()) return set_err(RS_ERR_INVALID, "tree has no showdown terminals");
    if (board_id >= P.n_boards[k]) return set_err(RS_ERR_INVALID, "board_id out of range");
    const uint32_t H = P.H[player];
    const uint32_t nl = S.n_live[board_id];
    if (n_live_out) *n_live_out = nl;
    if (cap < nl) return set_err(RS_ERR_CAPACITY, "output buffer too small");
    for (uint32_t i = 0; i < nl; ++i) {
        if (order_out) order_out[i] = S.sorted[size_t(board_id) * H + i];
        if (class_out) class_out[i] = S.cls[size_t(board_id) * H + i];
    }
    return RS_OK;
}

int rs_plan_local_tables(const rs_plan* p, uint32_t round_idx, uint32_t player, uint32_t board_id, uint32_t* hrec_words_out, uint16_t* cl_pos_out,
                         uint16_t* slot_of_pos_out, uint32_t dims_out[2]) {
    if (!p || player > 1 || !dims_out) return set_err(RS_ERR_INVALID, "bad argument");
    const Plan& P = p->p;
    if (round_idx >= P.n_rounds || board_id >= P.n_boards[round_idx]) return set_err(RS_ERR_INVALID, "round or board out of range");
    if (board_id < P.local_lo[round_idx] || board_id >= P.local_hi[round_idx]) return set_err(RS_ERR_INVALID, "board belongs to another rank");
    const LocalTables& L = P.loc[round_idx][player];
    dims_out[0] = L.Hpad;
    dims_out[1] = L.n_live[board_id];
    if (hrec_words_out) memcpy(hrec_words_out, &L.hrec[size_t(board_id) * L.Hpad], size_t(L.Hpad) * sizeof(HandRec));
    if (cl_pos_out) memcpy(cl_pos_out, &L.cl_pos[size_t(board_id) * 2 * L.Hpad], size_t(2) * L.Hpad * sizeof(uint16_t));
    if (slot_of_pos_out) memcpy(slot_of_pos_out, &L.slot_of_pos[size_t(board_id) * L.Hpad], size_t(L.Hpad) * sizeof(uint16_t));
    return RS_OK;
}

int rs_plan_check_execution_order(const rs_plan* p, uint32_t traverser, int force_board_major, uint32_t* n_tickets_out, uint32_t* n_moved_out) {
    if (!p || traverser > 1) return set_err(RS_ERR_INVALID, "bad argument");
    const Plan& P = p->p;
    uint32_t counts[3] = {0, 0, 0};
    for (uint32_t k = 0; k < P.n_rounds; ++k) counts[k] = P.boards_local(k);
    MaterializedTasks mt;
    materialize_tasks(P, int(traverser), counts, &mt);
    std::vector<uint32_t> ord;
    std::string err;
    if (!build_execution_order(P, int(traverser), mt, counts, force_board_major > 0, &ord, &err)) return set_err(RS_ERR_INVALID, err);
    if (force_board_major < 0) {  // self-test of the checker: tickets in REVERSE slot order must be rejected
        ord.resize(mt.n_tickets);
        for (uint32_t i = 0; i < mt.n_tickets; ++i) ord[i] = mt.n_tickets - 1 - i;
    }
    err = check_execution_order(P, int(traverser), mt, counts, ord);
    if (!err.empty()) return set_err(RS_ERR_INVALID, "execution order: " + err);
    if (n_tickets_out) *n_tickets_out = mt.n_tickets;
    if (n_moved_out) {
        uint32_t moved = 0;
        for (uint32_t i = 0; i < ord.size(); ++i) moved += ord[i] != i;
        *n_moved_out = moved;
    }
    return RS_OK;
}

int rs_plan_street_info(const rs_plan* p, uint32_t traverser, uint32_t out[8]) {
    if (!p || !out || traverser > 1) return set_err(RS_ERR_INVALID, "bad argument");
    const StreetPlan& S = p->p.street[traverser];
    out[0] = S.eligible ? 1u : 0u;
    out[1] = uint32_t(S.segs.size());
    out[2] = S.max_rows;
    out[3] = S.max_slots;
    out[4] = S.max_q_sd;
    out[5] = S.max_q_mo;
    out[6] = uint32_t(S.downs.size());
    out[7] = uint32_t(S.ups.size());
    if (!S.eligible) g_last_error = S.why;
    return RS_OK;
}

int rs_plan_street_program(const rs_plan* p, uint32_t traverser, uint32_t board_id, uint32_t* words_out, size_t cap,
                           uint32_t* n_words_out, uint32_t* hinfo_out, size_t hinfo_cap, uint32_t dims_out[4]) {
    if (!p || !n_words_out || !dims_out || traverser > 1) return set_err(RS_ERR_INVALID, "bad argument");
    const Plan& P = p->p;
    const StreetPlan& S = P.street[traverser];
    if (!S.eligible) return set_err(RS_ERR_INVALID, "the final round does not run on the street kernel: " + S.why);
    const uint32_t k = P.n_rounds - 1;
    if (board_id < P.local_lo[k] || board_id >= P.local_hi[k]) return set_err(RS_ERR_INVALID, "board is owned by another rank");
    const uint32_t lb = board_id - P.local_lo[k];
    const uint32_t n = S.prog_off[lb + 1] - S.prog_off[lb];
    const uint32_t HpP = P.loc[k][traverser].Hpad;
    *n_words_out = n;
    dims_out[0] = S.l_steps[lb];
    dims_out[1] = S.c_steps[lb];
    dims_out[2] = HpP;
    dims_out[3] = P.loc[k][1 - traverser].Hpad;
    if (words_out) {
        if (cap < n) return set_err(RS_ERR_CAPACITY, "output buffer too small");
        memcpy(words_out, S.prog.data() + S.prog_off[lb], size_t(n) * sizeof(uint32_t));
    }
    if (hinfo_out) {
        if (hinfo_cap < 2 * size_t(HpP)) return set_err(RS_ERR_CAPACITY, "hinfo buffer too small");
        memcpy(hinfo_out, S.hinfo.data() + size_t(lb) * HpP * 2, size_t(HpP) * 2 * sizeof(uint32_t));
    }
    return RS_OK;
}

static int score_impl(rs_engine* e, int mode, double out[2]) {
    if (!e || !out) return set_err(RS_ERR_INVALID, "null argument");
    Engine& E = e->e;
    if (E.aborted) return set_err(RS_ERR_CUDA, "an earlier traversal was aborted: create a new engine");
    CU(cudaSetDevice(E.device));
    for (int p = 0; p < 2; ++p) {
        uint64_t cnt = 0;
        int rc = E.enqueue_traversal(p, mode, &cnt);
        if (rc != RS_OK) return rc;
        CU(cudaStreamSynchronize(E.stream));
        if ((rc = E.check_abort(mode == KM_BR ? "rs_best_response" : "rs_average_value")) != RS_OK) return rc;
        double s = 0;
        rc = E.root_sum(p, &s);
        if (rc != RS_OK) return rc;
        // with subgame batches every rank owns different root boards: the caller sums over ranks
        out[p] = s;
    }
    return RS_OK;
}

int rs_best_response(rs_engine* e, double out[2]) { return score_impl(e, KM_BR, out); }
int rs_average_value(rs_engine* e, double out[2]) { return score_impl(e, KM_EVAL, out); }

int rs_root_values(rs_engine* e, uint32_t player, float* out, size_t cap) {
    if (!e || !out || player > 1) return set_err(RS_ERR_INVALID, "bad argument");
    Engine& E = e->e;
    const size_t n = size_t(E.rd[0].n_boards) * E.plan.H[player];
    if (cap < n) return set_err(RS_ERR_CAPACITY, "output buffer too small");
    CU(cudaSetDevice(E.device));
    return E.root_values_into(int(player), out);
}

int rs_set_range_weights(rs_engine* e, uint32_t player, const float* weights, size_t n) {
    if (!e || !weights || player > 1) return set_err(RS_ERR_INVALID, "bad argument");
    Engine& E = e->e;
    if (n != E.plan.H[player]) return set_err(RS_ERR_INVALID, "weights length must equal the range size");
    CU(cudaSetDevice(E.device));
    CU(cudaMemcpyAsync(E.root_weights[player].p, weights, n * sizeof(float), cudaMemcpyHostToDevice, E.stream));
    return RS_OK;
}

int rs_profile_iteration(rs_engine* e, rs_kernel_time* out, size_t cap, uint32_t* n_out) {
    if (!e || !n_out) return set_err(RS_ERR_INVALID, "null argument");
    Engine& E = e->e;
    CU(cudaSetDevice(E.device));
    std::vector<rs_kernel_time> rec;
    int rc = E.advance_rule();
    if (rc != RS_OK) return rc;
    E.prof = &rec;
    uint64_t cnt = 0;
    rc = E.enqueue_iteration(&cnt);
    E.prof = nullptr;
    cudaError_t se = cudaStreamSynchronize(E.stream);
    for (size_t i = 0; i < E.prof_events.size(); ++i) {
        if (rc == RS_OK && se == cudaSuccess && i < rec.size())
            cudaEventElapsedTime(&rec[i].ms, E.prof_events[i].first, E.prof_events[i].second);
        cudaEventDestroy(E.prof_events[i].first);
        cudaEventDestroy(E.prof_events[i].second);
    }
    E.prof_events.clear();
    if (rc != RS_OK) return rc;
    if (se != cudaSuccess) return set_err(RS_ERR_CUDA, cudaGetErrorString(se));
    E.iterations += 1;
    E.launches += cnt;
    *n_out = uint32_t(rec.size());
    if (out) {
        if (cap < rec.size()) return set_err(RS_ERR_CAPACITY, "output buffer too small");
        memcpy(out, rec.data(), rec.size() * sizeof(rs_kernel_time));
    }
    return RS_OK;
}

int rs_debug_task_timing(rs_engine* e, unsigned long long* out32, int reset) {
    if (!e || !out32) return set_err(RS_ERR_INVALID, "null argument");
    Engine& E = e->e;
    CU(cudaSetDevice(E.device));
    CU(cudaStreamSynchronize(E.stream));
    CU(cudaMemcpy(out32, E.timing.p, 96 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    if (reset) {
        std::vector<unsigned long long> init(96, 0);
        for (int i = 0; i < 32; ++i) init[32 + 2 * i] = ~0ull;  // min-start slots
        CU(cudaMemcpy(E.timing.p, init.data(), 96 * sizeof(unsigned long long), cudaMemcpyHostToDevice));
    }
    return RS_OK;
}

static void fill_stats(const Plan& P, rs_stats* s) {
    memset(s, 0, sizeof(*s));
    s->updates_per_iteration = P.updates_per_iter_local;
    s->updates_per_iteration_global = P.updates_per_iter_global;
    s->n_rounds = P.n_rounds;
    for (uint32_t k = 0; k < P.n_rounds; ++k) {
        s->n_boards[k] = P.n_boards[k];
        s->n_boards_local[k] = P.local_hi[k] - P.local_lo[k];
    }
    s->n_hands[0] = P.H[0];
    s->n_hands[1] = P.H[1];
    s->n_combos = P.n_combos.empty() ? 0 : P.n_combos[0];
}

int rs_plan_stats(const rs_plan* p, rs_stats* out) {
    if (!p || !out) return set_err(RS_ERR_INVALID, "null argument");
    fill_stats(p->p, out);
    return RS_OK;
}

int rs_stats_get(rs_engine* e, rs_stats* out) {
    if (!e || !out) return set_err(RS_ERR_INVALID, "null argument");
    fill_stats(e->e.plan, out);
    out->iterations = e->e.iterations;
    out->device_ms = e->e.device_ms;
    out->kernel_launches = e->e.launches;
    out->table_bytes = e->e.table_bytes;
    out->updates_per_iteration_global = e->e.updates_global;
    return RS_OK;
}

}  // extern "C"
