// Device side of the B200 CFR engine (sm_100a): a persistent dataflow kernel over the task graph
// of one traversal (tasks.h).  One CTA executes one (node-task, board) instance at a time; each
// thread owns FOUR consecutive hands of the board-local hand order, so every vector and table
// access is a 128-bit load/store.  Instances exchange opponent-reach and counterfactual-value
// vectors through L2-resident global buffers and order themselves with release/acquire flags, so
// every SM stays busy on independent boards/nodes and a whole traversal is ONE launch.
//
// Restates, in vector form (SURVEY.md App. C):
//   regret matching                Infoset::get_strategy          src/solver/infoset.rs:83-102
//   average strategy               Infoset::get_final_strategy    src/solver/infoset.rs:104-123
//   opponent reach propagation     cfr.rs:582-586
//   fold / showdown payoffs        cfr.rs:523-558
//   node value + table updates     cfr.rs:588, 612-621
//   chance scatter / gather        cfr.rs:502-522
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "plan.h"
#include "tasks.h"

namespace rs {

constexpr int MAX_ACTIONS = MAX_TASK_CHILDREN;
constexpr int RS_MAX_PEERS = 8;        // GPUs of one NVSwitch box
constexpr int FAST_ACTIONS = 4;        // nodes up to this many actions keep their table rows in registers
constexpr int MAX_TASK_THREADS = 352;  // ceil(1326 / 4) rounded up to a warp multiple

// KM_CFR_XS: CFR with per-hand sampled opponent actions.  KM_CFR_DR / KM_CFR_XS_DR: the same with the update rule of
// rs_set_update_rule (factors in TaskCtl::rule); the plain CFR builds carry no trace of it.
enum KernelMode { KM_CFR = 0, KM_BR = 1, KM_EVAL = 2, KM_CFR_XS = 3, KM_CFR_DR = 4, KM_CFR_XS_DR = 5 };

// Uniform number in [0, 1) of the sampled-opponent-action mode (rs_set_opponent_sampling): a counter-based hash of the
// traversal key, the action node, the GLOBAL board id and the opponent's hand slot, so that the draw does not depend
// on the board-local hand order, the sharding or the launch schedule.  24 bits: exact in fp32 and fp64.
__host__ __device__ inline float xs_uniform(unsigned long long key, uint32_t an_index, uint32_t board, uint32_t slot) {
    unsigned long long z = key ^ ((unsigned long long)an_index << 44) ^ ((unsigned long long)board << 20) ^ (unsigned long long)slot;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    return float(uint32_t(z >> 40)) * (1.0f / 16777216.0f);
}

struct DevRoundPlayer {  // round k, player q; every array is indexed [board][...] in board-local hand order
    const uint16_t* row_of_pos;   // [nb][Hpad]
    const uint16_t* row_start;    // [nb][Hpad+4]
    const uint16_t* row_pos;      // [nb][Hpad]
    const uint16_t* cl_pos;       // [nb][2*Hpad]  per-card lists (q as opponent)
    const uint16_t* parent_pos;   // [nb][Hpad]
    const uint16_t* child_pos;    // [nb][Hpad(parent)]
    const uint16_t* slot_of_pos;  // [nb][Hpad]  (round 0: initial range weights are given by hand slot)
    const HandRec* hrec;          // [nb][Hpad]  (q as traverser)
    const uint32_t* n_rows;       // [nb]
    const uint32_t* n_rows_pad;   // [nb]
    const uint32_t* n_live;       // [nb]
    const uint64_t* board_off;    // [nb]
    float* regrets;
    float* ssum;
    int identity;
    int pad;
};

struct RoundArgs {
    DevRoundPlayer rp[2];
    const float* chance_scale;    // [nb]
    const int32_t* parent_board;  // [nb] local id in the parent round
    float* rbuf;                  // [n_rbuf][nb][Hpad_opp]   opponent reach per buffer id
    float* cbuf;                  // [n_cbuf][nb][Hpad_trav]  counterfactual values per buffer id
    float* sbuf;                  // [n_sbuf][nb][Hpad_trav]  street-root values in the PARENT board's hand order (this traverser's pool)
    float* gathered;              // [n_leaves][nb][Hpad_trav]
    int n_boards;
    int per_parent;  // boards of the NEXT round per board of this one (0: every local next-round board hangs off board 0)
    int n_boards_next;
    int board_base;  // global id of local board 0 (board-sharded engines): only the sampled-opponent-action hash needs it
};

struct TaskArgs {
    RoundArgs rounds[3];
    const NodeTask* tasks;
    const TaskSrc* srcs;
    const uint32_t* task_of_ticket;  // [n_tickets] node-task index of every instance slot
    // Execution order.  Instances are identified by their SLOT = first slot of the node task + instance (flags, the
    // dependency fields and task_of_ticket go by slot); the dispatcher hands out TICKETS 0, 1, 2, ... and runs slot
    // order[ticket].  order is a permutation inside every launch's range [t0, t1) and a topological order of the
    // dependencies (null = identity: slots in task-major order).  The engine uses it to walk a round with thousands of
    // boards parent board by parent board and street segment by street segment, so that a board's index tables and
    // the vectors one task hands to the next are still in L2 when they are read again (engine.cu: materialize).
    const uint32_t* order;
    uint32_t n_tasks;
    uint32_t* flags;  // [n_tickets] epoch of completion
    TaskCtl* ctl;
    const float* root_weights[2];
    int H[2], Hpad[2];
    int trav;
    int HpP, HoP, Hx;  // padded range sizes of the traverser / the opponent / the larger: scalar kernel parameters are
                       // constant-bank operands, no registers and no indexed parameter loads in the kernel
    uint32_t t0, t1;  // ticket range of this launch
    // sampled-board mode (rs_iterate_sampled): rounds >= 1 only run on n_paths sampled run-outs.  Instance i of a
    // round-k task works on board sample_board[k][i]; the chance gather sums the sampled children only and
    // multiplies by gather_scale[k] = (#possible deals) / (#sampled children) (importance weight of uniform sampling)
    const int32_t* sample_board[3];  // null = every board (full traversal)
    int n_paths;
    float gather_scale[3];
    int slots;        // Hx-sized scratch vectors provisioned in shared memory
    float prune_threshold;  // traverser actions with regret <= this keep their regret (cfr.rs:352,379-386); -inf = off
    // In-kernel exchange of the chance-node partial sums between the GPUs of a board-sharded traversal (peer memory
    // over NVLink, engine.cu: rs_exchange_import).  xch_world <= 1: not used (single GPU, or the NCCL path).
    // Layout of every rank's buffer: [parity][leaf][parent board][rank][Hpad] floats and one flag per vector.
    float* xch_peer[RS_MAX_PEERS];
    uint32_t* xflag_peer[RS_MAX_PEERS];
    int xch_world, xch_rank;
    int xch_round;    // the sharded round: the gathers of round xch_round - 1 exchange their sums
    int xch_leaves;   // chance leaves of round xch_round - 1
    // Sampled opponent actions (KM_CFR_XS, cfr.rs:466-475 for every hand at once): at an opponent node each opponent hand
    // draws ONE action from its current strategy and keeps its whole reach on that child (xs_mode 1, unbiased external
    // sampling) or its reach times the probability of the drawn action (xs_mode 2, what the reference's code does).
    unsigned long long xs_key;  // key of this traversal
    int xs_mode;
    int xch_bump;     // this launch holds the exchanging gathers: the last CTA to leave advances ctl->xch_seq
    // Waits inside the kernel (producer flags, peer flags of the exchange) are bounded: a waiter gives up when the host
    // raised *host_abort (mapped pinned memory, rs_abort) or when one wait lasted longer than wait_timeout_ns (0: no
    // bound); it sets ctl->abort and every CTA leaves.  The host then reports RS_ERR_CUDA instead of hanging.
    const volatile uint32_t* host_abort;
    unsigned long long wait_timeout_ns;
    unsigned long long* timing;  // RS_TASK_TIMING builds: [8 kinds][count, wait cycles, body cycles, total cycles]
};

// dynamic shared memory of one CTA of the wide (352-thread) or the 288-thread build: the fixed arrays follow the build
size_t task_kernel_smem_bytes(bool wide, int slots, int Hp_pad, int Ho_pad);
// Two register specialisations of the kernel: blocks of up to 288 compute threads built for three resident CTAs per SM
// (64 registers), and a wide one (up to 352 threads, two CTAs per SM, 80 registers).  `wide` selects the second one for a
// block that would fit the first: a launch with too few tickets to populate a third CTA per SM is latency-bound and runs
// faster with the registers.
cudaError_t configure_task_kernels(size_t smem, int threads, bool wide, int* blocks_per_sm);
cudaError_t launch_task_kernel(const TaskArgs& a, int mode, int grid, int threads, bool wide, size_t smem, cudaStream_t st);

cudaError_t launch_scale(float* data, size_t n, float d, cudaStream_t st);
// ctl->rule = f: one thread, the factors travel as a kernel argument so that no host buffer must outlive the call
cudaError_t launch_set_rule(TaskCtl* ctl, const float f[4], cudaStream_t st);
// out[row][a] = regret-matched strategy of in[row][0..A)
cudaError_t launch_normalize(const float* in, float* out, uint32_t n_rows, uint32_t A, cudaStream_t st);
// out[board][hand slot] = in[board][position] for the live positions of every board (out must be zeroed): root values
// from the board-local hand order back to the caller's hand order
cudaError_t launch_unpermute(const float* in, const uint16_t* slot_of_pos, const uint32_t* n_live, float* out, uint32_t n_boards, uint32_t hp,
                             uint32_t H, cudaStream_t st);

}  // namespace rs
