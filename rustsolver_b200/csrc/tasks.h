// Task graph of one CFR traversal, shared by the host plan compiler and the device kernel.
//
// A traversal of the public tree (SURVEY.md App. C) is cut into node-tasks; each node-task is
// instantiated once per board of its round, and one CTA executes one instance.  Instances are
// numbered in a topological order ("tickets"); a persistent kernel hands tickets out with one
// atomic counter and instances wait on their producers through per-instance flags.
//
//   TK_DOWN        opponent action node: sigma from the opponent's table, reach of every child
//                  (cfr.rs:582-586); terminal children are valued on the spot (cfr.rs:523-558) and
//                  summed into the node's terminal partial value
//   TK_UP_OPP      opponent action node: value = terminal partial + sum of child values
//   TK_UP_TRAV     traverser action node: child values, node value, regret and strategy-sum update
//                  (cfr.rs:588, 612-621)
//   TK_GATHER      chance node: sum of the child-street root values over the dealt cards
//                  (cfr.rs:502-522)
//   TK_ROOT_SHOWDOWN / TK_CHANCE_DOWN / TK_CHANCE_UP   street roots created by the all-in run-out
//                  expansion (a bare showdown, or a pass-through chance node)
//   TK_TRAV_TERMS  traverser action node of a CHAIN round (a round with one or two boards, where the traversal is
//                  a chain of dependent tasks): the part of TK_UP_TRAV that only needs the opponent reach -- the
//                  scan and the per-hand mass / showdown terms -- runs as its own task during the down pass and
//                  leaves two vectors for the TK_UP_TRAV task, which is then short.  On chain rounds opponent nodes
//                  are split the same way: one TK_DOWN task writes the child reach (what the next level waits
//                  for), a second one values the terminal children.
#pragma once
#include <cstdint>

namespace rs {

enum TaskKind : uint8_t {
    TK_DOWN = 0,
    TK_UP_OPP = 1,
    TK_UP_TRAV = 2,
    TK_GATHER = 3,
    TK_ROOT_SHOWDOWN = 4,
    TK_CHANCE_DOWN = 5,
    TK_CHANCE_UP = 6,
    TK_TRAV_TERMS = 7
};
enum ChildKind : uint8_t {
    CK_ACTION = 0,    // TK_DOWN: non-terminal child, buf = reach buffer written for it
    CK_FOLD = 1,      // terminal, coef = +-pot
    CK_SHOWDOWN = 2,  // terminal, coef = pot
    CK_CHANCE = 3,    // TK_DOWN: chance child, buf = reach buffer the next street reads
    CK_VALUE = 4      // TK_UP_*: child value = sum of the task's sources [src_first, src_first + n_src)
};
enum DepKind : uint8_t { DK_NONE = 0, DK_SAME_BOARD = 1, DK_PARENT_BOARD = 2, DK_CHILD_BOARDS = 3 };
enum SrcKind : uint8_t { SK_CBUF = 0, SK_GATHERED = 1 };

constexpr int32_t RIN_INITIAL = -1;  // reach source = the opponent's range weights (root round)
constexpr int MAX_TASK_CHILDREN = 8;
constexpr int MAX_TASK_DEPS = 4;
constexpr int MAX_TERMINAL_CHILDREN = 3;  // terminal children of one opponent node staged in shared memory

struct TaskSrc {  // one value vector feeding a child value, with the task that produces it
    int32_t buf;  // value buffer id (SK_CBUF) or chance-leaf id (SK_GATHERED) of the task's round
    int32_t dep;  // producer: node-task index in the plan, first ticket of that task once uploaded; -1 = none
    uint8_t kind; // SrcKind
    uint8_t pad[3];
};

struct TaskChild {
    uint8_t kind;        // ChildKind
    uint8_t n_src;       // CK_VALUE
    uint16_t src_first;  // CK_VALUE: index into the traverser's TaskSrc array
    int32_t buf;         // TK_DOWN: reach buffer written for this child
    float coef;          // +-pot of a terminal child (cfr.rs:525-556)
};

struct NodeTask {
    uint8_t kind;     // TaskKind
    uint8_t round_k;  // round_idx of the node
    uint8_t n_act;
    uint8_t n_dep;
    uint8_t rin_parent_round;  // 1: r_in names a reach buffer of the PARENT round, read at the parent board
    uint8_t root_scatter;      // street root (round >= 1): the value is stored in the PARENT board's hand order
    uint16_t n_src_all;        // sources of all children, contiguous from src_all_first (waited on together)
    int32_t r_in;     // reach buffer id, or RIN_INITIAL
    uint32_t cum_a;   // slab offset = n_rows_pad(board) * cum_a inside the (round, player) table
    int32_t out;      // TK_DOWN: terminal-partial value buffer (-1: none); TK_UP_*, roots: value buffer; TK_GATHER: leaf id
    int32_t aux;      // TK_UP_OPP: terminal-partial buffer to add (-1 none); TK_GATHER: value buffer of the child street's root;
                      // TK_CHANCE_DOWN: reach buffer written; TK_CHANCE_UP: leaf id read
    uint32_t first;   // ticket of instance 0
    uint32_t count;   // instances = local boards of round_k
    uint32_t an_index;
    uint32_t src_all_first;
    int32_t dep[MAX_TASK_DEPS];      // producers: node-task index in the plan, first ticket once uploaded
    uint8_t dep_kind[MAX_TASK_DEPS]; // DepKind
    TaskChild child[MAX_TASK_CHILDREN];
    uint32_t pre_terms;  // TK_UP_TRAV: 1 = mass and showdown terms come from value buffers aux, aux + 1 (TK_TRAV_TERMS)
    uint32_t seg;        // street segment of the node inside its round (plan.h: Segment); gathers: the child segment
};
static_assert(sizeof(NodeTask) == 8 + 4 * 8 + 4 * MAX_TASK_DEPS + MAX_TASK_DEPS + 12 * MAX_TASK_CHILDREN + 8, "NodeTask layout");
static_assert(sizeof(NodeTask) % 4 == 0, "NodeTask is copied to shared memory as words");

// Per-hand record of the traverser on one board (16 bytes = four words, one 128-bit load), local hand order.  Every field
// is a ready-made BYTE offset into one of the scan's shared-memory arrays, so that a gather costs one mask or shift:
//   w0 = lo4 | hi4 << 16      P[lo], P[hi]: #opponent live hands strictly weaker / weaker-or-equal, x 4 (final round only)
//   w1 = a0  | b0  << 16      GB[s0 + dlo0], GB[s0 + dhi0] x 4: inside the opponent's list of card c0, the entries weaker /
//                             weaker-or-equal than the hand (final round; 0 = GB[0] = 0 when that list is empty)
//   w2 = a1  | b1  << 16      the same for card c1
//   w3 = k0 | k1 << 9 | same4 << 18
//        k0, k1  (9 bits)     ordinal of card c0 / c1 among the opponent's NON-EMPTY card lists, x 4: B[k] and B[k + 1]
//                             are the list's start and end prefix sums; HREC_K_NONE when the opponent holds no hand
//                             with that card (B[54] = B[55] = 0)
//        same4   (14 bits)    position of the identical combo in the opponent's order x 4, HREC_SAME_NONE if there is none
struct HandRec {
    uint32_t w0, w1, w2, w3;
};
static_assert(sizeof(HandRec) == 16, "HandRec is one 128-bit load");
constexpr uint32_t HREC_K_NONE = 54u * 4u;
constexpr uint32_t HREC_SAME_NONE = 0x3FFFu;
// The opponent's per-card lists (cl_pos, u16 entries, eight per thread):
//   bits 0-10   position of the hand in the opponent's order, CL_POS_NONE = padding
//   bits 11-13  entries 8t and 8t + 1 only: the low / high three bits of the number of lists that START before entry 8t
//               (thread t's first boundary ordinal); thread 0 stores the number of non-empty lists J there instead
//   bit 15      first entry of a (non-empty) card list: the scan stores its exclusive prefix as boundary B[ordinal]
constexpr uint32_t CL_POS_MASK = 0x7FFu, CL_POS_NONE = 0x7FFu, CL_FIRST = 0x8000u;

struct TaskCtl {  // device-resident dispatcher state, reset by the last CTA to leave
    unsigned long long ticket;
    unsigned int exited;
    unsigned int epoch;
    unsigned int abort;  // set by the first waiter that gives up (host abort word or bounded wait): every CTA leaves
    unsigned int xch_seq;  // number of the next EXCHANGING launch (board-sharded traversals): the value the exchange flags carry and
                           // the parity of the exchange buffer.  Counts the same on every rank however a traversal is cut into launches
    // Update-rule factors of the current iteration (rs_set_update_rule): {fp, fn, fs, floor}, floor = 0 (CFR+) or -inf.
    // Only the KM_CFR_DR builds read them.  Graph replay fixes kernel arguments, so they live here, next to the state the
    // kernel already reaches through TaskArgs::ctl; the engine rewrites them on its stream before every iteration.
    alignas(16) float rule[4];
};

}  // namespace rs
