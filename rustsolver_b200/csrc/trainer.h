// Host-side mirror of the reference's trainer surface, in C++ because no Rust toolchain exists
// in this environment.  It is what src/solver/cfr.rs would look like once its hot path is
// delegated to the C ABI in include/b200cfr.h (see INTEGRATION.md for the Rust version):
//
//   MCCFRTrainer::init(Options)      cfr.rs:159-184   -> build tree + abstraction, rs_create
//   MCCFRTrainer::train(iterations)  cfr.rs:188-297   -> rs_iterate
//   Infoset::get_strategy            infoset.rs:83    -> get_strategy(an_index, board, cluster)
//   Infoset::get_final_strategy      infoset.rs:104   -> get_final_strategy(...)
//   MCCFRTrainer::calc_br            cfr.rs:629-638   -> calc_br()
#pragma once
#include <string>
#include <vector>

#include "../../include/b200cfr.h"
#include "game.h"

namespace rs {

// flattened Tree<GameTreeNode> in the layout rs_tree points into
struct FlatTree {
    std::vector<uint8_t> type, player, round_idx, ttype, last_to_act, round;
    std::vector<int32_t> parent;
    std::vector<uint32_t> child_offset, children, an_index, value;
    std::vector<uint8_t> action_kind;   // per child edge
    std::vector<double> action_amount;  // per child edge
    rs_tree view() const;
};
FlatTree flatten_tree(const Tree& t);

enum class CardAbstractionKind { NONE = RS_ABS_NONE, ISOMORPHIC = RS_ABS_ISOMORPHIC, EMD = RS_ABS_CLUSTER_ARR, OCHS = RS_ABS_CLUSTER_ARR };

struct TrainerConfig {
    int device = 0;
    int rank = 0, world_size = 1;
    uint8_t nccl_id[RS_NCCL_ID_BYTES] = {0};
    uint32_t flags = 0;
    uint64_t discount_interval = 0, discount_cap = 0;
    // update rule of the table update (rs_set_update_rule); RS_RULE_VANILLA is train()'s plain CFR
    rs_update_rule update_rule = {RS_RULE_VANILLA, 1.5f, 0.f, 2.f};
    // card_abs vector of MCCFRTrainer::init (cfr.rs:167-172): one entry per betting round
    std::vector<uint32_t> abs_kind;
    std::vector<std::vector<uint32_t>> cluster_arr;  // per round, for EMD / OCHS
};

class MCCFRTrainer {
public:
    ~MCCFRTrainer();
    // returns nullptr and sets *err where the reference would panic
    static MCCFRTrainer* init(const Options& options, const TrainerConfig& cfg, std::string* err);
    bool train(size_t iterations, std::string* err);
    // strategies of one infoset row; board_id 0 for the root street
    std::vector<float> get_strategy(size_t an_index, size_t board_id, size_t cluster_idx, std::string* err);
    std::vector<float> get_final_strategy(size_t an_index, size_t board_id, size_t cluster_idx, std::string* err);
    std::vector<double> calc_br(std::string* err);
    rs_engine* engine() { return engine_; }
    const Tree& game_tree() const { return tree_; }
    const std::vector<HandRange>& hand_ranges() const { return ranges_; }

private:
    rs_engine* engine_ = nullptr;
    Tree tree_;
    std::vector<HandRange> ranges_;
    uint64_t initial_board_mask_ = 0;
};

// load a headerless little-endian u32 array (round_N_{emd,ochs}.dat, card_abstraction.rs:227-229)
bool load_cluster_file(const std::string& path, std::vector<uint32_t>* out, std::string* err);

}  // namespace rs
