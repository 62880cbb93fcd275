#include "trainer.h"

#include <cstdio>
#include <cstring>
#include <memory>

#include "hand_indexer.h"

namespace rs {

rs_tree FlatTree::view() const {
    rs_tree t;
    t.n_nodes = uint32_t(type.size());
    t.type = type.data();
    t.parent = parent.data();
    t.child_offset = child_offset.data();
    t.children = children.data();
    t.player = player.data();
    t.an_index = an_index.data();
    t.round_idx = round_idx.data();
    t.value = value.data();
    t.ttype = ttype.data();
    t.last_to_act = last_to_act.data();
    return t;
}

FlatTree flatten_tree(const Tree& t) {
    FlatTree f;
    const size_t n = t.nodes.size();
    f.type.resize(n);
    f.player.assign(n, 0);
    f.round_idx.assign(n, 0);
    f.ttype.assign(n, 0);
    f.last_to_act.assign(n, 0);
    f.round.assign(n, 0);
    f.parent.resize(n);
    f.an_index.assign(n, 0);
    f.value.assign(n, 0);
    f.child_offset.assign(n + 1, 0);
    for (size_t i = 0; i < n; ++i) {
        const TreeNode& nd = t.nodes[i];
        f.type[i] = uint8_t(nd.type);
        f.parent[i] = int32_t(nd.parent);
        f.player[i] = nd.player;
        f.round_idx[i] = nd.round_idx;
        f.ttype[i] = uint8_t(nd.ttype);
        f.last_to_act[i] = nd.last_to_act;
        f.round[i] = uint8_t(nd.round);
        f.an_index[i] = uint32_t(nd.index);
        f.value[i] = nd.value;
        f.child_offset[i] = uint32_t(f.children.size());
        for (size_t c = 0; c < nd.children.size(); ++c) {
            f.children.push_back(uint32_t(nd.children[c]));
            if (nd.type == NodeType::Action) {
                f.action_kind.push_back(uint8_t(nd.actions[c].kind));
                f.action_amount.push_back(nd.actions[c].amount);
            } else {
                f.action_kind.push_back(0xFF);
                f.action_amount.push_back(0.0);
            }
        }
    }
    f.child_offset[n] = uint32_t(f.children.size());
    return f;
}

bool load_cluster_file(const std::string& path, std::vector<uint32_t>* out, std::string* err) {
    FILE* f = std::fopen(path.c_str(), "rb");
    if (!f) {
        if (err) *err = "cannot open " + path;  // card_abstraction.rs:227 unwrap()
        return false;
    }
    std::fseek(f, 0, SEEK_END);
    long sz = std::ftell(f);
    std::fseek(f, 0, SEEK_SET);
    out->resize(size_t(sz) / 4);
    size_t got = std::fread(out->data(), 4, out->size(), f);
    std::fclose(f);
    if (got != out->size()) {
        if (err) *err = "short read on " + path;
        return false;
    }
    // file is little-endian u32 (bytepack LEUnpacker); so is every host this runs on
    return true;
}

MCCFRTrainer::~MCCFRTrainer() {
    if (engine_) rs_destroy(engine_);
}

MCCFRTrainer* MCCFRTrainer::init(const Options& options, const TrainerConfig& cfg, std::string* err) {
    std::unique_ptr<MCCFRTrainer> t(new MCCFRTrainer());
    t->ranges_ = options.hand_ranges;
    if (t->ranges_.size() != 2) {
        if (err) *err = "need two hand ranges";
        return nullptr;
    }
    remove_invalid_combos(t->ranges_, options.board_mask);  // cfr.rs:163
    size_t n_actions = 0;
    if (!build_game_tree(options, &n_actions, &t->tree_, err)) return nullptr;  // cfr.rs:165
    t->initial_board_mask_ = options.board_mask;

    FlatTree flat = flatten_tree(t->tree_);
    rs_tree tv = flat.view();
    rs_ranges rr;
    std::vector<uint8_t> hb[2];
    for (int q = 0; q < 2; ++q) {
        for (const HoleCards& h : t->ranges_[q].hands) {
            hb[q].push_back(h.c0);
            hb[q].push_back(h.c1);
        }
        rr.n_hands[q] = uint32_t(t->ranges_[q].hands.size());
        rr.hands[q] = hb[q].data();
    }
    rs_abstraction ab;
    std::memset(&ab, 0, sizeof(ab));
    ab.n_rounds = uint32_t(cfg.abs_kind.size() > 3 ? 3 : cfg.abs_kind.size());
    for (uint32_t k = 0; k < ab.n_rounds; ++k) {
        ab.rounds[k].kind = cfg.abs_kind[k];
        if (cfg.abs_kind[k] == RS_ABS_CLUSTER_ARR) {
            if (k >= cfg.cluster_arr.size()) {
                if (err) *err = "missing cluster_arr for round";
                return nullptr;
            }
            ab.rounds[k].cluster_arr = cfg.cluster_arr[k].data();
            ab.rounds[k].cluster_arr_len = cfg.cluster_arr[k].size();
        }
    }
    rs_config rc;
    std::memset(&rc, 0, sizeof(rc));
    rc.board_mask = options.board_mask;
    rc.device = cfg.device;
    rc.rank = cfg.rank;
    rc.world_size = cfg.world_size;
    std::memcpy(rc.nccl_id, cfg.nccl_id, RS_NCCL_ID_BYTES);
    rc.flags = cfg.flags;
    rc.discount_interval = cfg.discount_interval;
    rc.discount_cap = cfg.discount_cap;
    if (rs_create(&tv, &rr, &ab, &rc, &t->engine_) != RS_OK) {
        if (err) *err = rs_last_error();
        return nullptr;
    }
    if (cfg.update_rule.kind != RS_RULE_VANILLA && rs_set_update_rule(t->engine_, &cfg.update_rule) != RS_OK) {
        if (err) *err = rs_last_error();
        return nullptr;
    }
    return t.release();
}

bool MCCFRTrainer::train(size_t iterations, std::string* err) {
    if (rs_iterate(engine_, iterations) != RS_OK) {
        if (err) *err = rs_last_error();
        return false;
    }
    return true;
}

static std::vector<float> strategy_row(rs_engine* e, size_t an, size_t board, size_t cluster, bool avg, std::string* err) {
    uint32_t nr = 0, na = 0;
    int rc = avg ? rs_average_strategy(e, uint32_t(an), uint32_t(board), nullptr, 0, &nr, &na)
                 : rs_current_strategy(e, uint32_t(an), uint32_t(board), nullptr, 0, &nr, &na);
    if (rc != RS_OK || cluster >= nr) {
        if (err) *err = rc != RS_OK ? rs_last_error() : "cluster_idx out of range";
        return {};
    }
    std::vector<float> all(size_t(nr) * na);
    rc = avg ? rs_average_strategy(e, uint32_t(an), uint32_t(board), all.data(), all.size(), &nr, &na)
             : rs_current_strategy(e, uint32_t(an), uint32_t(board), all.data(), all.size(), &nr, &na);
    if (rc != RS_OK) {
        if (err) *err = rs_last_error();
        return {};
    }
    return std::vector<float>(all.begin() + cluster * na, all.begin() + (cluster + 1) * na);
}

std::vector<float> MCCFRTrainer::get_strategy(size_t an_index, size_t board_id, size_t cluster_idx, std::string* err) {
    return strategy_row(engine_, an_index, board_id, cluster_idx, false, err);
}
std::vector<float> MCCFRTrainer::get_final_strategy(size_t an_index, size_t board_id, size_t cluster_idx, std::string* err) {
    return strategy_row(engine_, an_index, board_id, cluster_idx, true, err);
}

std::vector<double> MCCFRTrainer::calc_br(std::string* err) {
    double out[2] = {0, 0};
    if (rs_best_response(engine_, out) != RS_OK) {
        if (err) *err = rs_last_error();
        return {};
    }
    return {out[0], out[1]};
}

}  // namespace rs
