// launchers.cpp -- TEST INFRASTRUCTURE: host restatements of every kernel launcher declared in csrc/kernels.cuh, so that
// csrc/engine.cu (the engine's HOST logic) can be linked and run without a GPU (see hostsim/cuda_runtime.h for the why).
//
// Each function below does, sequentially and in the plainest way, what the kernel behind the real launcher is SPECIFIED to do
// (DESIGN.md 3.x / 4.2, and the comment at the kernel) on the very data layouts the engine builds: the class-sorted node table, the
// HRW2 blob, the 16-byte directory slots, the bounded-load arrays.  They share csrc/spec.cuh and csrc/trie_table.hpp with the product
// (the same scalar functions the kernels use) but none of the kernels' structure -- no groups, no tiles, no staging.  A test that
// passes here says the engine's host side hands the right tables, flags, counters and round decisions to the device; what the
// KERNELS compute is proven on the GPU box against the oracle, never here.
#include <sched.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "../../../rio_rs_b200/csrc/kernels.cuh"
#include "../../../rio_rs_b200/csrc/spec.cuh"
#include "../../../rio_rs_b200/csrc/trie_table.hpp"

namespace rio {

namespace {

inline void count(const Launch &L) { if (L.launch_counter) ++*L.launch_counter; }

// ---- flat weighted rendezvous over the class-sorted table (DESIGN.md 3.4): lexicographic min of (E(u) * r, ~u, node index) ----
uint32_t hrw_over_table(uint64_t key, const NodeTabDev &tab) {
    const ObjHash o = obj_hash(key);
    uint64_t best_sc = 0;
    uint32_t best_u = 0, best_i = kNone;
    for (uint32_t c = 0; c < tab.n_classes; c++) {
        const uint32_t invw = tab.classes[c].invw;
        for (uint32_t q = tab.classes[c].start; q < tab.classes[c + 1].start; q++) {
            const NodeRec &r = tab.recs[q];
            const uint32_t u = pair_hash(o, r.s0, r.s1, r.s2);
            const uint64_t sc = (uint64_t)elog(u) * invw;
            if (best_i == kNone || cand_better(sc, u, r.nidx, best_sc, best_u, best_i)) { best_sc = sc; best_u = u; best_i = r.nidx; }
        }
    }
    return best_i;
}

const ContestRec *levels() {
    static const std::vector<ContestRec> v = trie_level_constants(16);
    return v.data();
}
uint32_t walk(uint64_t key, const TrieDev &t) { return trie_walk_host(reinterpret_cast<const uint32_t *>(t.blob), t.bits, levels(), obj_hash(key)); }

// The counter exchange of a pass over the ranks' windows (DESIGN.md 6; csrc/bounded_tail.cuh): window = slots[2][world][max_nodes]
// then flags[world].  My counters go into slot [epoch & 1][rank] of EVERY rank's window, then my flag in every window takes the epoch
// (release); I wait until every flag of MY window carries it (acquire) and sum my window's slots.  In this build the "peers" are other
// handles of the same process (the stand-in IPC handle is the pointer itself), each driven by its own thread.
void exchange(const uint32_t *local, uint32_t *const *win, uint32_t rank, uint32_t world, uint32_t M, uint32_t max_nodes, uint32_t epoch, uint32_t *out) {
    const size_t slot_words = (size_t)2 * world * max_nodes, par = (size_t)(epoch & 1u) * world * max_nodes;
    for (uint32_t p = 0; p < world; p++) memcpy(win[p] + par + (size_t)rank * max_nodes, local, (size_t)M * 4);
    for (uint32_t p = 0; p < world; p++) __atomic_store_n(win[p] + slot_words + rank, epoch, __ATOMIC_RELEASE);
    for (uint32_t r = 0; r < world; r++)
        while ((int32_t)(__atomic_load_n(win[rank] + slot_words + r, __ATOMIC_ACQUIRE) - epoch) < 0) sched_yield();
    for (uint32_t j = 0; j < M; j++) {
        uint32_t sum = 0;
        for (uint32_t r = 0; r < world; r++) sum += win[rank][par + (size_t)r * max_nodes + j];
        out[j] = sum;
    }
}

// the tail of a bounded-load pass (DESIGN.md 3.5 / 6; csrc/bounded_tail.cuh): exchange (world > 1), then the capacity check on the
// GLOBAL counters
void capacity_check(const BoundedTail &b, const uint32_t *local) {
    uint32_t any = 0, open = 0;
    if (b.world > 1) {
        exchange(local, b.peers.win, b.rank, b.world, b.M, b.max_nodes, b.xchg_epoch, b.glob);
        local = b.glob;
    }
    for (uint32_t j = 0; j < b.M; j++) {
        const uint32_t c = local[j], cp = b.cap[j], ce = b.closed_epoch[j];
        const bool live = b.state[j] & kNodeLive;
        const bool ov = live && c > cp;
        if (local != b.glob) b.glob[j] = c;
        b.over[j] = ov;
        b.thr[j] = ov ? (uint32_t)((((unsigned long long)(c - cp)) << 32) / c) : 0u;
        if (ov) b.closed_epoch[j] = b.call_epoch;
        any |= ov;
        open += live && !ov && ce != b.call_epoch;
        if (b.next_zero) b.next_zero[j] = 0;
    }
    uint32_t *f = const_cast<uint32_t *>(b.host_flags);
    f[0] = any; f[1] = open; f[3] = 0;
    f[2] = b.flag_seq;
}

// ---- directory (DESIGN.md 4.2) ----
inline unsigned long long norm_key(uint64_t k) { return k == kEmptyKey ? kEmptyKey - 1 : k; }
inline uint64_t home_slot(unsigned long long key, const DirDev &d) { return (key * kGolden64) >> d.shift; }
inline uint32_t node_of(const DirSlot &s) { return (uint32_t)s.val; }
inline void set_node(DirSlot &s, uint32_t node) { s.val = (s.val & 0xFFFFFFFF00000000ull) | node; }   // the sequence half stays

}  // namespace

// ---- solver ------------------------------------------------------------------------------------------------------------
uint64_t assign_wave_objects(int sm_count) { return (uint64_t)sm_count * 3 * 256 * 5; }
uint64_t trie_wave_objects(int sm_count) { return (uint64_t)sm_count * 5 * 256 * 4; }
void trie_upload_level_constants(int) {}

void launch_assign_hrw(const Launch &L, const uint64_t *keys, uint64_t n, const NodeTabDev &tab, uint32_t *out, uint32_t *counters, const uint32_t *sel, uint64_t n_sel) {
    const uint64_t n_work = sel ? n_sel : n;
    if (!n_work) return;
    for (uint64_t q = 0; q < n_work; q++) {
        const uint64_t i = sel ? sel[q] : q;
        const uint32_t j = hrw_over_table(keys[i], tab);
        out[i] = j;
        if (counters && j != kNone) counters[j]++;
    }
    count(L);
}

void launch_assign_trie(const Launch &L, const uint64_t *keys, uint64_t n, const TrieDev &t, uint32_t *out, uint32_t *counters, const uint32_t *sel, uint64_t n_sel, uint32_t,
                        const BoundedTail *tail) {
    const uint64_t n_work = sel ? n_sel : n;
    if (!n_work) return;
    for (uint64_t q = 0; q < n_work; q++) {
        const uint64_t i = sel ? sel[q] : q;
        const uint32_t j = walk(keys[i], t);
        out[i] = j;
        if (counters && j != kNone) counters[j]++;
    }
    if (!sel && tail && tail->enabled) capacity_check(*tail, counters);   // the fused tail: same pass, same launch
    count(L);
}

void launch_reassign_trie(const Launch &L, const uint64_t *keys, uint64_t n, const TrieDev &t, uint32_t *idx, uint32_t *counters, uint32_t, unsigned long long *moved) {
    if (!n) return;
    for (uint64_t i = 0; i < n; i++) {
        const uint32_t j = walk(keys[i], t);
        if (j != idx[i]) { idx[i] = j; ++*moved; }
        if (counters && j != kNone) counters[j]++;
    }
    count(L);
}

void launch_dir_reassign_trie(const Launch &L, const DirDev &dir, const TrieDev &t, unsigned long long *moved) {
    for (uint64_t i = 0; i <= dir.mask; i++) {
        DirSlot &s = dir.slots[i];
        if (s.key == kEmptyKey || node_of(s) == kNone) continue;
        const uint32_t j = walk(s.key, t);
        if (j != node_of(s)) { set_node(s, j); ++*moved; }
    }
    count(L);
}

void launch_assign_affinity(const Launch &L, const float *fobj, uint64_t n, const float *fnode, const uint32_t *live, uint32_t n_total, uint32_t K, uint32_t *out, float *out_cost,
                            uint32_t *counters) {
    if (!n) return;
    for (uint64_t i = 0; i < n; i++) {
        float best = 0.f;
        uint32_t bj = kNone;
        for (uint32_t j = 0; j < n_total; j++) {
            if (!live[j]) continue;
            float acc = 0.f;
            for (uint32_t k = 0; k < K; k++) acc = std::fmaf(fobj[i * K + k], fnode[(size_t)j * K + k], acc);   // the kernels' FFMA chain
            const float cost = -acc;
            if (bj == kNone || cost < best) { best = cost; bj = j; }   // ties -> lowest j
        }
        out[i] = bj;
        if (out_cost) out_cost[i] = best;
        if (counters && bj != kNone) counters[bj]++;
    }
    count(L);
}
uint32_t affinity_umma_max_nodes() { return 0; }                  // no tensor cores here: the engine takes its CUDA-core branch
void affinity_umma_set_timing_buffer(unsigned long long *) {}
bool launch_assign_affinity_umma(const Launch &, const float *, uint64_t, const float *, const float *, const uint32_t *, uint32_t, uint32_t, uint32_t, uint32_t *, float *, uint32_t *) {
    return false;
}

uint64_t launch_mix_rate(const Launch &L, uint32_t iters, uint32_t *) { count(L); return (uint64_t)iters * 1024; }
void launch_synth_keys(const Launch &L, uint64_t *keys, uint64_t first, uint64_t n, uint64_t seed) {
    if (!n) return;
    for (uint64_t i = 0; i < n; i++) keys[i] = synth_key(first + i, seed);
    count(L);
}
void launch_hash_ids(const Launch &L, const char *packed, const uint64_t *offsets, uint64_t n, uint64_t *keys) {
    if (!n) return;
    for (uint64_t i = 0; i < n; i++) keys[i] = mix64(fnv1a64(packed + offsets[i], (size_t)(offsets[i + 1] - offsets[i])));
    count(L);
}
void launch_fill_u32(const Launch &L, uint32_t *d, uint64_t n, uint32_t v) {
    if (!n) return;
    std::fill(d, d + n, v);
    count(L);
}
void launch_histogram(const Launch &L, const uint32_t *idx, uint64_t n, uint32_t *counters, uint32_t n_total) {
    if (!n) return;
    for (uint64_t i = 0; i < n; i++) if (idx[i] < n_total) counters[idx[i]]++;
    count(L);
}
void launch_l2_flush(const Launch &L, uint32_t *d, uint64_t n, uint32_t v) { launch_fill_u32(L, d, n, v); }

// ---- bounded-load rounds ---------------------------------------------------------------------------------------------------
void launch_select_spill(const Launch &L, const uint64_t *keys, const uint32_t *idx, uint64_t n, const uint32_t *thr, const uint8_t *over, uint32_t round, uint32_t *sel,
                         unsigned long long *nsel, uint32_t *counters) {
    if (!n) return;
    for (uint64_t i = 0; i < n; i++) {
        const uint32_t j = idx[i];
        if (j == kNone || !over[j] || !(spill_hash(keys[i], round) < thr[j])) continue;
        if (counters) counters[j]--;
        sel[(*nsel)++] = (uint32_t)i;
    }
    count(L);
}
void launch_exchange_check(const Launch &L, const uint32_t *local, const BoundedTail &b) {
    capacity_check(b, local);
    count(L);
}
void launch_exchange_p2p(const Launch &L, const uint32_t *local, uint32_t *const *win, uint32_t rank, uint32_t world, uint32_t M, uint32_t max_nodes, uint32_t epoch, uint32_t *out) {
    exchange(local, win, rank, world, M, max_nodes, epoch, out);
    count(L);
}
void launch_sum_gathered(const Launch &L, const uint32_t *g, uint32_t world, uint32_t M, uint32_t *out) {
    if (!M) return;
    for (uint32_t j = 0; j < M; j++) { uint32_t s = 0; for (uint32_t r = 0; r < world; r++) s += g[(size_t)r * M + j]; out[j] = s; }
    count(L);
}

// ---- rebalance of a dense set (DESIGN.md 3.7) ---------------------------------------------------------------------------------
namespace {
// the node an object belongs on after new_idx joined: new_idx iff it beats the incumbent; an incumbent that is not live is
// re-placed by the full rendezvous (what a fresh assignment would do)
uint32_t join_target(uint64_t key, uint32_t cur, uint32_t new_idx, const NodeTabDev &tab) {
    const uint4 nn = tab.by_idx[new_idx];
    if (cur == new_idx || cur >= tab.n_total || !nn.y) return cur;
    const uint4 c = tab.by_idx[cur];
    if (c.y == 0) return hrw_over_table(key, tab);
    const ObjHash o = obj_hash(key);
    const uint32_t un = pair_hash(o, nn.x, nn.z, nn.w), uc = pair_hash(o, c.x, c.z, c.w);
    return cand_better((uint64_t)elog(un) * nn.y, un, new_idx, (uint64_t)elog(uc) * c.y, uc, cur) ? new_idx : cur;
}
}  // namespace

void launch_rebalance_join(const Launch &L, const uint64_t *keys, uint32_t *idx, uint64_t n, const NodeTabDev &tab, uint32_t new_idx, uint32_t *counters, unsigned long long *moved) {
    if (!n) return;
    for (uint64_t i = 0; i < n; i++) {
        const uint32_t cur = idx[i], to = join_target(keys[i], cur, new_idx, tab);
        if (to == cur) continue;
        idx[i] = to;
        ++*moved;
        if (counters) { counters[cur]--; if (to != kNone) counters[to]++; }
    }
    count(L);
}
void launch_select_on_node(const Launch &L, const uint32_t *idx, uint64_t n, uint32_t node, uint32_t *sel, unsigned long long *nsel) {
    if (!n) return;
    for (uint64_t i = 0; i < n; i++) if (idx[i] == node) sel[(*nsel)++] = (uint32_t)i;
    count(L);
}

// ---- directory -----------------------------------------------------------------------------------------------------------------
void launch_dir_init(const Launch &L, DirSlot *slots, uint64_t cap) {
    for (uint64_t i = 0; i < cap; i++) { slots[i].key = kEmptyKey; slots[i].val = kEmptyVal; }
    count(L);
}
void launch_dir_lookup(const Launch &L, const DirDev &dir, const uint64_t *keys, uint64_t n, uint32_t *out) {
    if (!n) return;
    for (uint64_t i = 0; i < n; i++) {
        const unsigned long long key = norm_key(keys[i]);
        uint64_t s = home_slot(key, dir);
        uint32_t res = kNone;
        for (uint64_t probes = 0; probes <= dir.mask; probes++, s = (s + 1) & dir.mask) {
            if (dir.slots[s].key == key) { res = node_of(dir.slots[s]); break; }
            if (dir.slots[s].key == kEmptyKey) break;
        }
        out[i] = res;
    }
    count(L);
}
void launch_dir_upsert(const Launch &L, const DirDev &dir, const uint64_t *keys, const uint32_t *idx, uint32_t const_idx, uint64_t n, uint32_t seq_base, unsigned long long *new_keys,
                       uint32_t *error) {
    if (!n) return;
    for (uint64_t i = 0; i < n; i++) {
        const unsigned long long key = norm_key(keys[i]);
        const uint32_t node = idx ? idx[i] : const_idx;
        uint64_t s = home_slot(key, dir);
        bool placed = false;
        for (uint64_t probes = 0; probes <= dir.mask; probes++, s = (s + 1) & dir.mask) {
            if (dir.slots[s].key == kEmptyKey) { dir.slots[s].key = key; ++*new_keys; }
            if (dir.slots[s].key == key) { placed = true; break; }
        }
        if (!placed) { *error = 1; continue; }
        const unsigned long long v = ((unsigned long long)(seq_base + (uint32_t)i + 1u) << 32) | node;   // later in array order / later batch wins
        if (v > dir.slots[s].val) dir.slots[s].val = v;
    }
    count(L);
}
void launch_dir_clear_seq(const Launch &L, const DirDev &dir) {
    for (uint64_t i = 0; i <= dir.mask; i++) dir.slots[i].val &= 0xFFFFFFFFull;
    count(L);
}
void launch_dir_clean_node(const Launch &L, const DirDev &dir, uint32_t node, unsigned long long *removed) {
    for (uint64_t i = 0; i <= dir.mask; i++) {
        DirSlot &s = dir.slots[i];
        if (s.key != kEmptyKey && node_of(s) == node) { set_node(s, kNone); ++*removed; }
    }
    count(L);
}
void launch_dir_clean_flagged(const Launch &L, const DirDev &dir, const uint8_t *flag, uint32_t n_total, unsigned long long *removed) {
    for (uint64_t i = 0; i <= dir.mask; i++) {
        DirSlot &s = dir.slots[i];
        if (s.key != kEmptyKey && node_of(s) < n_total && flag[node_of(s)]) { set_node(s, kNone); ++*removed; }
    }
    count(L);
}
void launch_dir_rehash(const Launch &L, const DirDev &from, const DirDev &to, unsigned long long *new_keys, uint32_t *error) {
    for (uint64_t i = 0; i <= from.mask; i++) {
        const DirSlot &v = from.slots[i];
        if (v.key == kEmptyKey || node_of(v) == kNone) continue;      // unplaced keys are dropped
        uint64_t s = home_slot(v.key, to);
        bool moved = false;
        for (uint64_t probes = 0; probes <= to.mask; probes++, s = (s + 1) & to.mask)
            if (to.slots[s].key == kEmptyKey) { to.slots[s].key = v.key; to.slots[s].val = node_of(v); moved = true; break; }
        if (moved) ++*new_keys; else *error = 1;
    }
    count(L);
}
void launch_dir_count(const Launch &L, const DirDev &dir, unsigned long long *placed, uint32_t *counters, uint32_t n_total) {
    for (uint64_t i = 0; i <= dir.mask; i++) {
        const DirSlot &s = dir.slots[i];
        if (s.key == kEmptyKey || node_of(s) == kNone) continue;
        ++*placed;
        if (counters && node_of(s) < n_total) counters[node_of(s)]++;
    }
    count(L);
}
void launch_dir_rebalance_join(const Launch &L, const DirDev &dir, const NodeTabDev &tab, uint32_t new_idx, unsigned long long *moved) {
    for (uint64_t i = 0; i <= dir.mask; i++) {
        DirSlot &s = dir.slots[i];
        if (s.key == kEmptyKey || node_of(s) == kNone) continue;
        const uint32_t to = join_target(s.key, node_of(s), new_idx, tab);
        if (to != node_of(s)) { set_node(s, to); ++*moved; }
    }
    count(L);
}
void launch_dir_rebalance_leave(const Launch &L, const DirDev &dir, const NodeTabDev &tab, uint32_t gone, unsigned long long *moved) {
    for (uint64_t i = 0; i <= dir.mask; i++) {
        DirSlot &s = dir.slots[i];
        if (s.key == kEmptyKey || node_of(s) != gone) continue;
        set_node(s, hrw_over_table(s.key, tab));
        ++*moved;
    }
    count(L);
}

// ---- place_batch / check_address_batch support ---------------------------------------------------------------------------------
void launch_classify(const Launch &L, const uint32_t *cur, uint64_t n, const uint8_t *state, uint32_t n_total, uint32_t *sel, unsigned long long *nsel, uint8_t *dead_flag) {
    if (!n) return;
    for (uint64_t i = 0; i < n; i++) {
        const uint32_t c = cur[i];
        bool need = false;
        if (c == kNone || c >= n_total) need = true;                                       // service.rs:241-252
        else if (!(state[c] & kNodeLive)) { need = true; if (!(state[c] & kNodeMalformed)) dead_flag[c] = 1; }   // :226-238 / :213-222
        if (need) sel[(*nsel)++] = (uint32_t)i;
    }
    count(L);
}
void launch_check_address(const Launch &L, const uint32_t *idx, uint64_t n, const uint8_t *verdict_tab, uint32_t n_total, uint8_t *out, uint8_t *dead_flag, unsigned long long *ndead) {
    if (!n) return;
    for (uint64_t i = 0; i < n; i++) {
        const uint8_t v = idx[i] < n_total ? verdict_tab[idx[i]] : (uint8_t)3;
        out[i] = v;
        if (v == 2) { dead_flag[idx[i]] = 1; ++*ndead; }
    }
    count(L);
}
void launch_scatter_const(const Launch &L, uint32_t *out, const uint32_t *sel, uint64_t n_sel, uint32_t v) {
    if (!n_sel) return;
    for (uint64_t i = 0; i < n_sel; i++) out[sel[i]] = v;
    count(L);
}
void launch_gather_keys(const Launch &L, const uint64_t *keys, const uint32_t *sel, uint64_t n_sel, uint64_t *out_keys, const uint32_t *idx, uint32_t *out_idx) {
    if (!n_sel) return;
    for (uint64_t i = 0; i < n_sel; i++) { out_keys[i] = keys[sel[i]]; if (idx) out_idx[i] = idx[sel[i]]; }
    count(L);
}

}  // namespace rio
