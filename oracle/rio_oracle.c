/*
 * rio_oracle.c -- CPU ORACLE for the placement *solver* (test infrastructure, NOT product code).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load this library.  The product path (rio_rs_b200/csrc, librio_cuda.so) never links, loads or
 * calls anything in oracle/.
 *
 * PARITY STATUS: **parity unpinned** for everything in this file.  rcelha/rio-rs has no placement
 * solver: its policy is "the server that first receives the request claims the object"
 * (rio-rs/src/service.rs:241-253) behind a CRUD directory (rio-rs/src/object_placement/mod.rs:38-56).
 * No reference file, test or dependency defines a rendezvous hash, weights, affinity costs or
 * bounded-load rounds, so this file is a restatement of the spec written in DESIGN.md section 3
 * ("Solver spec"; pair hash at revision v3), written independently of the CUDA implementation (no shared headers), and
 * cross-checked by a third, pure-Python implementation in tests/spec_py.py plus the committed
 * golden vectors under tests/golden/.
 *
 * The *directory* oracle (the part the reference does pin) is oracle/directory_model.cpp.
 *
 * Inputs mirror the reference types:
 *   object key  = hash of the LocalObjectPlacement map key "{type}.{id}"
 *                 (rio-rs/src/object_placement/local.rs:26-29,43,61; ObjectId at
 *                 rio-rs/src/service_object.rs:19-26)
 *   node seed   = hash of Member::address() "ip:port" (rio-rs/src/cluster/storage/mod.rs:56-58)
 *
 * Build: see oracle/Makefile (gcc -O2 -pthread -shared -fPIC).
 */
#include <stdint.h>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>

#define ORC_NONE 0xFFFFFFFFu

/* ---- tiny pthread parallel-for (no OpenMP: the image's $CC lacks libgomp) ------------------------ */
#include <pthread.h>
typedef void (*range_fn)(void *ctx, size_t lo, size_t hi);
typedef struct { range_fn fn; void *ctx; size_t lo, hi; } par_job;
static void *par_tramp(void *p) { par_job *j = (par_job *)p; j->fn(j->ctx, j->lo, j->hi); return NULL; }
static void par_for(size_t n, int threads, range_fn fn, void *ctx) {
    if (threads <= 1 || n < 1024) { fn(ctx, 0, n); return; }
    if (threads > 256) threads = 256;
    pthread_t th[256]; par_job jobs[256];
    for (int t = 0; t < threads; t++) {
        jobs[t].fn = fn; jobs[t].ctx = ctx; jobs[t].lo = n * (size_t)t / threads; jobs[t].hi = n * (size_t)(t + 1) / threads;
        pthread_create(&th[t], NULL, par_tramp, &jobs[t]);
    }
    for (int t = 0; t < threads; t++) pthread_join(th[t], NULL);
}

/* ---- spec constants (DESIGN.md section 3.1) -------------------------------------------------- */
#define SALT_OBJ   0xD6E8FEB86659FD93ull
#define SALT_NODE2 0xA0761D6478BD642Full
#define SALT_SPILL 0x2545F4914F6CDD1Dull
#define GOLDEN64   0x9E3779B97F4A7C15ull
#define LOG_K0 0x71376877u
#define LOG_K1 0x44D58AB6u
#define LOG_K2 0x2677DB2Eu
#define LOG_K3 0x0B98D5FAu

/* ---- 3.1 scalar hashes ------------------------------------------------------------------------ */
uint64_t orc_mix64(uint64_t x) {
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
    x ^= x >> 27; x *= 0x94D049BB133111EBull;
    x ^= x >> 31; return x;
}

uint64_t orc_fnv1a64(const uint8_t *p, size_t n) {
    uint64_t h = 0xCBF29CE484222325ull;
    for (size_t i = 0; i < n; i++) { h ^= p[i]; h *= 0x100000001B3ull; }
    return h;
}

/* key of ObjectId(type,id): hash of the bytes of format!("{}.{}", type, id) (local.rs:26-29) */
uint64_t orc_object_key(const char *type, size_t tlen, const char *id, size_t ilen) {
    uint64_t h = 0xCBF29CE484222325ull;
    for (size_t i = 0; i < tlen; i++) { h ^= (uint8_t)type[i]; h *= 0x100000001B3ull; }
    h ^= (uint8_t)'.'; h *= 0x100000001B3ull;
    for (size_t i = 0; i < ilen; i++) { h ^= (uint8_t)id[i]; h *= 0x100000001B3ull; }
    return orc_mix64(h);
}

/* seed of a node address "ip:port" (storage/mod.rs:56-58) */
uint64_t orc_node_seed(const char *addr, size_t n) {
    return orc_mix64(orc_fnv1a64((const uint8_t *)addr, n));
}

/* ---- 3.2 monotone integer -log2 --------------------------------------------------------------- */
static inline uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }

/* Q32 approximation of log2(1+F/2^32); monotone non-decreasing in F (tests/test_oracle_spec.py) */
uint32_t orc_log2frac(uint32_t F) {
    uint32_t t2 = LOG_K2 - mulhi32(F, LOG_K3);
    uint32_t t1 = LOG_K1 - mulhi32(F, t2);
    uint32_t g  = LOG_K0 - mulhi32(F, t1);
    uint32_t q  = mulhi32(F, ~F);
    return F + mulhi32(q, g);
}

/* E(u) = Q26 fixed point of -log2((u+0.5)/2^32)-ish; monotone NON-INCREASING in u */
uint32_t orc_elog(uint32_t u) {
    uint32_t lz = u ? (uint32_t)__builtin_clz(u) : 32u;
    uint32_t m  = lz < 32 ? (u << lz) : 0u;
    uint32_t L  = orc_log2frac(m << 1);
    return ((lz + 1u) << 26) - (L >> 6);
}

/* ---- 3.3 pair hash ----------------------------------------------------------------------------- */
typedef struct { uint32_t b, ab; } orc_objh;

static inline orc_objh obj_hash(uint64_t key) {
    uint64_t h = orc_mix64(key ^ SALT_OBJ);
    uint32_t a = (uint32_t)h;
    orc_objh o; o.b = (uint32_t)(h >> 32) | 1u; o.ab = a * o.b; return o;
}

/* spec v3: u = (p * (s1 | 1) + s2) mod 2^32 with p = (s0*b + ab) mod 2^32 -- two multiply-adds;
 * (s0, s1) = (lo32, hi32) of the node seed, s2 = lo32(mix64(seed ^ SALT_NODE2)) */
static inline uint32_t pair_u(orc_objh o, uint64_t seed, uint32_t s2) {
    uint32_t p = (uint32_t)seed * o.b + o.ab;
    return p * ((uint32_t)(seed >> 32) | 1u) + s2;
}
uint32_t orc_pair_hash(uint64_t key, uint64_t node_seed) {
    return pair_u(obj_hash(key), node_seed, (uint32_t)orc_mix64(node_seed ^ SALT_NODE2));
}

uint32_t orc_inv_weight(uint32_t w) { return w ? 0xFFFFFFFFu / w : 0u; }

/* ---- 3.4 weighted rendezvous: lexicographic min over live nodes of (E(u)*r, ~u, j) ---------- */
/* weight[j]==0 means "not live".  mask (may be NULL): bit j set => node j excluded ("closed").  */
static uint32_t hrw_one(uint64_t key, const uint64_t *seed, const uint64_t *seed2, const uint32_t *invw,
                        const uint32_t *mask, uint32_t M, uint64_t *out_score, uint32_t *out_u) {
    orc_objh o = obj_hash(key);
    uint64_t best = ~0ull; uint32_t bu = 0, bj = ORC_NONE;
    for (uint32_t j = 0; j < M; j++) {
        if (!invw[j]) continue;
        if (mask && (mask[j >> 5] >> (j & 31) & 1u)) continue;
        uint32_t u = pair_u(o, seed[j], (uint32_t)seed2[j]);
        uint64_t sc = (uint64_t)orc_elog(u) * invw[j];
        if (bj == ORC_NONE || sc < best || (sc == best && u > bu)) { best = sc; bu = u; bj = j; }
    }
    if (out_score) *out_score = best;
    if (out_u) *out_u = bu;
    return bj;
}

typedef struct { uint64_t *seed2; uint32_t *invw; } node_tab;

static node_tab make_tab(const uint64_t *seed, const uint32_t *weight, uint32_t M) {
    node_tab t; t.seed2 = (uint64_t *)malloc(sizeof(uint64_t) * (M ? M : 1));
    t.invw = (uint32_t *)malloc(sizeof(uint32_t) * (M ? M : 1));
    for (uint32_t j = 0; j < M; j++) { t.seed2[j] = orc_mix64(seed[j] ^ SALT_NODE2); t.invw[j] = orc_inv_weight(weight[j]); }
    return t;
}

/* Flat weighted-HRW assignment.  out_score/out_u may be NULL.  threads<=1 => serial. */
typedef struct { const uint64_t *keys, *seed; node_tab t; const uint32_t *mask; uint32_t M;
                 uint32_t *out_idx; uint64_t *out_score; uint32_t *out_u; } hrw_ctx;
static void hrw_range(void *p, size_t lo, size_t hi) {
    hrw_ctx *c = (hrw_ctx *)p;
    for (size_t i = lo; i < hi; i++) {
        uint64_t sc; uint32_t u;
        c->out_idx[i] = hrw_one(c->keys[i], c->seed, c->t.seed2, c->t.invw, c->mask, c->M, &sc, &u);
        if (c->out_score) c->out_score[i] = sc;
        if (c->out_u) c->out_u[i] = u;
    }
}
void orc_assign_hrw(const uint64_t *keys, size_t n, const uint64_t *seed, const uint32_t *weight,
                    const uint32_t *mask, uint32_t M, uint32_t *out_idx, uint64_t *out_score,
                    uint32_t *out_u, int threads) {
    hrw_ctx c = { keys, seed, make_tab(seed, weight, M), mask, M, out_idx, out_score, out_u };
    par_for(n, threads, hrw_range, &c);
    free(c.t.seed2); free(c.t.invw);
}

/* ---- 3.5 bounded-load rounds -------------------------------------------------------------------
 * cap_j = ceil(cap_num * N * w_j / (cap_den * W)); each round: over = {live j: c_j > cap_j};
 * closed |= over; objects on an over node spill iff spillhash(key, round) < floor(2^32*(c-cap)/c);
 * spilled objects re-run HRW over live \ closed.  Returns number of assignment passes run.      */
uint32_t orc_spill_hash(uint64_t key, uint32_t round) {
    return (uint32_t)(orc_mix64(key ^ (SALT_SPILL + (uint64_t)round * GOLDEN64)) >> 32);
}

uint32_t orc_capacity(uint64_t n_total, uint32_t w, uint64_t w_sum, uint32_t cap_num, uint32_t cap_den) {
    if (!w || !w_sum || !cap_den) return 0;
    unsigned __int128 num = (unsigned __int128)cap_num * n_total * w;
    unsigned __int128 den = (unsigned __int128)cap_den * w_sum;
    unsigned __int128 q = (num + den - 1) / den;
    return q > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)q;
}

typedef struct { const uint64_t *keys, *seed; node_tab t; const uint32_t *closed; const uint8_t *over;
                 const uint32_t *thr; uint32_t M, round; uint32_t *out_idx; } spill_ctx;
uint32_t orc_spill_hash(uint64_t key, uint32_t round);
static void spill_range(void *p, size_t lo, size_t hi) {
    spill_ctx *c = (spill_ctx *)p;
    for (size_t i = lo; i < hi; i++) {
        uint32_t j = c->out_idx[i];
        if (j == ORC_NONE || !c->over[j]) continue;
        if (orc_spill_hash(c->keys[i], c->round) < c->thr[j])
            c->out_idx[i] = hrw_one(c->keys[i], c->seed, c->t.seed2, c->t.invw, c->closed, c->M, NULL, NULL);
    }
}

uint32_t orc_assign_bounded(const uint64_t *keys, size_t n, const uint64_t *seed, const uint32_t *weight,
                            uint32_t M, uint32_t cap_num, uint32_t cap_den, uint32_t max_rounds,
                            uint32_t *out_idx, uint32_t *out_counts, int threads) {
    node_tab t = make_tab(seed, weight, M);
    uint32_t words = (M + 31) / 32;
    uint32_t *closed = (uint32_t *)calloc(words ? words : 1, 4);
    uint32_t *cap = (uint32_t *)calloc(M ? M : 1, 4);
    uint32_t *thr = (uint32_t *)calloc(M ? M : 1, 4);
    uint8_t *over = (uint8_t *)calloc(M ? M : 1, 1);
    uint64_t W = 0;
    for (uint32_t j = 0; j < M; j++) W += weight[j];
    for (uint32_t j = 0; j < M; j++) cap[j] = orc_capacity(n, weight[j], W, cap_num, cap_den);
    hrw_ctx c0 = { keys, seed, t, NULL, M, out_idx, NULL, NULL };
    par_for(n, threads, hrw_range, &c0);
    uint32_t passes = 1;
    for (uint32_t r = 1; r < max_rounds; r++) {
        memset(out_counts, 0, 4 * (size_t)M);
        for (size_t i = 0; i < n; i++) if (out_idx[i] != ORC_NONE) out_counts[out_idx[i]]++;
        int any = 0; uint32_t open = 0;
        for (uint32_t j = 0; j < M; j++) {
            over[j] = weight[j] && out_counts[j] > cap[j];
            if (over[j]) { any = 1; closed[j >> 5] |= 1u << (j & 31);
                thr[j] = (uint32_t)((((uint64_t)(out_counts[j] - cap[j])) << 32) / out_counts[j]); }
        }
        for (uint32_t j = 0; j < M; j++) if (weight[j] && !(closed[j >> 5] >> (j & 31) & 1u)) open++;
        if (!any || !open) break;
        spill_ctx sc = { keys, seed, t, closed, over, thr, M, r, out_idx };
        par_for(n, threads, spill_range, &sc);
        passes++;
    }
    memset(out_counts, 0, 4 * (size_t)M);
    for (size_t i = 0; i < n; i++) if (out_idx[i] != ORC_NONE) out_counts[out_idx[i]]++;
    free(t.seed2); free(t.invw); free(closed); free(cap); free(thr); free(over);
    return passes;
}

/* ---- 3.6 affinity cost: cost_ij = -sum_k Fobj[i,k]*Fnode[j,k] evaluated in fp64; argmin, ties ->
 * lowest j.  live[j]==0 excludes node j.  out_gap = (second best cost - best cost) (inf if M_live<2) */
typedef struct { const float *fobj, *fnode; const uint32_t *weight; uint32_t M, K; uint32_t *out_idx;
                 double *out_cost, *out_gap; } aff_ctx;
static void aff_range(void *p, size_t lo, size_t hi) {
    aff_ctx *a = (aff_ctx *)p;
    const float *fobj = a->fobj, *fnode = a->fnode; const uint32_t *weight = a->weight;
    uint32_t M = a->M, K = a->K; uint32_t *out_idx = a->out_idx; double *out_cost = a->out_cost, *out_gap = a->out_gap;
    for (size_t i = lo; i < hi; i++) {
        double best = 0, second = 0; uint32_t bj = ORC_NONE; int have2 = 0;
        const float *fo = fobj + (size_t)i * K;
        for (uint32_t j = 0; j < M; j++) {
            if (!weight[j]) continue;
            const float *fn = fnode + (size_t)j * K;
            double d = 0;
            for (uint32_t k = 0; k < K; k++) d += (double)fo[k] * (double)fn[k];
            double c = -d;
            if (bj == ORC_NONE) { best = c; bj = j; }
            else if (c < best) { second = best; have2 = 1; best = c; bj = j; }
            else if (!have2 || c < second) { second = c; have2 = 1; }
        }
        out_idx[i] = bj;
        if (out_cost) out_cost[i] = best;
        if (out_gap) out_gap[i] = have2 ? second - best : __builtin_inf();
    }
}
void orc_assign_affinity(const float *fobj, const float *fnode, const uint32_t *weight, size_t n, uint32_t M,
                         uint32_t K, uint32_t *out_idx, double *out_cost, double *out_gap, int threads) {
    aff_ctx a = { fobj, fnode, weight, M, K, out_idx, out_cost, out_gap };
    par_for(n, threads, aff_range, &a);
}

/* ---- 3.6 in fp32 with the CUDA-core arithmetic: an IMPLEMENTATION RESTATEMENT, not spec ------------------------------
 * The spec (above) is the fp64 argmin.  This restates what the CUDA-core kernels (k_assign_affinity, K = 16, and
 * k_assign_affinity_generic) and the tensor-core path's fp32 re-scoring of its 8 candidates are specified to compute:
 * acc = fmaf(Fobj[i,k], Fnode[j,k], acc) for k = 0..K-1 starting from +0.f, cost = -acc, strict < over the live nodes in
 * index order (ties -> lowest j), ORC_NONE when no node is live.  libm fmaf is correctly rounded, so the chain is bit for
 * bit the device's FFMA chain; an emulation in fp64 would round twice. */
static float aff_cost_f32(const float *fo, const float *fn, uint32_t K) {
    float acc = 0.f;
    for (uint32_t k = 0; k < K; k++) acc = fmaf(fo[k], fn[k], acc);
    return -acc;
}
static void aff_f32_range(void *p, size_t lo, size_t hi) {
    aff_ctx *a = (aff_ctx *)p;
    for (size_t i = lo; i < hi; i++) {
        const float *fo = a->fobj + i * a->K;
        float best = 0.f; uint32_t bj = ORC_NONE;
        for (uint32_t j = 0; j < a->M; j++) {
            if (!a->weight[j]) continue;
            const float c = aff_cost_f32(fo, a->fnode + (size_t)j * a->K, a->K);
            if (bj == ORC_NONE || c < best) { best = c; bj = j; }
        }
        a->out_idx[i] = bj;
    }
}
void orc_assign_affinity_f32(const float *fobj, const float *fnode, const uint32_t *weight, size_t n, uint32_t M, uint32_t K,
                             uint32_t *out_idx, int threads) {
    aff_ctx a = { fobj, fnode, weight, M, K, out_idx, NULL, NULL };
    par_for(n, threads, aff_f32_range, &a);
}

/* the same fp32 cost for given (object, node) pairs */
typedef struct { const float *fobj, *fnode; const uint32_t *obj, *node; uint32_t K; float *out; } pair_ctx;
static void pair_range(void *p, size_t lo, size_t hi) {
    pair_ctx *c = (pair_ctx *)p;
    for (size_t q = lo; q < hi; q++) c->out[q] = aff_cost_f32(c->fobj + (size_t)c->obj[q] * c->K, c->fnode + (size_t)c->node[q] * c->K, c->K);
}
void orc_affinity_pair_cost_f32(const float *fobj, const float *fnode, const uint32_t *obj, const uint32_t *node, size_t n_pairs, uint32_t K,
                                float *out_cost, int threads) {
    pair_ctx c = { fobj, fnode, obj, node, K, out_cost };
    par_for(n_pairs, threads, pair_range, &c);
}

/* ---- synthetic inputs (SURVEY section 8d) --------------------------------------------------------- */
/* key[i] = mix64(GOLDEN*(i+1) ^ seed) */
void orc_synth_keys(uint64_t *out, size_t n, uint64_t first, uint64_t seed) {
    for (size_t i = 0; i < n; i++) out[i] = orc_mix64(GOLDEN64 * (first + i + 1) ^ seed);
}

/* histogram helper */
void orc_counts(const uint32_t *idx, size_t n, uint32_t M, uint32_t *out_counts) {
    memset(out_counts, 0, 4 * (size_t)M);
    for (size_t i = 0; i < n; i++) if (idx[i] < M) out_counts[idx[i]]++;
}

/* ---- 3.8 HRW2: hierarchical weighted rendezvous with fan-out 2 ("rendezvous trie") ----------------------------
 * Spec (DESIGN.md 3.8), restated here from the text, NOT from the CUDA host code (which precomputes a heap of
 * thresholds; this file re-derives every contest from prefix sums of the members sorted by position):
 *   pos(j)   = mix64(seed_j ^ SALT_POS);  bucket(j) = pos(j) >> (64 - bits)   (0 when bits == 0)
 *   v(key, s) = (p*m + (s2 & 0x7FFFFFFF)) mod 2^31 with p = (lo32(s)*b + ab) mod 2^32, m = hi32(s)|1, s2 = lo32(mix64(s ^ SALT_NODE2)),
 *               (b, ab) the object's hashed pair of 3.3 -- the flat pair hash reduced to 31 bits
 *   level l  acts as a pseudo-node with seed c_l = mix64(GOLDEN64*(l+1) ^ SALT_LVL)
 *   contest(key, s, WL, WR): T = floor(2^31 * WL / (WL + WR));  LEFT iff v(key, s) < T      (s = c_l on trie level l)
 *     -- the closed form of a 2-way weighted rendezvous between two subtrees: P(LEFT) = WL/(WL+WR) (+-2^-31)
 *   levels 0..bits-1 walk the binary trie over bucket ids, most significant bit first (LEFT = bit 0);
 *   inside the bucket the live members sorted by (pos, index) are m_0..m_{c-1}: for k = 0..c-2 the contest "m_k against
 *     the rest" is keyed by the member's own seed: contest(key, seed(m_k), w_k, sum_{i>k} w_i) LEFT
 *     takes m_k; nobody took -> m_{c-1}.  (Keyed by the member, not by its rank, so a member's hash survives others leaving.)
 *   weight 0 / masked nodes are not members.  No live member -> NONE. */
#define SALT_POS 0x8CB92BA72F3D8DD7ull
#define SALT_LVL 0x3C79AC492BA7B653ull

uint64_t orc_hrw2_pos(uint64_t seed) { return orc_mix64(seed ^ SALT_POS); }
uint64_t orc_hrw2_level_seed(uint32_t level) { return orc_mix64(GOLDEN64 * ((uint64_t)level + 1) ^ SALT_LVL); }
uint32_t orc_hrw2_threshold(uint64_t wl, uint64_t wr) {
    if (wl + wr == 0) return 0;
    return (uint32_t)((((unsigned __int128)wl) << 31) / (wl + wr));   /* <= 2^31 */
}

typedef struct { uint64_t pos, seed; uint32_t j, w; } h2_member;
static int h2_cmp(const void *a, const void *b) {
    const h2_member *x = (const h2_member *)a, *y = (const h2_member *)b;
    if (x->pos != y->pos) return x->pos < y->pos ? -1 : 1;
    return x->j < y->j ? -1 : (x->j > y->j);
}
typedef struct { const uint64_t *keys; const h2_member *mem; const uint64_t *pre; /* pre[i] = sum of w of mem[0..i) */
                 uint32_t c, bits; uint32_t *out_idx; } h2_ctx;

/* 31-bit contest hash of (key, seed): same multiply-add form as the flat pair hash, reduced mod 2^31 */
uint32_t orc_hrw2_v(uint64_t key, uint64_t seed) {
    orc_objh o = obj_hash(key);
    uint32_t p = (uint32_t)seed * o.b + o.ab;
    uint32_t s2 = (uint32_t)orc_mix64(seed ^ SALT_NODE2);
    return (p * ((uint32_t)(seed >> 32) | 1u) + (s2 & 0x7FFFFFFFu)) & 0x7FFFFFFFu;
}
static inline int h2_left(uint64_t key, uint64_t contest_seed, uint64_t wl, uint64_t wr) {
    return orc_hrw2_v(key, contest_seed) < orc_hrw2_threshold(wl, wr);
}
/* first member in [lo,hi) whose pos has bit `bit` (counted from the top, 0 = MSB) set; members are sorted by pos and
 * share the bits above, so this is the split point of the subtree */
static uint32_t h2_split(const h2_member *mem, uint32_t lo, uint32_t hi, uint32_t bit) {
    while (lo < hi) { uint32_t mid = lo + (hi - lo) / 2; if ((mem[mid].pos >> (63 - bit)) & 1u) hi = mid; else lo = mid + 1; }
    return lo;
}
static void h2_range(void *p, size_t a, size_t b) {
    h2_ctx *c = (h2_ctx *)p;
    for (size_t i = a; i < b; i++) {
        uint32_t lo = 0, hi = c->c;
        if (!hi) { c->out_idx[i] = ORC_NONE; continue; }
        const uint64_t key = c->keys[i];
        for (uint32_t l = 0; l < c->bits; l++) {
            uint32_t mid = h2_split(c->mem, lo, hi, l);
            uint64_t wl = c->pre[mid] - c->pre[lo], wr = c->pre[hi] - c->pre[mid];
            if (h2_left(key, orc_hrw2_level_seed(l), wl, wr)) hi = mid; else lo = mid;
        }
        uint32_t k = lo;
        for (; k + 1 < hi; k++)   /* the member's own pair hash (the flat rendezvous hash of (key, node)) decides "m_k or the rest" */
            if (h2_left(key, c->mem[k].seed, c->mem[k].w, c->pre[hi] - c->pre[k + 1])) break;
        c->out_idx[i] = c->mem[k].j;
    }
}
void orc_assign_hrw2(const uint64_t *keys, size_t n, const uint64_t *seed, const uint32_t *weight, const uint32_t *mask,
                     uint32_t M, uint32_t bits, uint32_t *out_idx, int threads) {
    h2_member *mem = (h2_member *)malloc(sizeof(h2_member) * (M ? M : 1));
    uint32_t c = 0;
    for (uint32_t j = 0; j < M; j++) {
        if (!weight[j]) continue;
        if (mask && (mask[j >> 5] >> (j & 31) & 1u)) continue;
        mem[c].pos = orc_hrw2_pos(seed[j]); mem[c].seed = seed[j]; mem[c].j = j; mem[c].w = weight[j]; c++;
    }
    qsort(mem, c, sizeof(h2_member), h2_cmp);
    uint64_t *pre = (uint64_t *)malloc(8 * ((size_t)c + 1));
    pre[0] = 0;
    for (uint32_t i = 0; i < c; i++) pre[i + 1] = pre[i] + mem[i].w;
    h2_ctx ctx = { keys, mem, pre, c, bits, out_idx };
    par_for(n, threads, h2_range, &ctx);
    free(mem); free(pre);
}

/* 3.5 bounded-load rounds on top of the HRW2 policy: identical round rule, the assignment passes use orc_assign_hrw2
 * (closed nodes are simply not members of the trie of the later passes). */
uint32_t orc_assign_bounded_hrw2(const uint64_t *keys, size_t n, const uint64_t *seed, const uint32_t *weight,
                                 uint32_t M, uint32_t bits, uint32_t cap_num, uint32_t cap_den, uint32_t max_rounds,
                                 uint32_t *out_idx, uint32_t *out_counts, int threads) {
    uint32_t words = (M + 31) / 32;
    uint32_t *closed = (uint32_t *)calloc(words ? words : 1, 4);
    uint32_t *cap = (uint32_t *)calloc(M ? M : 1, 4);
    uint32_t *thr = (uint32_t *)calloc(M ? M : 1, 4);
    uint8_t *over = (uint8_t *)calloc(M ? M : 1, 1);
    uint64_t *skeys = (uint64_t *)malloc(8 * (n ? n : 1));
    uint32_t *spos = (uint32_t *)malloc(4 * (n ? n : 1)), *sidx = (uint32_t *)malloc(4 * (n ? n : 1));
    uint64_t W = 0;
    for (uint32_t j = 0; j < M; j++) W += weight[j];
    for (uint32_t j = 0; j < M; j++) cap[j] = orc_capacity(n, weight[j], W, cap_num, cap_den);
    orc_assign_hrw2(keys, n, seed, weight, NULL, M, bits, out_idx, threads);
    uint32_t passes = 1;
    for (uint32_t r = 1; r < max_rounds; r++) {
        orc_counts(out_idx, n, M, out_counts);
        int any = 0; uint32_t open = 0;
        for (uint32_t j = 0; j < M; j++) {
            over[j] = weight[j] && out_counts[j] > cap[j];
            if (over[j]) { any = 1; closed[j >> 5] |= 1u << (j & 31);
                thr[j] = (uint32_t)((((uint64_t)(out_counts[j] - cap[j])) << 32) / out_counts[j]); }
        }
        for (uint32_t j = 0; j < M; j++) if (weight[j] && !(closed[j >> 5] >> (j & 31) & 1u)) open++;
        if (!any || !open) break;
        size_t ns = 0;
        for (size_t i = 0; i < n; i++) {
            uint32_t j = out_idx[i];
            if (j == ORC_NONE || !over[j]) continue;
            if (orc_spill_hash(keys[i], r) < thr[j]) { skeys[ns] = keys[i]; spos[ns] = (uint32_t)i; ns++; }
        }
        orc_assign_hrw2(skeys, ns, seed, weight, closed, M, bits, sidx, threads);
        for (size_t q = 0; q < ns; q++) out_idx[spos[q]] = sidx[q];
        passes++;
    }
    orc_counts(out_idx, n, M, out_counts);
    free(closed); free(cap); free(thr); free(over); free(skeys); free(spos); free(sidx);
    return passes;
}
