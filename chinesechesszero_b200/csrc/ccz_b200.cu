// ccz_b200.cu -- C-ABI entry points (include/ccz_b200.h) over the sm_100a kernels.
// One translation unit: the constant tables in ccz_rules.cuh are shared by all kernels.
#include "../../include/ccz_b200.h"

#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <utility>
#include <string>

#include "ccz_movegen.cuh"
#include "ccz_mcts.cuh"
#include "ccz_replay.cuh"
#include "ccz_conv.cuh"
#include "ccz_stem.cuh"
#include "ccz_heads.cuh"
#include "ccz_dedup.cuh"

#ifndef CCZ_CONV_DEFAULT_PAIRS
#define CCZ_CONV_DEFAULT_PAIRS 1
#endif

namespace {

thread_local std::string g_err;

int fail(int code, const char *what, cudaError_t e = cudaSuccess) {
    g_err = what;
    if (e != cudaSuccess) {
        g_err += ": ";
        g_err += cudaGetErrorString(e);
    }
    return code;
}

#define CCZ_CUDA(call)                                      \
    do {                                                    \
        cudaError_t e_ = (call);                            \
        if (e_ != cudaSuccess) return fail(-2, #call, e_);  \
    } while (0)

// ---- host-side constant tables -------------------------------------------------------------
struct HostTables {
    int16_t id_of[8100];
    uint8_t from_of[ccz::N_ACTIONS], to_of[ccz::N_ACTIONS];
    int16_t flip_of[ccz::N_ACTIONS];
    uint64_t zkeys[16 * 90 + 1];
    uint8_t start[ccz::BOARD_BYTES];
    uint16_t step_tab[ccz::STEP_TAB_ENTRIES];
    bool built = false;
};
HostTables g_tab;
bool g_dev_ready[64] = {false};
// generation-order policy (see ccz_set_order_policy): host copy, uploaded to every device on its next use
const ccz_order_policy kDefaultPolicy = {{0, 1, 0, 0, 0, 0, 0, 0}, 1, 1, 0, 0};
ccz_order_policy g_policy = kDefaultPolicy;
bool g_policy_is_default = true;
unsigned g_policy_version = 1, g_dev_policy_version[64] = {0};

int sq_of(const char *s) { return (s[0] - 'a') + 9 * (s[1] - '0'); }

// Step-piece move table for K1 (layout in ccz_movegen.cuh): per (piece kind, from-square) the
// targets `to | block << 7` (block = knight leg / elephant eye, 127 = none) sorted by target square
// DESCENDING (cchess generation order), 0xFFFF-terminated.
void build_step_table(uint16_t *tab) {
    for (int i = 0; i < ccz::STEP_TAB_ENTRIES; ++i) tab[i] = 0xFFFF;
    // piece: 0 pawn, 1 elephant, 2 advisor, 3 king (x colour), 4 knight
    for (int piece = 0; piece < 5; ++piece)
        for (int black = 0; black < (piece == 4 ? 1 : 2); ++black)
            for (int sq = 0; sq < 90; ++sq) {
                const int r = sq / 9, f = sq % 9;
                int to[8], blk[8], m = 0;
                auto add = [&](int rr, int ff, int b) {
                    if (rr < 0 || rr > 9 || ff < 0 || ff > 8) return;
                    to[m] = rr * 9 + ff;
                    blk[m++] = b;
                };
                auto in_palace = [&](int rr, int ff) {
                    return ff >= 3 && ff <= 5 && (black ? (rr >= 7 && rr <= 9) : (rr >= 0 && rr <= 2));
                };
                if (piece == 0) { // pawn: forward; sideways once across the river
                    add(r + (black ? -1 : 1), f, 127);
                    if (black ? r <= 4 : r >= 5) { add(r, f - 1, 127); add(r, f + 1, 127); }
                } else if (piece == 4) { // knight: leg next to the knight along the long axis
                    static const int d[8][2] = {{2, 1}, {2, -1}, {-2, 1}, {-2, -1}, {1, 2}, {1, -2}, {-1, 2}, {-1, -2}};
                    for (auto &k : d) {
                        const int lr = r + (k[0] == 2 ? 1 : k[0] == -2 ? -1 : 0);
                        const int lf = f + (k[1] == 2 ? 1 : k[1] == -2 ? -1 : 0);
                        add(r + k[0], f + k[1], lr * 9 + lf);
                    }
                } else if (piece == 1) { // elephant: eye in the middle, never crosses the river
                    for (int a = -2; a <= 2; a += 4)
                        for (int c = -2; c <= 2; c += 4) {
                            const int rr = r + a;
                            if (rr < 0 || rr > 9 || (black ? rr < 5 : rr > 4)) continue;
                            add(rr, f + c, (r + a / 2) * 9 + f + c / 2);
                        }
                } else if (piece == 2) { // advisor
                    for (int a = -1; a <= 1; a += 2)
                        for (int c = -1; c <= 1; c += 2)
                            if (in_palace(r + a, f + c)) add(r + a, f + c, 127);
                } else { // king
                    static const int d[4][2] = {{1, 0}, {-1, 0}, {0, 1}, {0, -1}};
                    for (auto &k : d)
                        if (in_palace(r + k[0], f + k[1])) add(r + k[0], f + k[1], 127);
                }
                for (int i = 0; i < m; ++i) // descending by target
                    for (int j = i + 1; j < m; ++j)
                        if (to[j] > to[i]) { std::swap(to[i], to[j]); std::swap(blk[i], blk[j]); }
                uint16_t *e = piece == 4 ? tab + sq * 8
                                         : tab + ccz::STEP_KNIGHT_ENTRIES + ((piece * 2 + black) * 90 + sq) * 4;
                for (int i = 0; i < m; ++i) e[i] = (uint16_t)(to[i] | (blk[i] << 7));
            }
}

// The fixed 2086-entry action table (tools.py:172-272): per source square in rank-major order
// the 9 same-file destinations by rank, the 8 same-rank destinations by file, then the knight
// jumps (drank,dfile) = (-2,-1) (-1,-2) (-2,1) (1,-2) (2,-1) (-1,2) (2,1) (1,2) that stay on
// the board; then the 16 advisor and 32 elephant moves in the reference's literal order.
void build_tables() {
    if (g_tab.built) return;
    HostTables &t = g_tab;
    for (int i = 0; i < 8100; ++i) t.id_of[i] = -1;
    int idx = 0;
    auto add = [&](int from, int to) {
        t.id_of[from * 90 + to] = (int16_t)idx;
        t.from_of[idx] = (uint8_t)from;
        t.to_of[idx] = (uint8_t)to;
        ++idx;
    };
    static const int kn[8][2] = {{-2, -1}, {-1, -2}, {-2, 1}, {1, -2}, {2, -1}, {-1, 2}, {2, 1}, {1, 2}};
    for (int rank = 0; rank < 10; ++rank)
        for (int file = 0; file < 9; ++file) {
            const int from = file + 9 * rank;
            for (int r2 = 0; r2 < 10; ++r2)
                if (r2 != rank) add(from, file + 9 * r2);
            for (int f2 = 0; f2 < 9; ++f2)
                if (f2 != file) add(from, f2 + 9 * rank);
            for (auto &k : kn) {
                const int r2 = rank + k[0], f2 = file + k[1];
                if (r2 >= 0 && r2 < 10 && f2 >= 0 && f2 < 9) add(from, f2 + 9 * r2);
            }
        }
    static const char *const advisor[] = {"d0e1", "e1d0", "f0e1", "e1f0", "d2e1", "e1d2", "f2e1", "e1f2",
                                          "d9e8", "e8d9", "f9e8", "e8f9", "d7e8", "e8d7", "f7e8", "e8f7"};
    static const char *const elephant[] = {
        "a2c0", "c0a2", "a2c4", "c4a2", "c0e2", "e2c0", "c4e2", "e2c4", "e2g0", "g0e2", "e2g4",
        "g4e2", "g0i2", "i2g0", "g4i2", "i2g4", "a7c5", "c5a7", "a7c9", "c9a7", "c5e7", "e7c5",
        "c9e7", "e7c9", "e7g5", "g5e7", "e7g9", "g9e7", "g5i7", "i7g5", "g9i7", "i7g9"};
    for (const char *m : advisor) add(sq_of(m), sq_of(m + 2));
    for (const char *m : elephant) add(sq_of(m), sq_of(m + 2));
    // file mirror of every action (tools.py:133-164, collect.py:117-122)
    for (int i = 0; i < ccz::N_ACTIONS; ++i) {
        const int f = t.from_of[i], to = t.to_of[i];
        const int mf = (8 - f % 9) + 9 * (f / 9), mt = (8 - to % 9) + 9 * (to / 9);
        t.flip_of[i] = t.id_of[mf * 90 + mt];
    }
    // position keys: splitmix64 stream
    uint64_t x = 0x0123456789ABCDEFull;
    for (int i = 0; i < 16 * 90 + 1; ++i) {
        x += 0x9E3779B97F4A7C15ull;
        uint64_t z = x;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        t.zkeys[i] = z ^ (z >> 31);
    }
    // start position: rnbakabnr/9/1c5c1/p1p1p1p1p/9/9/P1P1P1P1P/1C5C1/9/RNBAKABNR w
    std::memset(t.start, 0, sizeof(t.start));
    static const uint8_t back[9] = {3, 4, 5, 6, 7, 6, 5, 4, 3};
    for (int f = 0; f < 9; ++f) {
        t.start[f] = back[f];
        t.start[81 + f] = back[f] | 8;
    }
    t.start[19] = t.start[25] = 2;
    t.start[64] = t.start[70] = 2 | 8;
    for (int f = 0; f < 9; f += 2) {
        t.start[27 + f] = 1;
        t.start[54 + f] = 1 | 8;
    }
    t.start[ccz::OFF_TURN] = 1;
    build_step_table(t.step_tab);
    t.built = (idx == ccz::N_ACTIONS);
}

int ensure_device() {
    build_tables();
    if (!g_tab.built) return fail(-3, "action table construction failed");
    int dev = 0;
    CCZ_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return fail(-3, "device index out of range");
    if (g_dev_policy_version[dev] != g_policy_version) {
        CCZ_CUDA(cudaMemcpyToSymbol(ccz::d_order_policy, &g_policy, sizeof(g_policy)));
        g_dev_policy_version[dev] = g_policy_version;
    }
    if (g_dev_ready[dev]) return 0;
    CCZ_CUDA(cudaMemcpyToSymbol(ccz::d_id_of, g_tab.id_of, sizeof(g_tab.id_of)));
    CCZ_CUDA(cudaMemcpyToSymbol(ccz::d_from_of, g_tab.from_of, sizeof(g_tab.from_of)));
    CCZ_CUDA(cudaMemcpyToSymbol(ccz::d_to_of, g_tab.to_of, sizeof(g_tab.to_of)));
    CCZ_CUDA(cudaMemcpyToSymbol(ccz::d_flip_of, g_tab.flip_of, sizeof(g_tab.flip_of)));
    CCZ_CUDA(cudaMemcpyToSymbol(ccz::d_zkeys, g_tab.zkeys, sizeof(g_tab.zkeys)));
    CCZ_CUDA(cudaMemcpyToSymbol(ccz::d_start_board, g_tab.start, sizeof(g_tab.start)));
    CCZ_CUDA(cudaMemcpyToSymbol(ccz::d_step_tab, g_tab.step_tab, sizeof(g_tab.step_tab)));
    g_dev_ready[dev] = true;
    return 0;
}

int sm_count() {
    static int cached = 0;
    if (!cached) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
        if (cached <= 0) cached = 148;
    }
    return cached;
}

int check_launch(const char *what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(-2, what, e);
    return 0;
}

int check_arena(const ccz_arena *a) {
    if (!a) return fail(-1, "arena is NULL");
    if (a->n_games <= 0 || a->n_pages < a->n_games || a->max_pages < 1) return fail(-1, "arena geometry invalid");
    if (a->page_shift < 7 || a->page_shift > 16 || ((long long)a->n_pages << a->page_shift) > 0x7fffffffll)
        return fail(-1, "arena geometry invalid: page_shift must be 7..16 and n_pages << page_shift < 2^31");
    if (!a->d_nodes || !a->d_links || !a->d_free_ring || !a->d_pool_ctl || !a->d_page_list || !a->d_page_fill ||
        !a->d_n_pages || !a->d_n_pages_new || !a->d_list_sel || !a->d_alloc_page || !a->d_alloc_off || !a->d_root ||
        !a->d_n_nodes || !a->d_status || !a->d_root_boards || !a->d_root_keys)
        return fail(-1, "arena has a NULL array");
    if (((uintptr_t)a->d_nodes & 15) || ((uintptr_t)a->d_links & 7) || ((uintptr_t)a->d_pool_ctl & 7))
        return fail(-1, "arena node arrays must be 16-byte aligned");
    return 0;
}

inline int warps_grid(int n) { return (n + ccz::MCTS_WARPS - 1) / ccz::MCTS_WARPS; }

} // namespace

extern "C" {

int ccz_version(void) { return 200; }

const char *ccz_last_error(void) { return g_err.c_str(); }

int ccz_init(void) { return ensure_device(); }

int ccz_action_table(int16_t *id_of, uint8_t *from_of, uint8_t *to_of) {
    build_tables();
    if (!g_tab.built) return fail(-3, "action table construction failed");
    if (id_of) std::memcpy(id_of, g_tab.id_of, sizeof(g_tab.id_of));
    if (from_of) std::memcpy(from_of, g_tab.from_of, sizeof(g_tab.from_of));
    if (to_of) std::memcpy(to_of, g_tab.to_of, sizeof(g_tab.to_of));
    return ccz::N_ACTIONS;
}

int ccz_set_order_policy(const ccz_order_policy *p) {
    static_assert(sizeof(ccz_order_policy) == 12, "ccz_order_policy layout");
    const ccz_order_policy &q = p ? *p : kDefaultPolicy;
    if (q.capture_mode > 2 || q.from_descending > 1 || q.to_descending > 1 || q.check_king_first > 1)
        return fail(-1, "ccz_set_order_policy: from_descending / to_descending / check_king_first must be 0|1, capture_mode 0|1|2");
    for (int t = 1; t <= 7; ++t)
        if (q.class_rank[t] > 7) return fail(-1, "ccz_set_order_policy: class_rank must be 0..7");
    g_policy = q;
    g_policy.class_rank[0] = 0;
    g_policy_is_default = std::memcmp(&g_policy, &kDefaultPolicy, sizeof(g_policy)) == 0;
    ++g_policy_version; // uploaded (synchronously, cudaMemcpyToSymbol) by the next entry point on each device
    return 0;
}

int ccz_get_order_policy(ccz_order_policy *out) {
    if (!out) return fail(-1, "ccz_get_order_policy: NULL");
    *out = g_policy;
    return 0;
}

int ccz_boards_start(uint8_t *d_boards, int n, ccz_stream_t s) {
    if (n < 0 || (n > 0 && !d_boards)) return fail(-1, "ccz_boards_start: bad arguments");
    if (int rc = ensure_device()) return rc;
    if (n == 0) return 0;
    const int threads = 256, total = n * 6;
    ccz::boards_start_kernel<<<(total + threads - 1) / threads, threads, 0, s>>>(d_boards, n);
    return check_launch("boards_start_kernel");
}

int ccz_movegen_encode(const uint8_t *d_boards, int n, int16_t *d_move_ids, int16_t *d_counts, uint8_t *d_flags,
                       void *d_planes_bf16, ccz_stream_t s) {
    if (n < 0) return fail(-1, "ccz_movegen_encode: n < 0");
    if (n == 0) return 0;
    if (!d_boards || !d_move_ids || !d_counts || !d_flags) return fail(-1, "ccz_movegen_encode: NULL pointer");
    if (((uintptr_t)d_boards & 15) || ((uintptr_t)d_move_ids & 7) || ((uintptr_t)d_planes_bf16 & 15))
        return fail(-1, "ccz_movegen_encode: boards/planes must be 16-byte, move_ids 8-byte aligned");
    if (int rc = ensure_device()) return rc;
    const int n_quads = (n + 3) / 4;
    int grid = (n_quads + ccz::MG_WARPS - 1) / ccz::MG_WARPS;
    const int cap = sm_count() * CCZ_MG_MIN_BLOCKS; // one resident wave; warps claim quads dynamically
    if (grid > cap) grid = cap;
    static unsigned int *claim_base[64] = {nullptr};
    static unsigned launch_no = 0;
    int dev = 0;
    CCZ_CUDA(cudaGetDevice(&dev));
    if (!claim_base[dev]) {
        // static smem (tables + per-warp scratch) wants the full shared-memory carve-out
        cudaFuncSetAttribute(ccz::movegen_encode_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        cudaFuncSetAttribute(ccz::movegen_encode_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        CCZ_CUDA(cudaGetSymbolAddress(reinterpret_cast<void **>(&claim_base[dev]), ccz::d_mg_counter));
    }
    unsigned int *claim = claim_base[dev] + (launch_no++ % ccz::MG_COUNTER_SLOTS);
    CCZ_CUDA(cudaMemsetAsync(claim, 0, sizeof(unsigned int), s));
    if (g_policy_is_default)
        ccz::movegen_encode_kernel<false><<<grid, ccz::MG_WARPS * 32, 0, s>>>(d_boards, n, d_move_ids, d_counts, d_flags,
                                                                             static_cast<uint32_t *>(d_planes_bf16), claim);
    else // a non-default generation order: the same kernel + a warp sort of each legal list (ccz_set_order_policy)
        ccz::movegen_encode_kernel<true><<<grid, ccz::MG_WARPS * 32, 0, s>>>(d_boards, n, d_move_ids, d_counts, d_flags,
                                                                            static_cast<uint32_t *>(d_planes_bf16), claim);
    return check_launch("movegen_encode_kernel");
}

int ccz_board_keys_init(const uint8_t *d_boards, int n, uint64_t *d_keys, ccz_stream_t s) {
    if (n < 0 || (n > 0 && (!d_boards || !d_keys))) return fail(-1, "ccz_board_keys_init: bad arguments");
    if (int rc = ensure_device()) return rc;
    if (n == 0) return 0;
    CCZ_CUDA(cudaMemsetAsync(d_keys, 0xFF, (size_t)n * ccz::KEY_WINDOW * sizeof(uint64_t), s));
    ccz::board_keys_init_kernel<<<warps_grid(n), ccz::MCTS_WARPS * 32, 0, s>>>(d_boards, n, d_keys);
    return check_launch("board_keys_init_kernel");
}

int ccz_board_push(uint8_t *d_boards, const int16_t *d_move_ids, int n, uint64_t *d_keys, ccz_stream_t s) {
    if (n < 0 || (n > 0 && (!d_boards || !d_move_ids))) return fail(-1, "ccz_board_push: bad arguments");
    if (int rc = ensure_device()) return rc;
    if (n == 0) return 0;
    ccz::board_push_kernel<<<warps_grid(n), ccz::MCTS_WARPS * 32, 0, s>>>(d_boards, d_move_ids, n, d_keys);
    return check_launch("board_push_kernel");
}

int ccz_mcts_pool_init(const ccz_arena *a, ccz_stream_t s) {
    if (int rc = check_arena(a)) return rc;
    if (int rc = ensure_device()) return rc;
    const int n_free = a->n_pages - a->n_games;
    int blocks = (n_free + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > 1024) blocks = 1024;
    ccz::mcts_pool_init_kernel<<<blocks, 256, 0, s>>>(*a);
    if (int rc = check_launch("mcts_pool_init_kernel")) return rc;
    ccz::mcts_games_init_kernel<<<warps_grid(a->n_games), ccz::MCTS_WARPS * 32, 0, s>>>(*a);
    return check_launch("mcts_games_init_kernel");
}

int ccz_mcts_reset(const ccz_arena *a, const uint8_t *d_mask, ccz_stream_t s) {
    if (int rc = check_arena(a)) return rc;
    if (int rc = ensure_device()) return rc;
    ccz::mcts_reset_kernel<<<warps_grid(a->n_games), ccz::MCTS_WARPS * 32, 0, s>>>(*a, d_mask);
    return check_launch("mcts_reset_kernel");
}

int ccz_mcts_reserve(const ccz_arena *a, int pages_per_game, ccz_stream_t s) {
    if (int rc = check_arena(a)) return rc;
    if (pages_per_game < 1) return fail(-1, "ccz_mcts_reserve: pages_per_game < 1");
    if ((long long)a->n_games * (pages_per_game + 1) > a->n_pages || pages_per_game + 1 > a->max_pages)
        return fail(-1, "ccz_mcts_reserve: the pool cannot hold pages_per_game + 1 pages for every game");
    if (int rc = ensure_device()) return rc;
    ccz::mcts_reserve_kernel<<<warps_grid(a->n_games), ccz::MCTS_WARPS * 32, 0, s>>>(*a, pages_per_game);
    return check_launch("mcts_reserve_kernel");
}

int ccz_mcts_migrate(const ccz_arena *src, const ccz_arena *dst, ccz_stream_t s) {
    if (int rc = check_arena(src)) return rc;
    if (int rc = check_arena(dst)) return rc;
    if (src->n_games != dst->n_games) return fail(-1, "ccz_mcts_migrate: n_games differs");
    if (src->d_nodes == dst->d_nodes || src->d_pool_ctl == dst->d_pool_ctl)
        return fail(-1, "ccz_mcts_migrate: src and dst must be distinct arenas");
    if (int rc = ensure_device()) return rc;
    ccz::mcts_migrate_kernel<<<warps_grid(src->n_games), ccz::MCTS_WARPS * 32, 0, s>>>(*src, *dst);
    return check_launch("mcts_migrate_kernel");
}

int ccz_mcts_select(const ccz_arena *a, float c_puct, uint8_t *d_leaf_boards, int32_t *d_leaf_nodes,
                    ccz_stream_t s) {
    if (int rc = check_arena(a)) return rc;
    if (!d_leaf_boards || !d_leaf_nodes) return fail(-1, "ccz_mcts_select: NULL output");
    if (int rc = ensure_device()) return rc;
    // default: the child runs are staged in shared memory by one TMA bulk copy per level; CCZ_SELECT_STAGED=0 loads them
    // straight into registers instead -- a measurement switch, both variants give identical results (DESIGN.md, K3)
    static const bool staged = [] { const char *e = std::getenv("CCZ_SELECT_STAGED"); return !(e && e[0] == '0'); }();
    if (staged)
        ccz::mcts_select_kernel<true><<<warps_grid(a->n_games), ccz::MCTS_WARPS * 32, 0, s>>>(*a, c_puct, d_leaf_boards,
                                                                                             d_leaf_nodes);
    else
        ccz::mcts_select_kernel<false><<<warps_grid(a->n_games), ccz::MCTS_WARPS * 32, 0, s>>>(*a, c_puct, d_leaf_boards,
                                                                                              d_leaf_nodes);
    return check_launch("mcts_select_kernel");
}

int ccz_mcts_expand_backup(const ccz_arena *a, const int32_t *d_leaf_nodes, const float *d_policy, int policy_kind,
                           const float *d_values, const int16_t *d_move_ids, const int16_t *d_counts,
                           const uint8_t *d_flags, ccz_stream_t s) {
    if (int rc = check_arena(a)) return rc;
    if (!d_leaf_nodes || !d_policy || !d_values || !d_move_ids || !d_counts || !d_flags)
        return fail(-1, "ccz_mcts_expand_backup: NULL pointer");
    if (policy_kind != CCZ_POLICY_PROBS && policy_kind != CCZ_POLICY_LOGITS)
        return fail(-1, "ccz_mcts_expand_backup: unknown policy_kind");
    if (int rc = ensure_device()) return rc;
    ccz::mcts_expand_backup_kernel<<<warps_grid(a->n_games), ccz::MCTS_WARPS * 32, 0, s>>>(
        *a, d_leaf_nodes, d_policy, policy_kind, d_values, d_move_ids, d_counts, d_flags);
    return check_launch("mcts_expand_backup_kernel");
}

int ccz_mcts_root_visits(const ccz_arena *a, int16_t *d_acts, int32_t *d_visits, int16_t *d_counts,
                         ccz_stream_t s) {
    if (int rc = check_arena(a)) return rc;
    if (!d_acts || !d_visits || !d_counts) return fail(-1, "ccz_mcts_root_visits: NULL output");
    if (int rc = ensure_device()) return rc;
    ccz::mcts_root_visits_kernel<<<warps_grid(a->n_games), ccz::MCTS_WARPS * 32, 0, s>>>(*a, d_acts, d_visits,
                                                                                        d_counts);
    return check_launch("mcts_root_visits_kernel");
}

int ccz_mcts_advance(const ccz_arena *a, const int16_t *d_chosen, ccz_stream_t s) {
    if (int rc = check_arena(a)) return rc;
    if (!d_chosen) return fail(-1, "ccz_mcts_advance: NULL chosen");
    if (int rc = ensure_device()) return rc;
    // pop-only kernel (compaction into fresh pages), then push-only kernel (old pages back to the ring)
    ccz::mcts_advance_compact_kernel<<<warps_grid(a->n_games), ccz::MCTS_WARPS * 32, 0, s>>>(*a, d_chosen);
    if (int rc = check_launch("mcts_advance_compact_kernel")) return rc;
    ccz::mcts_advance_release_kernel<<<warps_grid(a->n_games), ccz::MCTS_WARPS * 32, 0, s>>>(*a);
    return check_launch("mcts_advance_release_kernel");
}

int ccz_replay_pack(const uint8_t *d_hist_boards, const uint8_t *d_turn_plane, const int16_t *d_acts,
                    const double *d_probs, const int16_t *d_counts, int n, void *d_states_f16, double *d_pi,
                    ccz_stream_t s) {
    if (n < 0) return fail(-1, "ccz_replay_pack: n < 0");
    if (n == 0) return 0;
    if (!d_hist_boards || !d_turn_plane || !d_acts || !d_probs || !d_counts || !d_states_f16 || !d_pi)
        return fail(-1, "ccz_replay_pack: NULL pointer");
    if (int rc = ensure_device()) return rc;
    const long long words = 2ll * n * ccz::WORDS_PER_POS;
    const int threads = 256;
    const long long blocks = (words + threads - 1) / threads;
    if (blocks > 0x7fffffffll) return fail(-1, "ccz_replay_pack: n too large");
    ccz::replay_states_kernel<<<(unsigned)blocks, threads, 0, s>>>(d_hist_boards, d_turn_plane, n,
                                                                   static_cast<uint32_t *>(d_states_f16));
    if (int rc = check_launch("replay_states_kernel")) return rc;
    CCZ_CUDA(cudaMemsetAsync(d_pi, 0, (size_t)2 * n * ccz::N_ACTIONS * sizeof(double), s));
    ccz::replay_pi_kernel<<<(n * 32 + threads - 1) / threads, threads, 0, s>>>(d_acts, d_probs, d_counts, n, d_pi);
    return check_launch("replay_pi_kernel");
}

}  // extern "C"

namespace {

// d_count == nullptr: n_boards boards.  Otherwise n_boards is the capacity the tensor maps are encoded for and the
// kernel convolves min(*d_count, n_boards) boards.
int conv3x3_c256_impl(const char *name, const void *d_x, const void *d_w, const float *d_bias, const void *d_skip, void *d_y,
                      int n_boards, const int32_t *d_count, int variant, ccz_stream_t s) {
    namespace cv = ccz::conv;
    std::string e_name(name);
    auto bad = [&](int code, const char *what) { return fail(code, (e_name + ": " + what).c_str()); };
    if (n_boards < 0) return bad(-1, "n_boards < 0");
    if (n_boards == 0) return 0;
    if (!d_x || !d_w || !d_bias || !d_y) return bad(-1, "NULL pointer");
    if (d_y == d_x) return bad(-1, "output must not alias the input (halo reads)");
    if (variant < 0 || variant >= 128) return bad(-1, "bad variant");
    // variant: 0 = default.  bits 0-1 CTA group (1 / 2), bit 2 = no tail split, bits 3-4 = traffic experiment
    // (skips loads, WRONG results), bits 5-6 = log2(CTA pairs per cluster sharing a weight stage)
    int cta_group = variant & 3;
    const int tail_split = !(variant & 4), dbg = (variant >> 3) & 3;
    int pairs = 1 << ((variant >> 5) & 3);
#ifndef CCZ_CONV_EXPERIMENTS
    if (dbg) return bad(-1, "the load-skipping measurement variants need a -DCCZ_CONV_EXPERIMENTS build");
#endif
    if (variant == 0) { cta_group = 2; pairs = CCZ_CONV_DEFAULT_PAIRS; }
    if (cta_group == 0) cta_group = 2;
    if (cta_group == 3 || pairs > 4 || (cta_group == 1 && pairs != 1))
        return bad(-1, "unsupported variant (cta_group 1|2, pairs 1|2|4, pairs > 1 needs cta_group 2)");
    if (((uintptr_t)d_x | (uintptr_t)d_w | (uintptr_t)d_y | (uintptr_t)d_skip) & 15)
        return bad(-1, "pointers must be 16-byte aligned");
    static cv::Driver drv;
    if (const char *err = cv::driver_init(drv)) return fail(-3, err);
    const long long m = (long long)n_boards * cv::BOARD_HW;
    const int rows_per_tile = cv::BM * cta_group * pairs;
    const int n_tiles = (int)((m + rows_per_tile - 1) / rows_per_tile);
    CUtensorMap tx, tw, ts, ty;
    if (!cv::encode_im2col(drv, &tx, d_x, n_boards)) return bad(-3, "cuTensorMapEncodeIm2col(x) failed");
    if (!cv::encode_rows(drv, &tw, d_w, cv::BN, 9 * cv::C, (uint32_t)(cv::BN / cta_group / pairs)))
        return bad(-3, "cuTensorMapEncodeTiled(w) failed");
    if (!cv::encode_rows(drv, &ty, d_y, (uint64_t)m, cv::C, cv::BM)) return bad(-3, "cuTensorMapEncodeTiled(y) failed");
    if (d_skip) {
        if (!cv::encode_rows(drv, &ts, d_skip, (uint64_t)m, cv::C, cv::BM)) return bad(-3, "cuTensorMapEncodeTiled(skip) failed");
    } else {
        ts = ty;
    }
    cudaError_t e;
#define CCZ_CONV_LAUNCH_C(CG, PAIRS, CNT)                                                                                  \
    (d_skip ? cv::launch_variant<CG, PAIRS, true, CNT>(tx, tw, ts, ty, d_bias, n_tiles, tail_split, dbg, d_count, n_boards, s) \
            : cv::launch_variant<CG, PAIRS, false, CNT>(tx, tw, ts, ty, d_bias, n_tiles, tail_split, dbg, d_count, n_boards, s))
#define CCZ_CONV_LAUNCH(CG, PAIRS) (d_count ? CCZ_CONV_LAUNCH_C(CG, PAIRS, true) : CCZ_CONV_LAUNCH_C(CG, PAIRS, false))
    if (cta_group == 1) e = CCZ_CONV_LAUNCH(1, 1);
    else if (pairs == 1) e = CCZ_CONV_LAUNCH(2, 1);
    else if (pairs == 2) e = CCZ_CONV_LAUNCH(2, 2);
    else e = CCZ_CONV_LAUNCH(2, 4);
#undef CCZ_CONV_LAUNCH
#undef CCZ_CONV_LAUNCH_C
    if (e != cudaSuccess) return fail(-2, "conv3x3_c256_kernel launch", e);
    return 0;
}

int stem_lookup_impl(const char *name, const uint8_t *d_boards, int n, const int32_t *d_count, const void *d_table,
                     const float *d_bias_turn, void *d_y, ccz_stream_t s) {
    namespace st = ccz::stem;
    std::string e_name(name);
    if (n < 0) return fail(-1, (e_name + ": n < 0").c_str());
    if (n == 0) return 0;
    if (!d_boards || !d_table || !d_bias_turn || !d_y) return fail(-1, (e_name + ": NULL pointer").c_str());
    if (((uintptr_t)d_boards & 3) || (((uintptr_t)d_table | (uintptr_t)d_bias_turn | (uintptr_t)d_y) & 15))
        return fail(-1, (e_name + ": pointers must be 16-byte aligned (boards 4-byte)").c_str());
    static int n_sm_dev[64] = {0};
    int dev = 0;
    CCZ_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return fail(-1, (e_name + ": device index out of range").c_str());
    int &n_sm = n_sm_dev[dev];
    if (!n_sm) {
        CCZ_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
        CCZ_CUDA(cudaFuncSetAttribute(st::stem_lookup_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, st::SMEM_BYTES));
        CCZ_CUDA(cudaFuncSetAttribute(st::stem_lookup_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, st::SMEM_BYTES));
    }
    int blocks = 2 * n_sm; // two resident CTAs (92 KB of tables each) per SM
    const int need = (n + st::WARPS - 1) / st::WARPS;
    if (blocks > need) blocks = need;
    const uint4 *tab = static_cast<const uint4 *>(d_table);
    const float4 *bt = reinterpret_cast<const float4 *>(d_bias_turn);
    uint4 *y = static_cast<uint4 *>(d_y);
    if (d_count)
        st::stem_lookup_kernel<true><<<blocks, st::WARPS * 32, st::SMEM_BYTES, s>>>(d_boards, n, tab, bt, y, d_count);
    else
        st::stem_lookup_kernel<false><<<blocks, st::WARPS * 32, st::SMEM_BYTES, s>>>(d_boards, n, tab, bt, y, nullptr);
    return check_launch("stem_lookup_kernel");
}

int heads_pack_impl(const char *name, const void *d_h, int n, const int32_t *d_rows, void *d_operands, int row_elems, int value_off,
                    ccz_stream_t s) {
    namespace hd = ccz::heads;
    std::string e_name(name);
    if (n < 0) return fail(-1, (e_name + ": n < 0").c_str());
    if (n == 0) return 0;
    if (!d_h || !d_operands) return fail(-1, (e_name + ": NULL pointer").c_str());
    if (((uintptr_t)d_h & 15) || ((uintptr_t)d_operands & 3) || ((uintptr_t)d_rows & 3))
        return fail(-1, (e_name + ": h must be 16-byte, operands and rows 4-byte aligned").c_str());
    if ((row_elems & 1) || (value_off & 1) || value_off < hd::N_POLICY * hd::HW || row_elems < value_off + hd::N_VALUE * hd::HW)
        return fail(-1, (e_name + ": operand row must hold 1530 policy + 630 value elements at even offsets").c_str());
    hd::heads_pack_kernel<<<n, hd::THREADS, 0, s>>>(static_cast<const uint4 *>(d_h), static_cast<uint32_t *>(d_operands), n,
                                                  row_elems / 2, value_off / 2, d_rows);
    return check_launch("heads_pack_kernel");
}

} // namespace

extern "C" {

int ccz_conv3x3_c256(const void *d_x, const void *d_w, const float *d_bias, const void *d_skip, void *d_y, int n_boards,
                     int variant, ccz_stream_t s) {
    return conv3x3_c256_impl("ccz_conv3x3_c256", d_x, d_w, d_bias, d_skip, d_y, n_boards, nullptr, variant, s);
}

int ccz_conv3x3_c256_count(const void *d_x, const void *d_w, const float *d_bias, const void *d_skip, void *d_y, int capacity,
                           const int32_t *d_n_boards, int variant, ccz_stream_t s) {
    if (!d_n_boards) return fail(-1, "ccz_conv3x3_c256_count: d_n_boards is NULL");
    return conv3x3_c256_impl("ccz_conv3x3_c256_count", d_x, d_w, d_bias, d_skip, d_y, capacity, d_n_boards, variant, s);
}

int ccz_conv3x3_plan(int n_boards, int variant, int resident_clusters, int32_t *out) {
    namespace cv = ccz::conv;
    if (n_boards <= 0 || resident_clusters <= 0 || !out || variant < 0 || variant >= 128)
        return fail(-1, "ccz_conv3x3_plan: bad argument");
    int cta_group = variant & 3, pairs = 1 << ((variant >> 5) & 3);
    if (variant == 0) { cta_group = 2; pairs = CCZ_CONV_DEFAULT_PAIRS; }
    if (cta_group == 0) cta_group = 2;
    if (cta_group == 3 || pairs > 4 || (cta_group == 1 && pairs != 1)) return fail(-1, "ccz_conv3x3_plan: unsupported variant");
    const long long m = (long long)n_boards * cv::BOARD_HW;
    const int rows_per_tile = cv::BM * cta_group * pairs;
    const int n_tiles = (int)((m + rows_per_tile - 1) / rows_per_tile);
    const cv::Plan pl = cv::plan_items(n_tiles, resident_clusters, !(variant & 4));
    out[0] = rows_per_tile; out[1] = n_tiles; out[2] = pl.n_items; out[3] = pl.n_full; out[4] = pl.split_log2; out[5] = pl.clusters;
    return 0;
}

int ccz_stem_lookup(const uint8_t *d_boards, int n, const void *d_table, const float *d_bias_turn, void *d_y, ccz_stream_t s) {
    return stem_lookup_impl("ccz_stem_lookup", d_boards, n, nullptr, d_table, d_bias_turn, d_y, s);
}

int ccz_stem_lookup_count(const uint8_t *d_boards, int capacity, const int32_t *d_n_boards, const void *d_table, const float *d_bias_turn,
                          void *d_y, ccz_stream_t s) {
    if (!d_n_boards) return fail(-1, "ccz_stem_lookup_count: d_n_boards is NULL");
    return stem_lookup_impl("ccz_stem_lookup_count", d_boards, capacity, d_n_boards, d_table, d_bias_turn, d_y, s);
}

int ccz_heads_pack(const void *d_h, int n, void *d_operands, int row_elems, int value_off, ccz_stream_t s) {
    return heads_pack_impl("ccz_heads_pack", d_h, n, nullptr, d_operands, row_elems, value_off, s);
}

int ccz_heads_pack_rows(const void *d_h, int n, const int32_t *d_rows, void *d_operands, int row_elems, int value_off, ccz_stream_t s) {
    if (!d_rows) return fail(-1, "ccz_heads_pack_rows: d_rows is NULL");
    return heads_pack_impl("ccz_heads_pack_rows", d_h, n, d_rows, d_operands, row_elems, value_off, s);
}

int ccz_leaf_unique(const uint8_t *d_boards, int n, int32_t *d_rows, uint8_t *d_uniq_boards, int32_t *d_n_unique,
                    unsigned long long *d_unique_total, ccz_stream_t s) {
    namespace dd = ccz::dedup;
    if (n < 0 || n > dd::MAX_BOARDS) return fail(-1, "ccz_leaf_unique: n must be 0..16384");
    if (!d_n_unique) return fail(-1, "ccz_leaf_unique: d_n_unique is NULL");
    if (n == 0) {
        CCZ_CUDA(cudaMemsetAsync(d_n_unique, 0, sizeof(int32_t), s));
        return 0;
    }
    if (!d_boards || !d_rows || !d_uniq_boards) return fail(-1, "ccz_leaf_unique: NULL pointer");
    if (((uintptr_t)d_boards | (uintptr_t)d_uniq_boards) & 15) return fail(-1, "ccz_leaf_unique: boards must be 16-byte aligned");
    if (d_uniq_boards == d_boards) return fail(-1, "ccz_leaf_unique: uniq_boards must not alias boards");
    static bool attr_set[64] = {false};
    int dev = 0;
    CCZ_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return fail(-1, "ccz_leaf_unique: device index out of range");
    if (!attr_set[dev]) {
        CCZ_CUDA(cudaFuncSetAttribute(dd::leaf_unique_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dd::smem_bytes(dd::MAX_BOARDS)));
        attr_set[dev] = true;
    }
    dd::leaf_unique_kernel<<<1, dd::THREADS, dd::smem_bytes(n), s>>>(d_boards, n, d_rows, d_uniq_boards, d_n_unique, d_unique_total);
    return check_launch("leaf_unique_kernel");
}

} // extern "C"
