/*
 * ccz_b200.h -- C ABI of the B200-native Xiangqi self-play hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference (Symb0x76/ChineseChessZero) is
 * pure Python and has no FFI; its seams are Python call signatures.  Each entry point below
 * replaces the arithmetic behind one of those seams and is what a ctypes binding in the
 * reference's own files would call (INTEGRATION.md shows the stubs):
 *
 *   ccz_movegen_encode      <- board.legal_moves + move_action2move_id (net.py:154-157),
 *                              decode_board + plane assembly (tools.py:74-106, net.py:160-177),
 *                              is_game_over / is_tie predicates (tools.py:109-123, mcts.py:116)
 *   ccz_board_push          <- board.push (game.py:201, mcts.py:111)
 *   ccz_mcts_select         <- Node.select / puct_value + path pushes (mcts.py:41-61,105-111)
 *   ccz_mcts_expand_backup  <- exp(log_p)[legal] gather (net.py:202-203), Node.expand
 *                              (mcts.py:31-39), terminal values (mcts.py:116-126),
 *                              update_recursive (mcts.py:63-78)
 *   ccz_mcts_root_visits    <- root child visit read-out (mcts.py:163-164)
 *   ccz_mcts_advance        <- MCTS.update_with_move (mcts.py:168-178) + board.push of the move
 *   ccz_replay_pack         <- CollectPipeline.preprocess / flip_data (collect.py:64-131)
 *
 * Conventions: every pointer named d_* is a DEVICE pointer owned by the caller (torch tensors
 * on the Python side); the library never allocates device memory, never synchronises, and
 * enqueues all work on the given stream.  Return value 0 = OK, negative = error, message via
 * ccz_last_error().  Thread-compatible: one host thread per device at a time.
 */
#ifndef CCZ_B200_H
#define CCZ_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st *ccz_stream_t; /* == cudaStream_t */

#define CCZ_BOARD_BYTES 96   /* sq[90], turn, halfmove clock, repetition count, 3 pad */
#define CCZ_MAX_MOVES 128    /* >= max legal moves of any Xiangqi position (119) */
#define CCZ_N_ACTIONS 2086   /* tools.py:172-272 */
#define CCZ_PLANE_ELEMS 10710 /* 17*7*10*9, net.py:12-13 */
#define CCZ_KEY_WINDOW 128   /* position keys kept since the last capture */

/* flag byte written by ccz_movegen_encode */
#define CCZ_FLAG_CHECK 1        /* side to move is in check */
#define CCZ_FLAG_NOMOVES 2      /* no legal move: checkmate (with CHECK) or stalemate */
#define CCZ_FLAG_INSUFFICIENT 4 /* board.is_insufficient_material() */
#define CCZ_FLAG_FOURFOLD 8     /* board.is_fourfold_repetition() */
#define CCZ_FLAG_SIXTY 16       /* board.is_sixty_moves() */
#define CCZ_FLAG_TIE_MASK (CCZ_FLAG_INSUFFICIENT | CCZ_FLAG_FOURFOLD | CCZ_FLAG_SIXTY)

/* per-game status bits (ccz_arena.d_status); sticky until the slot is reset for a new game */
#define CCZ_STATUS_EXPAND_FAILED 1 /* a leaf stayed unexpanded: the page pool was exhausted (last resort) */
#define CCZ_STATUS_TREE_DROPPED 2  /* the kept sub-tree was dropped to free pool pages (reserve / advance) */
#define CCZ_STATUS_NODE_OVERFLOW CCZ_STATUS_EXPAND_FAILED /* round-1 name */

/* kinds of policy input accepted by ccz_mcts_expand_backup */
#define CCZ_POLICY_PROBS 0  /* fp32 probabilities, gathered as-is (bit-exact path) */
#define CCZ_POLICY_LOGITS 1 /* fp32 logits; softmax over all 2086 fused into the gather */

/* special values of d_chosen[g] in ccz_mcts_advance */
#define CCZ_ADVANCE_NEW_GAME (-1)  /* start position, fresh root */
#define CCZ_ADVANCE_DROP_TREE (-2) /* keep the position, fresh root */
#define CCZ_ADVANCE_KEEP (-3)      /* keep the position and the tree (a slot that does not move) */

/* A tree node is two records so that one 16-byte load per lane brings everything PUCT needs of a
 * child (N, Q, P) plus the link to ITS children, and the cold fields stay out of that stream. */
typedef struct {
    int32_t visits;      /* N   (mcts.py:16) */
    float value;         /* Q   (mcts.py:15), fp32 incremental mean */
    float prior;         /* P   (mcts.py:17) */
    int32_t first_child; /* pool index of the first child, -1 if none */
} ccz_node;              /* 16 B */
typedef struct {
    int32_t parent;  /* pool index, -1 for the root */
    int16_t move;    /* action id that leads to this node */
    int16_t n_child; /* 0 = leaf (mcts.py:19-23) */
} ccz_link;          /* 8 B */

/* control words of the page pool (ccz_arena.d_pool_ctl, int64 each) */
#define CCZ_CTL_HEAD 0          /* pages popped from the free ring so far */
#define CCZ_CTL_TAIL 1          /* pages pushed to the free ring so far; free = TAIL - HEAD */
#define CCZ_CTL_EXPAND_FAILED 2 /* cumulative count of leaves left unexpanded (never cleared by reset / advance) */
#define CCZ_CTL_TREES_DROPPED 3 /* cumulative count of sub-trees dropped (never cleared by reset / advance) */
#define CCZ_CTL_MIN_FREE 4      /* low-water mark of free pages */
#define CCZ_CTL_WORDS 8

/* Pooled MCTS arena: `n_games` independent trees whose nodes come from ONE pool of `n_pages` pages
 * of 2^page_shift nodes (the reference's tree, mcts.py:31-39, has no capacity: a game that keeps a
 * large sub-tree borrows pages that games with small trees do not need).  A node is addressed by
 * its pool index; the children of a node are the contiguous slots [first_child, first_child +
 * n_child) -- always inside one page -- in cchess generation order (the reference's
 * insertion-ordered dict, mcts.py:37-39).  Each game bump-allocates child runs in its current page
 * and pops a new page from the free ring when a run does not fit; ccz_mcts_advance compacts the
 * kept sub-tree into fresh pages and returns the old ones.  The page lists ping-pong between the
 * two halves of d_page_list (d_list_sel[g] names the live half). */
typedef struct {
    int32_t n_games;
    int32_t n_pages;    /* pool size in pages; n_pages << page_shift < 2^31 */
    int32_t page_shift; /* 7..16: a page must hold one child run (<= 128 nodes) */
    int32_t max_pages;  /* page-list capacity of one game */
    ccz_node *d_nodes;  /* [n_pages << page_shift] */
    ccz_link *d_links;  /* [n_pages << page_shift] */
    int32_t *d_free_ring;   /* [n_pages] page ids; live entries are HEAD .. TAIL-1 (mod n_pages) */
    int64_t *d_pool_ctl;    /* [CCZ_CTL_WORDS] */
    int32_t *d_page_list;   /* [2, n_games, max_pages] pages owned by each game */
    int32_t *d_page_fill;   /* [n_games, max_pages] scratch of ccz_mcts_advance: nodes used in each new page */
    int32_t *d_n_pages;     /* [n_games] entries of the live page list */
    int32_t *d_n_pages_new; /* [n_games] scratch of ccz_mcts_advance */
    int32_t *d_list_sel;    /* [n_games] 0 / 1: live half of d_page_list */
    int32_t *d_alloc_page;  /* [n_games] page the next child run is carved from */
    int32_t *d_alloc_off;   /* [n_games] first unused slot of that page */
    int32_t *d_root;        /* [n_games] pool index of the root node */
    int32_t *d_n_nodes;     /* [n_games] live nodes of the tree */
    int32_t *d_status;      /* [n_games] CCZ_STATUS_* bits */
    uint8_t *d_root_boards; /* [n_games, 96] position at the root */
    uint64_t *d_root_keys;  /* [n_games, 128] position keys since the last capture; entry
                               `clock` is the root position itself */
} ccz_arena;

int ccz_version(void);
const char *ccz_last_error(void);

/* Upload the constant tables (action table, position-key table) to the current device.  Called
 * implicitly by every entry point; exposed so start-up cost can be kept out of timed regions. */
int ccz_init(void);

/* Host copies of the action table: id_of[from*90+to] (-1 = not an action), from/to square of
 * each id.  Any pointer may be NULL. */
int ccz_action_table(int16_t *id_of, uint8_t *from_of, uint8_t *to_of);

/* Generation order of `board.legal_moves` (net.py:154-157), which is the insertion order of the tree's
 * children and so decides every PUCT tie-break (mcts.py:59-61).  cchess is not pinned by the reference and
 * not installable where this library is built, so the order is a policy: legal moves come out sorted by
 * (class_rank[piece type] -- the king ahead of everything while in check if check_king_first --, from-square,
 * capture flag, to-square).  The default -- non-pawn pieces by
 * from-square descending, destinations descending, then the pawns likewise (python-chess lineage) -- is the
 * order the kernel generates natively; any other policy adds a warp sort per position.  The oracle mirrors
 * the same struct (xq_set_order_policy); scripts/pin_cchess.py derives the policy from a real cchess. */
typedef struct {
    uint8_t class_rank[8];   /* index = piece type 1..7 (PAWN CANNON ROOK KNIGHT BISHOP ADVISOR KING): lower ranks first */
    uint8_t from_descending; /* 1: larger from-square first */
    uint8_t to_descending;   /* 1: larger to-square first */
    uint8_t capture_mode;    /* 0: destination order only; 1: a piece's quiet moves before its captures; 2: captures first */
    uint8_t check_king_first; /* 1: when the side to move is in check its king moves come first, then the other pieces by
                                 class (python-chess generates evasions that way); 0: same order in and out of check */
} ccz_order_policy;

/* NULL = the default policy.  Host-side state of the library: takes effect for every later call on any device
 * (do not change it while work that depends on the order is in flight). */
int ccz_set_order_policy(const ccz_order_policy *p);
int ccz_get_order_policy(ccz_order_policy *out);

/* Fill `n` board records with the start position (device memory). */
int ccz_boards_start(uint8_t *d_boards, int n, ccz_stream_t s);

/* Legal moves (ordered, as action ids, -1 padded), count, flag byte and -- unless d_planes is
 * NULL -- the dense bf16 (17,7,10,9) search-time net input for each of n board records. */
int ccz_movegen_encode(const uint8_t *d_boards, int n, int16_t *d_move_ids /*[n,128]*/,
                       int16_t *d_counts /*[n]*/, uint8_t *d_flags /*[n]*/,
                       void *d_planes_bf16 /*[n,10710] or NULL*/, ccz_stream_t s);

/* Apply move id d_move_ids[i] to board record i (ids < 0 leave the board untouched).  If
 * d_keys is not NULL it is the [n,128] key window of each board and is updated so that the
 * record's repetition count stays exact. */
int ccz_board_push(uint8_t *d_boards, const int16_t *d_move_ids, int n, uint64_t *d_keys,
                   ccz_stream_t s);

/* Initialise the [n,128] key windows of history-less board records (entry `clock` = the key of
 * the record, earlier entries = a sentinel that matches nothing). */
int ccz_board_keys_init(const uint8_t *d_boards, int n, uint64_t *d_keys, ccz_stream_t s);

/* First use of an arena: builds the free ring, hands every game one page and resets every tree to a
 * single unvisited root (Node(None, 1.0), mcts.py:94) over the start position (game.py:148).  The
 * cumulative counters in d_pool_ctl start at zero.  Needs n_pages >= n_games. */
int ccz_mcts_pool_init(const ccz_arena *a, ccz_stream_t s);

/* Reset trees to a single unvisited root over the start position; the pages of the old tree go
 * back to the pool.  d_mask NULL = every game, else only games with d_mask[g] != 0 (slot refill). */
int ccz_mcts_reset(const ccz_arena *a, const uint8_t *d_mask /*[n_games] or NULL*/, ccz_stream_t s);

/* Guarantee, before a search, that every game can grow by `pages_per_game` pages: if the free ring
 * holds fewer than n_games * pages_per_game pages, or a game's page list would overflow, the trees
 * of the games that hold more than their share (n_pages / n_games - pages_per_game) are dropped
 * (fresh root on the same position, CCZ_STATUS_TREE_DROPPED, CCZ_CTL_TREES_DROPPED += 1).  After
 * it no expansion of the following pages_per_game-page search can fail.  Callers that may
 * synchronise grow the pool instead (ccz_mcts_migrate) and never reach the dropping branch. */
int ccz_mcts_reserve(const ccz_arena *a, int pages_per_game, ccz_stream_t s);

/* Move every tree, root position and key window into another (larger) arena of the same n_games;
 * dst must have been initialised with ccz_mcts_pool_init.  Cumulative counters carry over. */
int ccz_mcts_migrate(const ccz_arena *src, const ccz_arena *dst, ccz_stream_t s);

/* One selection pass per game: descend by PUCT from the root to a leaf, replaying the moves.
 * Writes the leaf position and the leaf's pool index. */
int ccz_mcts_select(const ccz_arena *a, float c_puct, uint8_t *d_leaf_boards /*[n,96]*/,
                    int32_t *d_leaf_nodes /*[n]*/, ccz_stream_t s);

/* Expand each leaf (unless terminal) with priors gathered from d_policy[n,2086] and back the
 * leaf value up to the root with alternating sign. */
int ccz_mcts_expand_backup(const ccz_arena *a, const int32_t *d_leaf_nodes, const float *d_policy,
                           int policy_kind, const float *d_values /*[n]*/,
                           const int16_t *d_move_ids, const int16_t *d_counts,
                           const uint8_t *d_flags, ccz_stream_t s);

/* Root children in generation order: action ids (-1 padded), visit counts, count. */
int ccz_mcts_root_visits(const ccz_arena *a, int16_t *d_acts /*[n,128]*/,
                         int32_t *d_visits /*[n,128]*/, int16_t *d_counts /*[n]*/, ccz_stream_t s);

/* Play d_chosen[g] in game g (MCTS.update_with_move, mcts.py:168-178): the chosen child's sub-tree
 * is compacted breadth-first into fresh pages (tree reuse; visit counts and Q carry over), the
 * pages of the rest go back to the pool, the root board and key window advance.
 * CCZ_ADVANCE_NEW_GAME resets game g to the start position with a fresh root,
 * CCZ_ADVANCE_DROP_TREE keeps the position but drops the tree, CCZ_ADVANCE_KEEP leaves the slot
 * as it is; an id that is not a root child
 * gives a fresh root as in the reference (mcts.py:177-178). */
int ccz_mcts_advance(const ccz_arena *a, const int16_t *d_chosen, ccz_stream_t s);

/* Replay densification (collect.py:64-131): for each of n samples scatter the sparse visit
 * distribution into a dense float64 row of 2086 and its file-mirrored twin, and write the
 * (17,7,10,9) float16 state stack and its mirror from 8 board records of history (red planes
 * of slot i -> play i, black planes of slot i -> play 8+i, game.py:23-44). */
int ccz_replay_pack(const uint8_t *d_hist_boards /*[n,8,96]: history slots, most recent first*/,
                    const uint8_t *d_turn_plane /*[n] 1 = ones */, const int16_t *d_acts /*[n,128]*/,
                    const double *d_probs /*[n,128]*/, const int16_t *d_counts, int n,
                    void *d_states_f16 /*[2n,10710]*/, double *d_pi /*[2n,2086]*/, ccz_stream_t s);

/* K9: the residual-tower convolution of Net.forward (net.py:33-41, 82-90) with eval-mode BatchNorm folded
 * in: y = relu(conv3x3_pad1(x, w) + bias [+ skip]) over n_boards boards of 10x9, 256 -> 256 channels.
 * d_x, d_skip, d_y: [n_boards,10,9,256] bf16 (NHWC = torch channels_last); d_w: [256][3][3][256] bf16
 * (out, kh, kw, in = a channels_last [256,256,3,3] weight); d_bias: fp32[256]; d_skip NULL = no skip
 * connection (conv1 of a block), d_skip may alias d_y but d_y must not alias d_x.  tcgen05 implicit GEMM
 * with TMA im2col loads.  variant 0 = the library default; otherwise bits 0-1 = CTA group (1: 128x256 tiles per
 * CTA, 2: CTA pairs on 256x256 tiles), bit 2 = no channel-sliced tail round, bits 5-6 = log2 of the CTA pairs
 * per cluster that share (multicast) one weight stage; bits 3-4 (skip every other weight / activation load:
 * WRONG results, energy-sensitivity measurements only) are rejected unless the library was built with
 * -DCCZ_CONV_EXPERIMENTS. */
int ccz_conv3x3_c256(const void *d_x, const void *d_w, const float *d_bias, const void *d_skip, void *d_y,
                     int n_boards, int variant, ccz_stream_t s);

/* K9 over a board count that lives on the device: the buffers hold `capacity` boards (the tensor maps are encoded
 * for it) and the kernel convolves the first min(*d_n_boards, capacity) of them, planning its work items on the
 * device exactly as ccz_conv3x3_plan does for that count.  Every resident cluster is launched; clusters without an
 * item exit.  Output rows past the count (up to the end of the last tile) hold unspecified values.  Capture-safe: no
 * host synchronisation.  Each board's output is bit-identical to ccz_conv3x3_c256 over the same boards. */
int ccz_conv3x3_c256_count(const void *d_x, const void *d_w, const float *d_bias, const void *d_skip, void *d_y,
                           int capacity, const int32_t *d_n_boards, int variant, ccz_stream_t s);

/* Host-only: the work plan ccz_conv3x3_c256 would launch for n_boards on a device with `resident_clusters`
 * co-resident clusters of the variant's shape (74 CTA pairs on a B200).  out[6] = {pixel rows per cluster tile,
 * cluster tiles, work items, whole-tile items, log2 of the channel slices of the last partial round, clusters
 * launched}.  Work item i < out[3] is tile i over all 256 channels; item out[3] + j is channel slice
 * j % 2^out[4] (256 >> out[4] channels) of tile out[3] + (j >> out[4]); cluster c runs items c, c + out[5], ... */
int ccz_conv3x3_plan(int n_boards, int variant, int resident_clusters, int32_t *out);

/* K10: the stem convolution of Net.forward (conv_block 119->256 + BN + ReLU, net.py:84) for SEARCH-TIME
 * inputs, computed from the board records themselves.  policy_value_fn (net.py:160-177) feeds 7 zero
 * history states + the current one-hot piece planes + a constant turn plane, so each output pixel is
 * bias + at most nine rows of the folded weight tensor:
 *   d_table     bf16 [9 taps][16 piece codes][256]: W[co, channel(code), tap] (codes 0 and 8: zero rows;
 *               code = type | 8*black -> channel 49+type-1 (red) or 105+type-1 (black); tap = kh*3+kw)
 *   d_bias_turn fp32 [2 turn][9 border classes][256]: bias + turn * (sum of the 7 turn-plane weights over the
 *               taps that stay on the board; class = 3*(h==0?0:h==9?2:1) + (w==0?0:w==8?2:1))
 *   d_y         bf16 [n,10,9,256] NHWC, what ccz_conv3x3_c256 consumes. */
int ccz_stem_lookup(const uint8_t *d_boards, int n, const void *d_table, const float *d_bias_turn, void *d_y,
                    ccz_stream_t s);

/* K10 over the first min(*d_n_boards, capacity) boards of d_boards (the count read on the device); output rows
 * past the count are not written. */
int ccz_stem_lookup_count(const uint8_t *d_boards, int capacity, const int32_t *d_n_boards, const void *d_table,
                          const float *d_bias_turn, void *d_y, ccz_stream_t s);

/* K11: ReLU + NHWC -> channel-major packing between the fused 1x1 head convolutions and the FC layers of
 * Net.forward (net.py:94-107).  d_h: bf16 [n*90][32] head-convolution outputs per pixel row (channels 0..16 policy,
 * 17..23 value, bias added, before the ReLU).  d_operands: bf16 [n][row_elems]; row b receives
 * relu(policy) as x.view(-1, 17*90) (net.py:97) at element 0 and relu(value) as x.view(-1, 7*90) (net.py:104) at element
 * value_off; other elements of the row (GEMM K padding) are left untouched. */
int ccz_heads_pack(const void *d_h, int n, void *d_operands, int row_elems, int value_off, ccz_stream_t s);

/* K11 with a row map: operand row b is packed from board d_rows[b] of d_h (each d_rows[b] must be a board of d_h).
 * With ccz_leaf_unique's rows this expands the heads of the distinct leaves back to one operand row per game. */
int ccz_heads_pack_rows(const void *d_h, int n, const int32_t *d_rows, void *d_operands, int row_elems, int value_off,
                        ccz_stream_t s);

/* K12: the distinct positions of a leaf batch.  Identity is bytes 0..90 of the record (squares + side to move, all
 * the search-time net input depends on; boards that differ only in the clock or repetition bytes are one position).
 * d_boards [n,96] -> d_uniq_boards [n,96]: the distinct records in rows 0..U-1 in order of first occurrence (lowest
 * game index), rows >= U untouched; d_rows[g] = the row of game g's position; *d_n_unique = U; d_unique_total
 * (may be NULL) += U.  One launch, no host synchronisation, no allocation (capture-safe); n <= 16384; both board
 * arrays 16-byte aligned and distinct. */
int ccz_leaf_unique(const uint8_t *d_boards, int n, int32_t *d_rows, uint8_t *d_uniq_boards, int32_t *d_n_unique,
                    unsigned long long *d_unique_total, ccz_stream_t s);

#ifdef __cplusplus
}
#endif
#endif /* CCZ_B200_H */
