/*
 * cchess_b200.h -- C ABI of the B200-native batched MCTS self-play engine.
 *
 * The reference (chengstone/cchess-zero) is pure Python and has no FFI; this header is
 * the boundary a maintainer would bind from the reference's Python (ctypes stub in
 * INTEGRATION.md).  Each entry point names the reference code it replaces
 * (file:line relative to the reference tree).
 *
 * Conventions
 *   - every function returns an int status: CZ_OK (0) or a negative CZ_E* code; nothing
 *     throws across the boundary; cz_last_error() gives a thread-local message.
 *   - plain pointers and sizes only.  "host" buffers are ordinary (ideally pinned) host
 *     memory owned by the caller; "dev" pointers are CUDA device pointers owned by the
 *     caller (e.g. torch tensors' data_ptr()).  `stream` is a cudaStream_t passed as void*
 *     (NULL = default stream); asynchronous work is ordered on it.
 *   - boards are 90 bytes, row-major sq = y*9 + x (y = rank 0..9 = row of the reference's
 *     state string, x = file a..i), piece codes 0 = empty, 1..7 = K A R B N P C (red /
 *     upper-case / 'w'), 8..14 = k a r b n p c (black / 'b')  [pieces_order, main.py:208].
 *   - a move is uint16: src_sq | dst_sq << 7.   side: 0 = 'w' (red), 1 = 'b'.
 *   - a handle is bound to one GPU; calls on one handle are not thread-safe.
 */
#ifndef CCHESS_B200_H
#define CCHESS_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CZ_OK 0
#define CZ_EINVAL (-1)   /* bad argument */
#define CZ_ECUDA (-2)    /* CUDA runtime error (see cz_last_error) */
#define CZ_ENOMEM (-3)   /* allocation failed */
#define CZ_EENGINE (-4)  /* a game raised an engine error flag (see cz_engine_counters) */

#define CZ_NSQ 90
#define CZ_NLABEL 2086       /* labels_len, main.py:212 */
#define CZ_MAXCHILD 128      /* upper bound on pseudo-legal moves of one position */
#define CZ_ENC_LEN 1260      /* 9*10*14, main.py:550 */

/* nn input element types accepted by encode / wave */
#define CZ_F32 0
#define CZ_BF16 1
#define CZ_F16 2
#define CZ_BOARD 3           /* wave only: row g = 96 bytes, the side-to-move-canonical board (for cz_net_first_conv) */

/* per-game error flags (cz_engine_counters) */
#define CZ_ERR_NOMOVES 1     /* expanded node with zero legal moves (reference: ValueError from max(), main.py:159) */
#define CZ_ERR_NOLABEL 2     /* move outside the 2086-label table (reference: KeyError, main.py:181) */
#define CZ_ERR_DEPTH 4       /* search path deeper than the path stack */
#define CZ_ERR_ARENA 8       /* tree arena exhausted */
#define CZ_ERR_CHILDREN 16   /* more than CZ_MAXCHILD moves */
#define CZ_ERR_NOCHILD 32    /* move is not a child of an expanded root (reference: KeyError in update_tree, main.py:275) */

const char *cz_last_error(void);
int cz_version(void);

/* ---- move-label codec: create_uci_labels main.py:30-65, label2i 217, unflipped_index 213-214 ---- */
int cz_labels(char *out /* [2086*4] host, no terminators */);
int cz_label_index(int src_sq, int dst_sq);           /* >= 0 label index, -1 if not a label */
int cz_unflipped_index(int32_t *out /* [2086] host */);

/* ---- state strings: GameBoard.board_to_pos_name main.py:705-714, re-compression 691-699 ---- */
int cz_from_state(const char *state, uint8_t *board /* [90] */);
int cz_to_state(const uint8_t *board, char *out /* >= 100 bytes */);

/* ---- stateless, batched rules; HOST buffers, computed on the GPU (copies included) ----
 * cz_legal_moves_batch  replaces GameBoard.get_legal_moves            main.py:743-1109 (same ORDER)
 * cz_apply_moves_batch  replaces GameBoard.sim_do_action + is_kill_move  main.py:647-702, 219-227
 * cz_encode_batch       replaces MCTS_tree.generate_inputs (try_flip + state_to_positions, incl. the
 *                       rank*9+file indexing of the [9][10][14] tensor) main.py:531-574            */
int cz_legal_moves_batch(int device, const uint8_t *boards /* [n][90] */, const uint8_t *sides /* [n] */, int n,
                         uint16_t *moves /* [n][128] */, int32_t *counts /* [n] */);
int cz_apply_moves_batch(int device, uint8_t *boards /* [n][90] in/out */, const uint16_t *moves /* [n] */, int n,
                         uint8_t *captured /* [n] piece code captured or 0 */);
int cz_encode_batch(int device, const uint8_t *boards, const uint8_t *sides, int n, float *out /* [n][9][10][14] */);
/* device-pointer variants (no copies; async on stream) */
int cz_legal_moves_dev(const uint8_t *boards, const uint8_t *sides, int n, uint16_t *moves, int32_t *counts, void *stream);
int cz_encode_dev(const uint8_t *boards, const uint8_t *sides, int n, void *out, int dtype, void *stream);

/* ---- the batched engine: n_games independent (GameBoard, MCTS_tree) pairs resident in HBM ---- */
typedef struct cz_engine cz_engine;

/* arena_words: uint32 words of tree storage per game per half (two halves, ping-pong re-rooting);
 * 0 selects the default (2 Mi words = 8 MiB per half; a 1200-playout self-play soak peaks at 0.74 Mi words). */
int cz_engine_create(int n_games, int64_t arena_words, int device, cz_engine **out);
/* Leaf-parallel variant: up to `leaves` (1..64) leaves per game per wave inside one tree (virtual-loss batching; the
 * search_threads > 1 idea of main.py:337-440 with a deterministic schedule of its own -- not bit-comparable with the
 * reference's coroutine interleaving).  Network rows are then g*leaves + slot: nn_in [n_games*leaves][...],
 * logits [n_games*leaves][2086], value [n_games*leaves].  leaves == 1 is cz_engine_create; leaves == -1 runs the
 * leaf-parallel kernel with a single slot (test hook: must equal the one-leaf kernel bit for bit). */
int cz_engine_create_ex(int n_games, int64_t arena_words, int device, int leaves, cz_engine **out);
/* search_threads = K > 1 EXACTLY as the reference schedules it (main.py:337-470 on uvloop), in canonical deterministic form: every
 * playout is a task, at most K hold the semaphore, the event loop's FIFO batches, the two-hop asyncio.sleep(1e-4) spin on
 * now_expanding nodes and prediction_worker's batching are simulated per game by one warp (k_wave_fifo); node blocks carry the
 * stored Q of back_up_value (main.py:193) because concurrent virtual losses make it differ from W/N.  Specification:
 * oracle/detloop.py (the reference's own coroutines on a deterministic loop) and the C oracle (co_tree_search_fifo), both
 * pinned to real uvloop runs of the reference (tests/golden/k16_stats.json.gz).  Network rows as for `leaves`: g*K + slot.
 * search_threads: 1..32 (1 reproduces cz_engine_create's results with the 6-array blocks). */
int cz_engine_create_fifo(int n_games, int64_t arena_words, int device, int search_threads, cz_engine **out);
int cz_engine_is_fifo(const cz_engine *e);
int cz_engine_leaves(const cz_engine *e);
int cz_engine_destroy(cz_engine *e);
int cz_engine_n_games(const cz_engine *e);

/* GameBoard.reload (main.py:604-608) + MCTS_tree.reload (255-258) for the games with mask[g] != 0
 * (mask NULL = all).  boards/sides/rr NULL = the start position, 'w', 0. All host pointers. */
int cz_engine_reset(cz_engine *e, void *stream, const uint8_t *mask, const uint8_t *boards, const uint8_t *sides,
                    const int32_t *rr);

/* Override side-to-move / restrict_round of the root without touching the tree: MCTS_tree.main takes
 * current_player and restrict_round as call arguments (main.py:473).  Host pointers, any may be NULL. */
int cz_engine_set_root_meta(cz_engine *e, void *stream, const uint8_t *mask, const uint8_t *sides, const int32_t *rr);

/* Start a search of `playouts` playouts (MCTS_tree.main's loop count, main.py:490) on the games with
 * mask[g] != 0 (NULL = every non-terminal game). */
int cz_engine_begin_search(cz_engine *e, void *stream, const uint8_t *mask, int playouts);

/* One wave = one kernel launch (capturable in a CUDA graph; no host sync, no allocation):
 *   1. for every game with a pending leaf: expand it from logits/value of the previous wave
 *      (leaf_node.expand main.py:175-187 incl. flip_policy 1152-1155 and the legal-move generation),
 *      undo the virtual loss and back the value up (main.py:426-435, 189-194);
 *   2. run playouts of start_tree_search (main.py:350-440, search_threads = 1 semantics) until the
 *      game needs a network evaluation: PUCT selection (108-116, 158-159), virtual loss (403-404),
 *      terminal / 60-ply rule (409-416); terminal playouts are backed up in-kernel and the game
 *      continues with its next playout;
 *   3. encode the leaf (main.py:531-557) into row g of nn_in.
 * nn_in: dev [n_games][9][10][14] of `nn_dtype`; logits: dev f32 [n_games][2086]; value: dev f32 [n_games].
 * A game's row of logits/value is only read if that game has a pending leaf.                              */
int cz_engine_wave(cz_engine *e, void *stream, void *nn_in, int nn_dtype, const float *logits, const float *value);
/* search_threads = K engines (cz_engine_create_fifo): one wave WITH ROW COMPACTION of the K-rows-per-game network batch.  On average
 * ~11 of the 16 slots of a searching game carry a leaf (the rest spin on a node that is being expanded, main.py:354-355), and games
 * whose search is complete carry none; evaluating only those rows is what the reference's prediction_worker does (main.py:442-464
 * evaluates "whatever is queued").  nn_stage [B*K rows] is written like cz_engine_wave's nn_in; nn_dense [B*K rows] receives the rows
 * that need an evaluation, densely, in (game, slot) order; logits / value are read through the row map of the PREVIOUS call: between
 * two calls the caller evaluates nn_dense[0 .. n) into logits[0 .. n) / value[0 .. n), n = cz_engine_live_rows (stream sync).
 * Results are identical to cz_engine_wave's whenever the evaluator is row-independent. */
int cz_engine_wave_compact(cz_engine *e, void *stream, void *nn_stage, void *nn_dense, int nn_dtype, const float *logits, const float *value);
int cz_engine_live_rows(cz_engine *e, void *stream, int32_t *out_rows);

/* the two halves of a wave as separate launches */
int cz_engine_select(cz_engine *e, void *stream, void *nn_in, int nn_dtype);
int cz_engine_expand_backup(cz_engine *e, void *stream, const float *logits, const float *value);

/* Board hashing (north_star): when switched on, every wave also leaves the 64-bit Zobrist key of each pending leaf's position
 * (piece-square keys XOR side-to-move key, maintained incrementally along the descent; the root's key lives in the game's header
 * line and is updated by cz_engine_play) in a device array indexed like the network batch rows.  The reference has no position
 * hashing (nodes are keyed by object identity, main.py:246-247); the keys exist for evaluation de-duplication studies and
 * transposition statistics, they never influence the search.  Capturable; read by waves launched / captured afterwards. */
int cz_engine_enable_hashing(cz_engine *e, int on);
int cz_engine_leaf_hashes(cz_engine *e, uint64_t **dev_keys /* out: device pointer, [n_games*leaves] */);
int cz_engine_root_keys(cz_engine *e, void *stream, uint64_t *keys /* host [B] */);

/* Number of games that still have playouts to run or a leaf pending (device->host, synchronises stream). */
int cz_engine_unfinished(cz_engine *e, void *stream, int32_t *out_count);
/* Asynchronous form: writes the count to *dev_count (device int32) without synchronising. */
int cz_engine_unfinished_async(cz_engine *e, void *stream, int32_t *dev_count);

/* Root statistics in child (= move generation) order: what get_action reads from root.child
 * (main.py:1339) and MCTS_tree.Q (261-270).  HOST buffers; synchronises stream.
 * q = f32(W/N) (0 when N == 0).  Any pointer may be NULL. */
int cz_engine_root_children(cz_engine *e, void *stream, int32_t *n_children /* [B] (-1: root not expanded) */,
                            uint16_t *moves /* [B][128] */, int32_t *visits /* [B][128] */,
                            float *w /* [B][128] */, float *p /* [B][128] */, float *q /* [B][128] */);

/* Play child_index[g] (index into the root's children; < 0 = leave game g alone):
 * GameBoard state update (main.py:1522-1528) + MCTS_tree.update_tree (272-276): the chosen child's
 * subtree is compacted into the other arena half and becomes the root; terminal flags are updated
 * (main.py:1532-1545).  child_index is a HOST buffer. */
int cz_engine_play(cz_engine *e, void *stream, const int32_t *child_index /* [B] */);
/* Same, and returns every game's packed status record (one kernel, one device->host copy, one synchronisation):
 * CZ_STATUS_BYTES per game: [0,90) board | 90 side | 91 terminal | 92 winner (int8) | 96 ply i32 | 100 restrict_round i32 |
 * 104 Q (f32) of the move just played = MCTS_tree.Q(act), main.py:1350 | 108 N of the new root i32. */
#define CZ_STATUS_BYTES 112
int cz_engine_play_status(cz_engine *e, void *stream, const int32_t *child_index /* [B] */, uint8_t *status /* host [B][112] or NULL */);
int cz_engine_status_packed(cz_engine *e, void *stream, uint8_t *status /* host [B][112] */);
/* MCTS_tree.update_tree(act) keyed by the MOVE (main.py:272-276, as human_move calls it at 1418) + the board update: for every game
 * the root child whose move equals moves[g] is played exactly as cz_engine_play_status plays its index; the status record's Q is
 * Q(act) of THIS tree (human_move's win_rate).  moves[g] == CZ_NOMOVE leaves game g alone.  A move that is not a child of the root,
 * or any move at a root that was never expanded, sets CZ_ERR_NOCHILD on that game and leaves it untouched (status still written). */
#define CZ_NOMOVE 0xFFFF
int cz_engine_play_moves(cz_engine *e, void *stream, const uint16_t *moves /* host [B] */, uint8_t *status /* host [B][112] or NULL */);

/* Game status (cchess_main.check_end main.py:1380-1392): HOST buffers, any may be NULL; synchronises.
 * terminal: 0 running, 1 king captured, 2 draw (restrict_round >= 60); winner: 0 'w', 1 'b', -1 none. */
int cz_engine_status(cz_engine *e, void *stream, uint8_t *terminal, int8_t *winner, int32_t *ply, int32_t *rr,
                     uint8_t *side, uint8_t *boards /* [B][90] */);

/* Counters since creation, summed over games: out[0] expansions (calls of expand), out[1] playouts,
 * out[2] sum of path lengths L, out[3] sum of scanned children c_l, out[4] OR of per-game error flags,
 * out[5] max arena words in use, out[6] index of first game with an error (or -1), out[7] max path length,
 * out[8] sum over expansions of the number of children C. */
int cz_engine_counters(cz_engine *e, void *stream, int64_t *out /* [9] */);

/* Test hook: flat DFS signature of game g's tree, records of 6 int64
 * (label index, N, W bits, P bits, Q bits, n_children), children in order. Returns record count via *n. */
int cz_engine_tree_signature(cz_engine *e, void *stream, int game, int64_t *out, int64_t cap, int64_t *n);

/* ---- network ends (policy_value_network.py:45-48 and 55-74), hand-written; the residual tower is library code ----
 * cz_net_first_conv: canonical boards (dev u8 [B][96], from cz_engine_wave with CZ_BOARD) ->
 *     ReLU(conv3x3(14->128) + bias) as fp16 NHWC [B][90][128].  w1: dev fp16 [9 taps][14 pieces][128], b1: dev f32 [128]
 *     (batch norm already folded in).  The one-hot [9][10][14] tensor of main.py:547-557 is never materialised.
 * cz_net_heads: x fp16 [B][90][128] -> logits f32 [B][2086] (raw, no softmax) and value f32 [B] (tanh).
 *     wh f32 [3][128] / bh [3]: 1x1 convs of the policy (2) and value (1) heads with BN folded; w1t f32 [90][256], b1 [256],
 *     w2 [256], b2 [1] (device pointers, so that weights can be refreshed under a captured CUDA graph): value MLP; wp fp16 [2112][192] / bp f32 [2112]: policy FC zero-padded; hp_scratch fp16 [B][192],
 *     hv_scratch f32 [B][96]. */
int cz_net_first_conv(const uint8_t *canon_boards, int B, const void *w1, const float *b1, void *out, void *stream);
/* Same result on the tcgen05 tensor cores: the one-hot im2col matrix is built in shared memory, the accumulators live in
 * TMEM.  w_umma: dev fp16, the weights in the canonical K-major UMMA layout [18 k-chunks][16 groups][8 channels][8 k]
 * with k = tap*16 + piece code (code 0 rows are zero; row (centre tap, code 15) holds the bias, every other code-15 row is
 * zero); 36 864 bytes.  b1 is ignored (kept for signature symmetry with cz_net_first_conv). */
int cz_net_first_conv_tc(const uint8_t *canon_boards, int B, const void *w_umma, const float *b1, void *out, void *stream);
/* Same result on mma.sync with the one-hot operand built in registers (alternative first layer; slower than the gather-add, see DESIGN.md).  w_frag: dev, the
 * weights of cz_net_first_conv_tc's K = tap*16 + piece-code convention (bias row included) in m16n8k16 B-fragment order
 * [9 k-steps][16 n-tiles][32 lanes][2 words]: word0 = {W[k0+2t][n], W[k0+2t+1][n]}, word1 = the same at k + 8, n = 8*tile + lane/4, t = lane%4. */
int cz_net_first_conv_mma(const uint8_t *canon_boards, int B, const void *w_frag, void *out, void *stream);
int cz_net_heads(const void *x, int B, const float *wh, const float *bh, const float *w1t, const float *b1, const float *w2, const float *b2,
                 const void *wp, const float *bp, void *hp_scratch, float *hv_scratch, float *logits, float *value, void *stream);

/* ---- host side: get_action's sampling for a whole batch of games (main.py:1339-1348), bit-identical to the numpy calls ----
 * For every game g with live[g] != 0 (live NULL = all):  probs = ex[g][:n] / np.sum(ex[g][:n])  (ex = exp(log(visits)/T - max), computed
 * by the caller with numpy);  exploration: p = 0.75 * probs + 0.25 * RandomState.dirichlet(0.3 * ones(n));  choice[g] =
 * RandomState.choice(n, p = p).  mt_states: one legacy MT19937 state per game, CZ_MT_WORDS uint32 each = key[624], pos, 0 --
 * exactly numpy.random.RandomState.get_state()[1:3] -- advanced in place by the same number of draws numpy would make.
 * probs [B][128] receives the normalised (un-noised) probabilities, i.e. the recorded pi.  fallback[g] = 1 when the vector would
 * make numpy raise (NaN / negative / not summing to 1): the caller lets numpy itself handle that game (after the Dirichlet draws,
 * which have been consumed as in the reference).  All pointers are HOST memory; no GPU involved. */
#define CZ_MT_WORDS 626
int cz_host_choose_moves(int n_games, const uint8_t *live, const int32_t *n_children, const double *ex /* [B][128] */, int exploration,
                         uint32_t *mt_states /* [B][626] */, int32_t *choice /* [B] */, double *probs /* [B][128] */, uint8_t *fallback /* [B] */,
                         int n_threads);

/* cz_net_heads for large batches: policy FC on tcgen05 + TMEM (operands bulk-copied in the UMMA layout), 1x1 head convolution on
 * mma.sync, value MLP concurrently.  wp_tiled: dev fp16 [17 label tiles][24 k-chunks][128 labels][8 features] (labels >= 2086 zero),
 * bp f32 [2176]; hp_tiled_scratch: fp16, ceil(B/128) * 49152 bytes, zero-initialised once by the caller. */
int cz_net_heads_tc(const void *x, int B, const float *wh, const float *bh, const float *w1t, const float *b1, const float *w2, const float *b2,
                    const void *wp_tiled, const float *bp, void *hp_tiled_scratch, float *hv_scratch, float *logits, float *value, void *stream);

/* The second half of cz_net_heads alone: value MLP and policy FC on head features that are already computed
 * (hp fp16 [B][192], hv f32 [B][96]) -- what follows cz_net_tower_small. */
int cz_net_heads_fc(const void *hp, const float *hv, int B, const float *w1t, const float *b1, const float *w2, const float *b2,
                    const void *wp, const float *bp, float *logits, float *value, void *stream);

/* ---- the whole convolutional trunk for a FEW positions in one launch (play mode / single-tree search, BASELINE config 5) ----
 * policy_value_network.py:45-74, 151-162 with batch norm folded: first conv3x3(14->128) from the canonical board bytes,
 * n_conv = 2*res_block_nums 3x3 convolutions (residual blocks), the two 1x1 head convolutions; output = the head features
 * hp fp16 [n_pos][192] / hv f32 [n_pos][96] that cz_net_heads_fc turns into logits and value.
 * One thread-block cluster of `cluster` (1, 2, 4, 8) CTAs per position: activations stay in shared memory (UMMA K-major layout,
 * 3x3 taps = descriptor start offsets), weights stream from L2 by TMA, tcgen05.mma accumulates in TMEM, epilogues exchange
 * channel slices through distributed shared memory.  See csrc/cz_tower.cu.
 *   w1     dev fp16 [9][14][128]   (as cz_net_first_conv);  bias dev f32 [1 + n_conv][128];  wh f32 [3][128], bh f32 [3]
 *   wblob  dev fp16, cz_net_tower_blob_bytes(n_conv) bytes, arranged for THIS cluster size:
 *          [conv][tap 9][rank `cluster`][k-chunk 16][out channel 128/cluster][8 in channels]   (in channel = 8*chunk + i) */
int64_t cz_net_tower_blob_bytes(int n_conv);
int cz_net_tower_small(const uint8_t *canon_boards, int n_pos, int cluster, int n_conv, const void *w1, const void *wblob, const float *bias,
                       const float *wh, const float *bh, void *hp, float *hv, void *stream);

/* ---- fp32-accurate inference on the tensor cores (net.py: SplitTf32Plan; policy_value_network.py:202-214 is fp32) ----
 * y dev f32 [n_pix][128] (NHWC activations) -> hi dev f32 [n_pix][128] = tf32(y) (round to the 10-bit mantissa) and
 * x2 dev fp16 [n_pix][256] = { (y - hi) * 2^11 | hi } (both exact in fp16).  A TF32 convolution of hi with hi(w) and an fp16
 * convolution of x2 with { hi(w) | lo(w) * 2^11 } accumulate hi*hi and (lo*hi + hi*lo) * 2^11 in two separate f32 chains (the
 * tensor cores' accumulator truncates, measured -6.6e-9 relative per accumulated term: the full-size terms get the short chain). */
int cz_net_split_tf32(const float *y, float *hi, void *x2, long long n_pix, void *stream);
/* The f32 epilogue of such a convolution fused with the split for the next one, one streaming pass:
 *   v = ReLU(t + 2^-11 s + bias [+ skip]);   x = v (optional);   hi, x2 = split of v (optional, both or neither)
 * t dev f32 [n_pix][128] (hi*hi, raw); s dev fp16 [n_pix][128] or NULL (cross terms, raw, scaled by 2^11); bias dev f32 [128];
 * skip dev f32 [n_pix][128] or NULL (x may alias skip). */
int cz_net_epilogue_split(const float *t, const void *s, const float *bias, const float *skip, float *x, float *hi, void *x2, long long n_pix, void *stream);

#ifdef __cplusplus
}
#endif
#endif
