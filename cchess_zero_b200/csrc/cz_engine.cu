// cz_engine.cu -- batched MCTS self-play engine for sm_100a (one warp per game) + its C ABI.
//
// Replaces, for thousands of concurrent games, the reference's leaf_node / MCTS_tree /
// GameBoard hot path (main.py:93-206, 234-577, 579-1109) with search_threads = 1 semantics
// (SURVEY Appendix A.4).  Results are bit-exact: every float op below is an explicit
// round-to-nearest IEEE intrinsic in the width numpy uses (f32 for P/W/Q, f64 for U and Q+U).
//
// HBM layout (SoA over games; B = n_games, A = arena words per half):
//   hdr         u32 [B][16]     ONE 64-byte line per game with every scalar of its search and game state (flags: active /
//                               pending / side / arena half / terminal / winner; done, target, restrict_round, root N / count /
//                               base, arena top, path length, ply, high-water marks, error flags, Zobrist key of the root).
//                               A wave reads it with one coalesced load and writes it back with one coalesced store.
//   root_board  u8  [B][96]     90-byte mailbox + pad, 24 coalesced u32 per game; the packed bitboards the move generator
//                               works on (occupancy, red set, file-major occupancy) are derived from it by ballots (cz_rules.cuh)
//   arena       u32 [B][2][A]   per-game bump arena of node blocks, two halves (ping-pong
//                               compaction when the root moves, MCTS_tree.update_tree)
//   node block  = 8-word header {n_children,...} followed by five arrays of stride
//                 cs = roundup8(n_children):  P f32 | W f32 | N i32 | META u32 | CHILD u32
//                 META = move | n_grandchildren << 16, CHILD = base of the child's block or NONE.
//                 One node = one contiguous run, each array sector-aligned, so a warp reads
//                 all PUCT inputs of a node with coalesced loads in a single round trip.
//   path        uint2 [B][MAXD] {slot of P[idx], cs | move << 8} of the edges of the current playout
//   leaf_board  u8  [B][96]     board at the pending leaf (+ side in byte 90)
//
// Latency plan of a wave (the kernel is a chain of dependent loads, not a bandwidth problem): everything whose address is
// known at entry -- header line, leaf board, root board, the first 32 path entries, the evaluated value -- is requested before
// the first use (round trip 1); the W / N words of the path (back-up operands) are requested next and arrive under the move
// generation (round trip 2); the root block of the next descent is requested before the logit gather of the expansion (round
// trips 3 and 4 overlap); after that one round trip per tree level remains, which is the pointer chase itself.  Counters are
// fire-and-forget reductions (RED), never read-modify-write chains.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/cchess_b200.h"
#include "cz_rules.cuh"

#define MAXD 256
#define NONE 0xFFFFFFFFu
#define HDR 8
#define WARPS_PER_BLOCK 4
#define MAX_INKERNEL_PLAYOUTS 16
#define MAX_WPB 10                 // warps per CTA of the wave kernels
#define SPATH 32                   // path entries mirrored in shared memory / prefetched in registers

// per-game header line
enum { H_FLAGS = 0, H_DONE, H_TARGET, H_RR, H_ROOTN, H_ROOTCNT, H_ROOTBASE, H_ALLOC, H_PLEN, H_PLY, H_MAXALLOC, H_ERR, H_MAXDEPTH,
       H_HASHLO, H_HASHHI, H_SPARE, HW = 16 };
#define F_ACTIVE 1u
#define F_PEND(f) (((f) >> 1) & 3u)                 // 0 none, 1 leaf evaluation pending, 2 root expansion pending
#define F_SETPEND(f, p) (((f) & ~6u) | ((uint32_t)(p) << 1))
#define F_SIDE 8u
#define F_CUR 16u
#define F_TERM(f) (((f) >> 8) & 3u)                 // 0 running, 1 king captured, 2 draw
#define F_WIN(f) ((int)(((f) >> 10) & 3u) - 1)      // -1 none, 0 'w', 1 'b'

namespace {

thread_local std::string g_err;
int fail(int code, const char *what, cudaError_t ce = cudaSuccess) {
    g_err = what;
    if (ce != cudaSuccess) { g_err += ": "; g_err += cudaGetErrorString(ce); }
    return code;
}
#define CUDA_TRY(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) return fail(CZ_ECUDA, #x, _e); } while (0)

// ------------------------------------------------------------------------------------------
// host-side label table (create_uci_labels, main.py:30-65): same enumeration order
// ------------------------------------------------------------------------------------------
struct Labels {
    char text[CZ_NLABEL][4];
    int16_t of[CZ_NSQ * CZ_NSQ];
    int32_t unflipped[CZ_NLABEL];
    Labels() {
        int n = 0;
        auto put = [&](int l1, int n1, int l2, int n2) {
            text[n][0] = char('a' + l1); text[n][1] = char('0' + n1);
            text[n][2] = char('a' + l2); text[n][3] = char('0' + n2);
            n++;
        };
        const int kdx[8] = {-2, -1, -2, 1, 2, -1, 2, 1}, kdy[8] = {-1, -2, 1, -2, -1, 2, 1, 2};
        for (int l1 = 0; l1 < 9; l1++)
            for (int n1 = 0; n1 < 10; n1++) {
                for (int t = 0; t < 9; t++) if (t != l1) put(l1, n1, t, n1);       // along the rank
                for (int t = 0; t < 10; t++) if (t != n1) put(l1, n1, l1, t);      // along the file
                for (int k = 0; k < 8; k++) {                                      // knight jumps
                    int l2 = l1 + kdx[k], n2 = n1 + kdy[k];
                    if (l2 >= 0 && l2 < 9 && n2 >= 0 && n2 < 10) put(l1, n1, l2, n2);
                }
            }
        const char *adv = "d7e8e8d7e8f9f9e8d0e1e1d0e1f2f2e1d2e1e1d2e1f0f0e1d9e8e8d9e8f7f7e8";
        const char *bis = "a2c4c4a2c0e2e2c0e2g4g4e2g0i2i2g0a7c9c9a7c5e7e7c5e7g9g9e7g5i7i7g5"
                          "a2c0c0a2c4e2e2c4e2g0g0e2g4i2i2g4a7c5c5a7c9e7e7c9e7g5g5e7g9i7i7g9";
        for (int i = 0; i < 16; i++) { memcpy(text[n], adv + 4 * i, 4); n++; }
        for (int i = 0; i < 32; i++) { memcpy(text[n], bis + 4 * i, 4); n++; }
        for (auto &v : of) v = -1;
        for (int i = 0; i < CZ_NLABEL; i++) {
            int s = (text[i][1] - '0') * 9 + (text[i][0] - 'a'), d = (text[i][3] - '0') * 9 + (text[i][2] - 'a');
            if (of[s * CZ_NSQ + d] < 0) of[s * CZ_NSQ + d] = (int16_t)i;
        }
        for (int i = 0; i < CZ_NLABEL; i++) {  // flipped_uci_labels (main.py:23-27): rank digit d -> 9-d
            int s = (9 - (text[i][1] - '0')) * 9 + (text[i][0] - 'a'), d = (9 - (text[i][3] - '0')) * 9 + (text[i][2] - 'a');
            unflipped[i] = of[s * CZ_NSQ + d];
        }
    }
};
const Labels &labels() { static Labels L; return L; }

// ------------------------------------------------------------------------------------------
// device state
// ------------------------------------------------------------------------------------------
struct Dev {
    int B;
    long long A;
    int K;                            // leaves per game per wave (1 = the reference's search_threads=1 schedule)
    int hash_on;                      // maintain Zobrist keys of the pending leaves (board hashing; off by default)
    int narr;                         // arrays per node block: 5 (P W N META CHILD), 6 in FIFO mode (+ stored Q, main.py:193)
    uint32_t *fifo;                   // [B][FW] event-loop state of the search_threads = K schedule (k_wave_fifo); NULL otherwise
    // row compaction of the K-row network batch (cz_engine_wave_compact): only rows that carry a leaf are evaluated
    int compact;                      // this launch reads logits / value through row_map and publishes live_mask
    uint32_t *live_mask;              // [B] bit s = slot s of the game awaits an evaluation queued by THIS launch
    int32_t *row_map;                 // [B*K] (game, slot) -> row of the dense batch its leaf was evaluated in
    int32_t *src_of;                  // [B*K] dense row -> g*K + slot
    int32_t *dense_count;             // [1]   rows of the dense batch
    uint32_t *hdr;                    // [B][HW]
    uint8_t *root_board;              // [B][96]
    uint8_t *leaf_board;              // [B][96]
    uint2 *path;                      // [B][MAXD]
    uint8_t *pendK;                   // [B][K] leaf-parallel mode: per-slot pending flag, path length, path, leaf board
    int32_t *plenK;
    uint2 *pathK;
    uint8_t *leafK;
    uint32_t *arena;
    unsigned long long *cnt_expand, *cnt_playout, *cnt_L, *cnt_c, *cnt_C;
    unsigned long long *leaf_hash;    // [B*K] Zobrist key of the position in network row r (valid when hash_on)
    const unsigned long long *zob;    // [16][96] piece-square keys; zob[95] = side-to-move key
    const int16_t *label_of;
    // staging
    int32_t *st_n, *st_visits, *st_choice;
    uint16_t *st_moves;
    float *st_w, *st_p, *st_q;
    int32_t *st_count;
    uint8_t *st_status;               // [B][CZ_STATUS_BYTES]
};

__device__ __forceinline__ uint32_t *arena_half(const Dev &E, int g, int cur) {
    return E.arena + ((size_t)g * 2 + cur) * (size_t)E.A;
}

struct WarpSmem {
    uint8_t board[96];
    uint16_t moves[136];
    uint16_t li[128];
    float ps[128];
    uint2 path[SPATH];
    cz::MoveScratch scratch;
};

// order-preserving map of a double onto uint64 (NaN must be removed by the caller, -0 canonicalised)
__device__ __forceinline__ unsigned long long dkey(double s) {
    long long b = __double_as_longlong(s);
    return (unsigned long long)(b ^ ((b >> 63) | (long long)0x8000000000000000ULL));
}

// a path entry names one edge: {word index of its P entry, stride cs (low byte) | move << 8}
__device__ __forceinline__ uint2 path_entry(uint32_t slot, uint32_t cs, uint32_t move) { return make_uint2(slot, cs | (move << 8)); }
#define PE_CS(pe) ((pe).y & 0xFFu)
#define PE_MOVE(pe) ((pe).y >> 8)

// VL undo + back_up_value of ONE edge (main.py:426-435, 189-194); (Wbits, Nbits) were loaded earlier.
// val = value handed to the deepest edge; sign alternates going up.
// `inflight`: leaf-parallel mode keeps a per-edge count of playouts currently holding a virtual loss on it (META bits 24-30).
__device__ __forceinline__ void backup_edge(uint32_t *ar, uint2 pe, int d, int depth, float val, uint32_t Wbits, uint32_t Nbits, bool inflight) {
    const uint32_t slot = pe.x, cs = PE_CS(pe);
    const float v = ((depth - 1 - d) & 1) ? -val : val;
    ar[slot + cs] = __float_as_uint(__fadd_rn(__fadd_rn(__uint_as_float(Wbits), 3.0f), v));
    ar[slot + 2 * cs] = (uint32_t)((int)Nbits - 3 + 1);
    if (inflight) ar[slot + 3 * cs] -= (1u << 24);
}
// whole path from memory (global or shared), any depth
__device__ void warp_backup_path(const uint2 *path, uint32_t *ar, int depth, float val, int lane, bool inflight) {
    for (int d = lane; d < depth; d += 32) {
        const uint2 pe = path[d];
        backup_edge(ar, pe, d, depth, val, ar[pe.x + PE_CS(pe)], ar[pe.x + 2 * PE_CS(pe)], inflight);
    }
    __syncwarp();
}

// Move list of the leaf staged in S.board (+ side in byte 90), in reference order, and the label index of every move (with
// flip_policy, main.py:1152-1155, folded into the index: rank y -> 9-y for black).  Leaves S.moves[i] / S.li[i]; returns n.
__device__ int warp_leaf_moves(const Dev &E, WarpSmem &S, uint32_t &errf, int lane) {
    const int lside = S.board[90];
    int n = cz::warp_legal_moves(S.board, lside, S.moves, S.scratch, lane);
    if (n == 0) errf |= CZ_ERR_NOMOVES;
    if (n > CZ_MAXCHILD) { errf |= CZ_ERR_CHILDREN; n = CZ_MAXCHILD; }
    for (int i = lane; i < n; i += 32) {
        const int mv = S.moves[i];
        int src = mv & 127, dst = mv >> 7;
        if (lside == 1) {
            src = (9 - src / 9) * 9 + src % 9;
            dst = (9 - dst / 9) * 9 + dst % 9;
        }
        int li = __ldg(E.label_of + src * CZ_NSQ + dst);
        if (li < 0) { errf |= CZ_ERR_NOLABEL; li = 0; }
        S.li[i] = (uint16_t)li;
    }
    __syncwarp();
    return n;
}

// leaf_node.expand (main.py:175-187) in three parts.
// 1: move generation + arena reservation.  Returns n > 0, or 0 when the expansion cannot happen (no moves / arena full).
__device__ int expand_reserve(const Dev &E, WarpSmem &S, uint32_t &alloc, uint32_t &base, uint32_t &errf, int lane) {
    uint32_t ef = 0;
    const int n = warp_leaf_moves(E, S, ef, lane);
    const uint32_t cs = (uint32_t)((n + 7) & ~7), size = HDR + (uint32_t)E.narr * cs;
    base = alloc;
    if ((long long)base + size > E.A) ef |= CZ_ERR_ARENA;
    ef = __reduce_or_sync(CZ_FULL, ef);
    errf |= ef;
    if (ef & (CZ_ERR_ARENA | CZ_ERR_NOMOVES)) return 0;
    alloc = base + size;
    return n;
}
// 2: prior gather (lg = this leaf's logits row), serial float32 normalisation, block write
__device__ void expand_write(uint32_t *ar, WarpSmem &S, const float *lg, int n, uint32_t base, int lane, bool with_q = false) {
    for (int i = lane; i < n; i += 32) S.ps[i] = __ldg(lg + S.li[i]);
    __syncwarp();
    const uint32_t cs = (uint32_t)((n + 7) & ~7);
    float tot = 1e-8f;  // tot_p = 1e-8 accumulated in float32, in move order (main.py:176, 184)
#pragma unroll 8
    for (int i = 0; i < n; i++) tot = __fadd_rn(tot, S.ps[i]);   // strictly serial adds; unrolled so the LDS latency overlaps
    uint32_t *blk = ar + base;
    if (lane < HDR) blk[lane] = lane == 0 ? (uint32_t)n : 0u;
    for (int i = lane; i < (int)cs; i += 32) {
        const bool live = i < n;
        blk[HDR + i] = live ? __float_as_uint(__fdiv_rn(S.ps[i], tot)) : 0u;   // n.P /= tot_p (main.py:187)
        blk[HDR + cs + i] = 0u;                                                // W = 0
        blk[HDR + 2 * cs + i] = 0u;                                            // N = 0
        blk[HDR + 3 * cs + i] = live ? (uint32_t)S.moves[i] : 0u;              // META: move, no grandchildren yet
        blk[HDR + 4 * cs + i] = NONE;
        if (with_q) blk[HDR + 5 * cs + i] = 0u;                                // stored Q = 0 (leaf_node.__init__, main.py:96)
    }
    __syncwarp();
}
// 3: link the new block under the edge it was reached by (plain stores: the move travels in the path entry).
// META: move (0-15) | n_children (16-23) | in-flight count (24-30, leaf-parallel mode) | claimed (31, cleared here)
__device__ __forceinline__ void expand_link(uint32_t *ar, uint2 pe, int n, uint32_t base, uint32_t inflight) {
    ar[pe.x + 3 * PE_CS(pe)] = PE_MOVE(pe) | ((uint32_t)n << 16) | (inflight << 24);
    ar[pe.x + 4 * PE_CS(pe)] = base;
}

// Zobrist key delta of one move on the mailbox board (piece p moves src -> dst, capturing q): board hashing of north_star
__device__ __forceinline__ unsigned long long zob_move(const unsigned long long *z, int p, int q, int src, int dst) {
    unsigned long long h = __ldg(z + p * 96 + src) ^ __ldg(z + p * 96 + dst) ^ __ldg(z + 95);   // mover leaves / arrives, side flips
    if (q) h ^= __ldg(z + q * 96 + dst);
    return h;
}
__device__ unsigned long long zob_board(const unsigned long long *z, const uint8_t *b, int side) {
    unsigned long long h = side ? z[95] : 0ull;
    for (int s = 0; s < 90; s++) if (b[s]) h ^= z[b[s] * 96 + s];
    return h;
}

// row: index of this leaf's row in the network batch (g in one-leaf mode, g*K+slot in leaf-parallel mode)
template <typename T>
__device__ void store_leaf_at(uint8_t *leaf_board, WarpSmem &S, int side, T *nn_in, size_t row, int lane) {
    if (lane == 0) S.board[90] = (uint8_t)side;
    __syncwarp();
    uint32_t *lb = reinterpret_cast<uint32_t *>(leaf_board);
    if (lane < 24) lb[lane] = reinterpret_cast<const uint32_t *>(S.board)[lane];
    if constexpr (sizeof(T) == 1) {
        // CZ_BOARD: the evaluator reads the side-to-move-canonical board itself (try_flip, main.py:560-574);
        // cz_net_first_conv applies the reference's cell indexing, so no [9][10][14] tensor is written.
        uint8_t *o = reinterpret_cast<uint8_t *>(nn_in) + row * 96;
        for (int i = lane; i < 96; i += 32) {
            int p = 0;
            if (i < 90) {
                if (side == 0) p = S.board[i];
                else { const int yy = i / 9, xx = i - yy * 9; p = cz::swap_colour(S.board[(9 - yy) * 9 + xx]); }
            }
            o[i] = (uint8_t)p;
        }
    } else {
        cz::warp_encode<T>(S.board, side, nn_in + row * CZ_ENC_LEN, lane);
    }
    __syncwarp();      // every lane is done reading S.board before the caller stages the next position in it (racecheck, round 2)
}

// The PUCT inputs of one node block in registers: lane l holds children l, l+32, l+64, l+96.
struct BlockRegs {
    uint32_t P[4], W[4], N[4], meta[4], child[4], Q[4];
};
template <bool WITH_Q = false>
__device__ __forceinline__ void load_block(const uint32_t *ar, uint32_t base, int cnt, int lane, BlockRegs &R) {
    const uint32_t cs = (uint32_t)((cnt + 7) & ~7);
    const uint32_t *blk = ar + base + HDR;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int i = lane + 32 * k;
        if (i < cnt) {
            R.P[k] = blk[i]; R.W[k] = blk[cs + i]; R.N[k] = blk[2 * cs + i]; R.meta[k] = blk[3 * cs + i]; R.child[k] = blk[4 * cs + i];
            if (WITH_Q) R.Q[k] = blk[5 * cs + i];
        }
    }
}
__device__ __forceinline__ uint32_t pick(const uint32_t (&a)[4], int k) { return k == 0 ? a[0] : k == 1 ? a[1] : k == 2 ? a[2] : a[3]; }

// select_new (main.py:158-159) over get_Q_plus_U_new (108-116) on a block held in registers: index of the FIRST maximum.
// MULTI: Q is taken from the loss-free statistics (in-flight count in META bits 24-30), see k_wave_multi.
// MODE 2 (search_threads = K schedule): the STORED Q of the last back_up_value, exactly what get_Q_plus_U_new reads (main.py:116).
template <int MODE>
__device__ __forceinline__ uint32_t select_child(const BlockRegs &R, int cnt, int parentN, int lane) {
    constexpr bool MULTI = MODE == 1;
    const double sq = __dsqrt_rn((double)parentN);
    double bs = 0.0;
    uint32_t bi = NONE;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int i = lane + 32 * k;
        if (i < cnt) {
            const float P = __uint_as_float(R.P[k]);
            float W = __uint_as_float(R.W[k]);
            const int N = (int)R.N[k];
            int Nr = N;
            if (MULTI) {
                const int c = (int)((R.meta[k] >> 24) & 0x7Fu);                       // playouts holding a virtual loss here
                Nr = N - 3 * c;
                if (c) W = __fadd_rn(W, (float)(3 * c));
            }
            const float Q = MODE == 2 ? __uint_as_float(R.Q[k]) : (Nr > 0 ? __fdiv_rn(W, (float)Nr) : 0.0f);   // Q = W / N in float32 (of the last real backup)
            const float p5 = __fmul_rn(5.0f, P);                                      // c_puct * P in float32
            const double U = __ddiv_rn(__dmul_rn((double)p5, sq), (double)(1 + N));
            double s = __dadd_rn((double)Q, U);
            if (i > 0 && s != s) s = -INFINITY;   // a NaN score never displaces an earlier candidate
            if (k == 0 || s > bs) { bs = s; bi = (uint32_t)i; }
        }
    }
    // warp arg-max, first maximum wins (python max(): strict >)
    const bool nan0 = __shfl_sync(CZ_FULL, (int)(bs != bs), 0) != 0;   // only lane 0 (i == 0) can hold a NaN
    if (nan0) return 0;
    const unsigned long long key = bi == NONE ? 0ull : dkey(__dadd_rn(bs, 0.0));
    const uint32_t hi = (uint32_t)(key >> 32), lo = (uint32_t)key;
    const uint32_t mhi = __reduce_max_sync(CZ_FULL, hi);
    const uint32_t mlo = __reduce_max_sync(CZ_FULL, hi == mhi ? lo : 0u);
    return __reduce_min_sync(CZ_FULL, (bi != NONE && hi == mhi && lo == mlo) ? bi : NONE);
}

#define HGET(f) __shfl_sync(CZ_FULL, h, (f))
#define HSET(f, v) do { if (lane == (f)) h = (uint32_t)(v); } while (0)

// One wave for one game (one warp).  DO_EXPAND: consume the previous evaluation; DO_SELECT: run playouts
// until the next leaf.
// Launch shape: one CTA per SM whenever the games fit (warps per CTA = ceil(B / #SMs), <= MAX_WPB), so that every SM carries
// the same number of game-warps; shared memory is sized per launch (sizeof(WarpSmem) per warp).
template <typename T, bool DO_EXPAND, bool DO_SELECT>
__global__ void __launch_bounds__(32 * MAX_WPB, 1) k_wave(Dev E, T *nn_in, const float *logits, const float *value) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WarpSmem *smem = reinterpret_cast<WarpSmem *>(smem_raw);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int g = blockIdx.x * (blockDim.x >> 5) + w;
    if (g >= E.B) return;
    WarpSmem &S = smem[w];
    // ---- round trip 1: everything addressed by g alone ----
    uint32_t *hp = E.hdr + (size_t)g * HW;
    uint32_t h = lane < HW ? hp[lane] : 0u;
    uint32_t lbw = 0, rbw = 0;
    if (lane < 24) {
        if (DO_EXPAND) lbw = reinterpret_cast<const uint32_t *>(E.leaf_board + (size_t)g * 96)[lane];
        if (DO_SELECT) rbw = reinterpret_cast<const uint32_t *>(E.root_board + (size_t)g * 96)[lane];
    }
    uint2 pth = make_uint2(0, 0);
    float val = 0.f;
    if (DO_EXPAND) { pth = E.path[(size_t)g * MAXD + lane]; val = value[g]; }
    uint32_t flags = HGET(H_FLAGS);
    if (!(flags & F_ACTIVE)) return;
    uint32_t *ar = arena_half(E, g, (flags & F_CUR) ? 1 : 0);
    int pend = (int)F_PEND(flags);
    int done = (int)HGET(H_DONE);
    const int target = (int)HGET(H_TARGET);
    uint32_t alloc = HGET(H_ALLOC), errf = 0;
    uint32_t root_base = HGET(H_ROOTBASE);
    int root_cnt = (int)HGET(H_ROOTCNT);
    const int root_N = (int)HGET(H_ROOTN);
    int plen = (int)HGET(H_PLEN);
    BlockRegs R;
    bool have_root = false;

    if (DO_EXPAND && pend) {
        const int depth = pend == 1 ? plen : 0;
        // ---- round trip 2: the W / N words of the path (back-up operands) fly under the move generation ----
        uint32_t bW = 0, bN = 0;
        if (lane < depth && lane < SPATH) { bW = ar[pth.x + PE_CS(pth)]; bN = ar[pth.x + 2 * PE_CS(pth)]; }
        if (lane < 24) reinterpret_cast<uint32_t *>(S.board)[lane] = lbw;
        __syncwarp();
        uint32_t base;
        const int n = expand_reserve(E, S, alloc, base, errf, lane);
        const bool ok = n > 0;
        if (pend == 1) {
            // leaf returns -v (main.py:384); on an engine error the playout is closed with 0
            const float v = ok ? -val : 0.0f;
            if (lane < depth && lane < SPATH) backup_edge(ar, pth, lane, depth, v, bW, bN, false);
            for (int d = SPATH + lane; d < depth; d += 32) {          // (paths longer than the prefetch window)
                const uint2 pe = E.path[(size_t)g * MAXD + d];
                backup_edge(ar, pe, d, depth, v, ar[pe.x + PE_CS(pe)], ar[pe.x + 2 * PE_CS(pe)], false);
            }
            done++;
            if (lane == 0) atomicAdd(E.cnt_playout + g, 1ull);
        }
        __syncwarp();
        if (!ok && pend == 2) {      // the root could not be expanded: the game leaves the search
            HSET(H_FLAGS, F_SETPEND(flags & ~F_ACTIVE, 0));
            if (lane == H_ERR) h |= errf;
            if (lane < HW) hp[lane] = h;
            return;
        }
        // ---- round trip 3 (root block of the next descent) is requested BEFORE the logit gather (round trip 4) ----
        if (DO_SELECT && pend == 1 && done < target) { load_block<false>(ar, root_base, root_cnt, lane, R); have_root = true; }
        if (ok) {
            expand_write(ar, S, logits + (size_t)g * CZ_NLABEL, n, base, lane);
            if (pend == 2) { root_base = base; root_cnt = n; }
            else {
                uint2 last;
                if (depth - 1 < SPATH) { last.x = __shfl_sync(CZ_FULL, pth.x, depth - 1); last.y = __shfl_sync(CZ_FULL, pth.y, depth - 1); }
                else last = E.path[(size_t)g * MAXD + depth - 1];
                if (lane == 0) expand_link(ar, last, n, base, 0);
                if (have_root && depth == 1) {        // the new node hangs under the root: patch the prefetched copy of that edge
                    const uint32_t e = last.x - (root_base + HDR);
                    if (lane == (int)(e & 31)) {
#pragma unroll
                        for (int k = 0; k < 4; k++)
                            if (k == (int)(e >> 5)) { R.meta[k] = PE_MOVE(last) | ((uint32_t)n << 16); R.child[k] = base; }
                    }
                }
            }
            if (lane == 0) { atomicAdd(E.cnt_expand + g, 1ull); atomicAdd(E.cnt_C + g, (unsigned long long)n); }
        }
        pend = 0;
        __syncwarp();
    }

    uint32_t maxdep = HGET(H_MAXDEPTH);
    if (DO_SELECT && !pend) {
        const int side0 = (flags & F_SIDE) ? 1 : 0, rr0 = (int)HGET(H_RR);
        unsigned long long rhash = 0;
        if (E.hash_on) rhash = (unsigned long long)HGET(H_HASHLO) | ((unsigned long long)HGET(H_HASHHI) << 32);
        if (root_cnt < 0) {
            // MCTS_tree.main: expand the root first (main.py:475-487); not a playout
            if (lane < 24) reinterpret_cast<uint32_t *>(S.board)[lane] = rbw;
            __syncwarp();
            store_leaf_at<T>(E.leaf_board + (size_t)g * 96, S, side0, nn_in, (size_t)g, lane);
            if (E.hash_on && lane == 0) E.leaf_hash[g] = rhash;
            pend = 2; plen = 0;
        } else {
            unsigned long long accL = 0, accC = 0;
            // Terminal playouts are resolved here without the network.  A position with a king capture at the root sends
            // nearly all of its playouts down that edge; bounding the number resolved per launch keeps one such game from
            // stretching the wave for the other games (it simply continues in the next wave; per-game order is unchanged).
            int budget = MAX_INKERNEL_PLAYOUTS;
            while (done < target && budget-- > 0) {
                // ---- one playout of start_tree_search (main.py:350-440) ----
                if (lane < 24) reinterpret_cast<uint32_t *>(S.board)[lane] = rbw;
                __syncwarp();
                int side = side0, rr = rr0, depth = 0;
                uint32_t base = root_base;
                int cnt = root_cnt;
                int parentN = root_N;
                unsigned long long hash = rhash;
                bool leaf = false, fault = false;
                float tval = 0.0f;
                if (!have_root) load_block<false>(ar, base, cnt, lane, R);
                have_root = false;
                for (;;) {
                    if (cnt <= 0 || depth >= MAXD) {
                        errf |= cnt <= 0 ? CZ_ERR_NOMOVES : CZ_ERR_DEPTH;
                        fault = true;
                        break;
                    }
                    const uint32_t cs = (uint32_t)((cnt + 7) & ~7);
                    uint32_t *blk = ar + base + HDR;
                    const uint32_t e = select_child<0>(R, cnt, parentN, lane);
                    const int owner = e & 31, ke = (int)(e >> 5);
                    const uint32_t meta = __shfl_sync(CZ_FULL, pick(R.meta, ke), owner);
                    const uint32_t child = __shfl_sync(CZ_FULL, pick(R.child, ke), owner);
                    const int eN = (int)__shfl_sync(CZ_FULL, pick(R.N, ke), owner);
                    if (lane == owner) {  // virtual loss (main.py:403-404)
                        blk[cs + e] = __float_as_uint(__fadd_rn(__uint_as_float(pick(R.W, ke)), -3.0f));
                        blk[2 * cs + e] = (uint32_t)(eN + 3);
                    }
                    if (lane == 0) {
                        const uint2 pe = path_entry(base + HDR + e, cs, meta & 0xFFFFu);
                        E.path[(size_t)g * MAXD + depth] = pe;
                        if (depth < SPATH) S.path[depth] = pe;
                    }
                    depth++;
                    accL += 1; accC += (unsigned)cnt;
                    const int src = meta & 127, dst = (meta >> 7) & 127;
                    const int cap = S.board[dst], mover = S.board[src];
                    __syncwarp();
                    if (lane == 0) { S.board[dst] = (uint8_t)mover; S.board[src] = 0; }
                    __syncwarp();
                    if (E.hash_on) hash ^= zob_move(E.zob, mover, cap, src, dst);
                    side ^= 1;                                   // main.py:392
                    rr = cap == 0 ? rr + 1 : 0;                  // is_kill_move, main.py:393-396
                    if (cap == 1 || cap == 8) {                  // king captured: main.py:409-414
                        const float v = cap == 1 ? (side == 1 ? 1.0f : -1.0f) : (side == 1 ? -1.0f : 1.0f);
                        tval = -v;
                        break;
                    }
                    if (rr >= 60) { tval = 0.0f; break; }        // main.py:415-416
                    if (child == NONE) { leaf = true; break; }   // main.py:357: not expanded -> evaluate
                    base = child;
                    cnt = (int)((meta >> 16) & 0xFFu);
                    parentN = eN + 3;                            // the child's N carries the virtual loss just added
                    load_block<false>(ar, base, cnt, lane, R);   // one round trip per level: the pointer chase itself
                }
                if ((uint32_t)depth > maxdep) maxdep = (uint32_t)depth;
                if (leaf) {
                    store_leaf_at<T>(E.leaf_board + (size_t)g * 96, S, side, nn_in, (size_t)g, lane);
                    if (E.hash_on && lane == 0) E.leaf_hash[g] = hash;
                    pend = 1; plen = depth;
                    break;
                }
                __syncwarp();
                // terminal (or faulted) playout: VL undo + backup, also from the shared-memory mirror of the path
                warp_backup_path(depth <= SPATH ? S.path : E.path + (size_t)g * MAXD, ar, depth, tval, lane, false);
                done++;
                if (lane == 0) atomicAdd(E.cnt_playout + g, 1ull);
                if (fault) break;
            }
            if (lane == 0 && accL) { atomicAdd(E.cnt_L + g, accL); atomicAdd(E.cnt_c + g, accC); }
        }
    }
    if (DO_SELECT && E.hash_on && pend == 0 && lane == 0) E.leaf_hash[g] = 0ull;    // no leaf of this game in the batch
    // ---- the header line goes back with one coalesced store ----
    HSET(H_FLAGS, F_SETPEND(flags, pend));
    HSET(H_DONE, done);
    HSET(H_ALLOC, alloc);
    HSET(H_PLEN, plen);
    HSET(H_ROOTBASE, root_base);
    HSET(H_ROOTCNT, root_cnt);
    HSET(H_MAXDEPTH, maxdep);
    if (lane == H_MAXALLOC && alloc > h) h = alloc;
    if (lane == H_ERR) h |= errf;
    if (lane < HW) hp[lane] = h;
}

__constant__ uint8_t c_start[96];   // start position, uploaded by cz_engine_create

// ---- leaf-parallel wave: up to K leaves per game per launch (virtual-loss batching inside one tree) ---------------
// NOT the reference's coroutine schedule (that one depends on the event loop, SURVEY 0.7) and therefore not bit-comparable
// with search_threads > 1 of the reference; with K = 1 it is exactly the one-leaf kernel above (tested against the oracle).
// Differences from k_wave: every slot has its own path / leaf board / network row; an edge counts the playouts that
// currently hold a virtual loss on it (META bits 24-30) so that Q is taken from the loss-free statistics like the reference's
// stale Q (main.py:403-404 never touches Q); an unexpanded child that is already being evaluated is `claimed` (bit 31) and a
// second descent that reaches it backs off (the reference waits on now_expanding, main.py:354-355).
template <typename T>
__global__ void __launch_bounds__(32 * MAX_WPB, 1) k_wave_multi(Dev E, T *nn_in, const float *logits, const float *value) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WarpSmem *smem = reinterpret_cast<WarpSmem *>(smem_raw);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int g = blockIdx.x * (blockDim.x >> 5) + w;
    if (g >= E.B) return;
    WarpSmem &S = smem[w];
    uint32_t *hp = E.hdr + (size_t)g * HW;
    uint32_t h = lane < HW ? hp[lane] : 0u;
    uint32_t rbw = lane < 24 ? reinterpret_cast<const uint32_t *>(E.root_board + (size_t)g * 96)[lane] : 0u;
    uint32_t flags = HGET(H_FLAGS);
    if (!(flags & F_ACTIVE)) return;
    uint32_t *ar = arena_half(E, g, (flags & F_CUR) ? 1 : 0);
    const int K = E.K;
    int done = (int)HGET(H_DONE);
    const int target = (int)HGET(H_TARGET);
    uint32_t alloc = HGET(H_ALLOC), errf = 0, maxdep = HGET(H_MAXDEPTH);
    uint32_t root_base = HGET(H_ROOTBASE);
    int root_cnt = (int)HGET(H_ROOTCNT);
    const int root_N = (int)HGET(H_ROOTN);
    const int side0 = (flags & F_SIDE) ? 1 : 0, rr0 = (int)HGET(H_RR);
    unsigned long long rhash = 0;
    if (E.hash_on) rhash = (unsigned long long)HGET(H_HASHLO) | ((unsigned long long)HGET(H_HASHHI) << 32);
    bool dead = false;

    // ---- phase 1: consume the evaluations of the previous wave, slot by slot ----
    for (int s = 0; s < K && !dead; s++) {
        const size_t idx = (size_t)g * K + s;
        const int pend = E.pendK[idx];
        if (!pend) continue;
        const int depth = E.plenK[idx];
        const uint2 *path = E.pathK + idx * MAXD;
        if (lane < 24) reinterpret_cast<uint32_t *>(S.board)[lane] = reinterpret_cast<const uint32_t *>(E.leafK + idx * 96)[lane];
        __syncwarp();
        uint32_t base;
        const int n = expand_reserve(E, S, alloc, base, errf, lane);
        const bool ok = n > 0;
        if (ok) {
            expand_write(ar, S, logits + idx * CZ_NLABEL, n, base, lane);
            if (pend == 2) { root_base = base; root_cnt = n; }
            else if (lane == 0) expand_link(ar, path[depth - 1], n, base, 1u);    // exactly one playout (ours) holds a loss on a claimed edge
            if (lane == 0) { atomicAdd(E.cnt_expand + g, 1ull); atomicAdd(E.cnt_C + g, (unsigned long long)n); }
        }
        __syncwarp();
        if (pend == 1) {
            warp_backup_path(path, ar, depth, ok ? -value[idx] : 0.0f, lane, true);
            done++;
            if (lane == 0) atomicAdd(E.cnt_playout + g, 1ull);
        }
        if (lane == 0) E.pendK[idx] = 0;
        if (!ok && pend == 2) { flags &= ~F_ACTIVE; dead = true; }
        __syncwarp();
    }

    if (!dead && root_cnt < 0) {   // root expansion first (main.py:475-487), one slot
        if (lane < 24) reinterpret_cast<uint32_t *>(S.board)[lane] = rbw;
        __syncwarp();
        store_leaf_at<T>(E.leafK + (size_t)g * K * 96, S, side0, nn_in, (size_t)g * K, lane);
        if (lane == 0) { E.pendK[(size_t)g * K] = 2; E.plenK[(size_t)g * K] = 0; if (E.hash_on) E.leaf_hash[(size_t)g * K] = rhash; }
    } else if (!dead) {
        // ---- phase 2: up to K descents with virtual loss ----
        unsigned long long accL = 0, accC = 0;
        int inflight = 0, budget = MAX_INKERNEL_PLAYOUTS + K;
        bool stop = false;
        BlockRegs R;
        for (int s = 0; s < K && !stop; s++) {
            const size_t idx = (size_t)g * K + s;
            uint2 *path = E.pathK + idx * MAXD;
            while (done + inflight < target && budget-- > 0) {
                if (lane < 24) reinterpret_cast<uint32_t *>(S.board)[lane] = rbw;
                __syncwarp();
                int side = side0, rr = rr0, depth = 0;
                uint32_t base = root_base;
                int cnt = root_cnt;
                int parentN = root_N;
                unsigned long long hash = rhash;
                int outcome = 0;   // 1 leaf, 2 terminal, 3 collision, 4 fault
                float tval = 0.0f;
                for (;;) {
                    if (cnt <= 0 || depth >= MAXD) {
                        errf |= cnt <= 0 ? CZ_ERR_NOMOVES : CZ_ERR_DEPTH;
                        outcome = 4;
                        break;
                    }
                    const uint32_t cs = (uint32_t)((cnt + 7) & ~7);
                    uint32_t *blk = ar + base + HDR;
                    load_block<false>(ar, base, cnt, lane, R);
                    const uint32_t e = select_child<1>(R, cnt, parentN, lane);
                    const int owner = e & 31, ke = (int)(e >> 5);
                    const uint32_t meta = __shfl_sync(CZ_FULL, pick(R.meta, ke), owner);
                    const uint32_t child = __shfl_sync(CZ_FULL, pick(R.child, ke), owner);
                    const int eN = (int)__shfl_sync(CZ_FULL, pick(R.N, ke), owner);
                    const bool claimed = (meta & 0x80000000u) != 0;
                    const int src = meta & 127, dst = (meta >> 7) & 127;
                    const int cap = S.board[dst], mover = S.board[src];
                    const bool term = cap == 1 || cap == 8 || (cap == 0 ? rr + 1 : 0) >= 60;
                    if (child == NONE && claimed && !term) { outcome = 3; break; }     // someone else is evaluating this leaf
                    if (lane == owner) {  // virtual loss + in-flight count (+ claim when this becomes our leaf)
                        blk[cs + e] = __float_as_uint(__fadd_rn(__uint_as_float(pick(R.W, ke)), -3.0f));
                        blk[2 * cs + e] = (uint32_t)(eN + 3);
                        blk[3 * cs + e] = (meta + (1u << 24)) | ((child == NONE && !term) ? 0x80000000u : 0u);
                    }
                    if (lane == 0) path[depth] = path_entry(base + HDR + e, cs, meta & 0xFFFFu);
                    depth++;
                    accL += 1; accC += (unsigned)cnt;
                    __syncwarp();
                    if (lane == 0) { S.board[dst] = (uint8_t)mover; S.board[src] = 0; }
                    __syncwarp();
                    if (E.hash_on) hash ^= zob_move(E.zob, mover, cap, src, dst);
                    side ^= 1;
                    rr = cap == 0 ? rr + 1 : 0;
                    if (cap == 1 || cap == 8) {
                        const float v = cap == 1 ? (side == 1 ? 1.0f : -1.0f) : (side == 1 ? -1.0f : 1.0f);
                        tval = -v; outcome = 2;
                        break;
                    }
                    if (rr >= 60) { tval = 0.0f; outcome = 2; break; }
                    if (child == NONE) { outcome = 1; break; }
                    base = child;
                    cnt = (int)((meta >> 16) & 0xFFu);
                    parentN = eN + 3;
                }
                if ((uint32_t)depth > maxdep) maxdep = (uint32_t)depth;
                __syncwarp();
                if (outcome == 1) {
                    store_leaf_at<T>(E.leafK + idx * 96, S, side, nn_in, idx, lane);
                    if (lane == 0) { E.pendK[idx] = 1; E.plenK[idx] = depth; if (E.hash_on) E.leaf_hash[idx] = hash; }
                    inflight++;
                    break;                                   // next slot
                }
                if (outcome == 3) {                          // back off: take the virtual losses of this partial path back
                    for (int d = lane; d < depth; d += 32) {
                        const uint2 pe = path[d];
                        const uint32_t cs = PE_CS(pe);
                        ar[pe.x + cs] = __float_as_uint(__fadd_rn(__uint_as_float(ar[pe.x + cs]), 3.0f));
                        ar[pe.x + 2 * cs] -= 3u;
                        ar[pe.x + 3 * cs] -= (1u << 24);
                    }
                    __syncwarp();
                    stop = true;
                    break;
                }
                warp_backup_path(path, ar, depth, tval, lane, true);   // terminal (or faulted) playout
                done++;
                if (lane == 0) atomicAdd(E.cnt_playout + g, 1ull);
                if (outcome == 4) { stop = true; break; }
            }
            if (!(done + inflight < target)) break;
        }
        if (lane == 0 && accL) { atomicAdd(E.cnt_L + g, accL); atomicAdd(E.cnt_c + g, accC); }
    }
    HSET(H_FLAGS, flags);
    HSET(H_DONE, done);
    HSET(H_ALLOC, alloc);
    HSET(H_ROOTBASE, root_base);
    HSET(H_ROOTCNT, root_cnt);
    HSET(H_MAXDEPTH, maxdep);
    if (lane == H_MAXALLOC && alloc > h) h = alloc;
    if (lane == H_ERR) h |= errf;
    if (lane < HW) hp[lane] = h;
}


// ---- search_threads = K: the reference's coroutine schedule in canonical FIFO form --------------------------------------
// One warp per game runs the little event loop that oracle/detloop.py (the reference's own coroutines on a deterministic loop)
// and the C oracle (co_tree_search_fifo) specify, and that reproduces the real uvloop runs of the reference
// (tests/golden/k16_stats.json.gz).  Every playout is a task; at most K are admitted (the semaphore, main.py:250, 342); the ready
// queue is processed in batches ("iterations"); prediction_worker (442-464) is the last callback of every odd iteration and
// evaluates whatever was queued.  Entries: STEP (start a playout, or re-check after a spin), AHOP (first hop of
// asyncio.sleep(1e-4), main.py:354-355), RESUME (evaluation arrived: expand + unwind, 368-384).  Virtual losses of suspended
// tasks stay on their paths; back_up_value stores Q = W / N of that moment (193), losses of other tasks included, so node blocks
// carry a sixth array with the stored Q.  A launch runs iterations until an evaluation is needed (at most K rows per game:
// network row g*K + slot) or the search is complete.
enum { FI_ITER = 0, FI_NCUR, FI_NQ, FI_STARTED, FI_CUR = 4, FI_QUEUE = 20, FW = 28 };     // cur: 64 entry bytes, queue: 32 slot bytes
#define EV_STEP 0u
#define EV_AHOP 1u
#define EV_RESUME 2u
#define FIFO_MAX_ITERS 8

__device__ __forceinline__ void backup_edge_q(uint32_t *ar, uint2 pe, int d, int depth, float val) {
    const uint32_t slot = pe.x, cs = PE_CS(pe);
    const float v = ((depth - 1 - d) & 1) ? -val : val;
    const float W = __fadd_rn(__fadd_rn(__uint_as_float(ar[slot + cs]), 3.0f), v);     // node.W += virtual_loss; then W += value
    const int N = (int)ar[slot + 2 * cs] - 3 + 1;
    ar[slot + cs] = __float_as_uint(W);
    ar[slot + 2 * cs] = (uint32_t)N;
    ar[slot + 5 * cs] = __float_as_uint(__fdiv_rn(W, (float)N));                          // self.Q = self.W / self.N (main.py:193)
}
__device__ void warp_unwind_q(const uint2 *path, uint32_t *ar, int depth, float val, int lane) {
    for (int d = lane; d < depth; d += 32) backup_edge_q(ar, path[d], d, depth, val);
    __syncwarp();
}

template <typename T>
__global__ void __launch_bounds__(32 * MAX_WPB, 1) k_wave_fifo(Dev E, T *nn_in, const float *logits, const float *value) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WarpSmem *smem = reinterpret_cast<WarpSmem *>(smem_raw);
    __shared__ uint8_t s_cur[MAX_WPB][64], s_nxt[MAX_WPB][64], s_queue[MAX_WPB][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int g = blockIdx.x * (blockDim.x >> 5) + w;
    if (g >= E.B) return;
    WarpSmem &S = smem[w];
    uint8_t *cur = s_cur[w], *nxt = s_nxt[w], *queue = s_queue[w];
    uint32_t *hp = E.hdr + (size_t)g * HW;
    uint32_t h = lane < HW ? hp[lane] : 0u;
    uint32_t *fp = E.fifo + (size_t)g * FW;
    uint32_t fw = lane < FW ? fp[lane] : 0u;
    const uint32_t rbw = lane < 24 ? reinterpret_cast<const uint32_t *>(E.root_board + (size_t)g * 96)[lane] : 0u;
    uint32_t flags = HGET(H_FLAGS);
    if (!(flags & F_ACTIVE)) { if (E.compact && lane == 0) E.live_mask[g] = 0u; return; }
    uint32_t *ar = arena_half(E, g, (flags & F_CUR) ? 1 : 0);
    const int K = E.K;
    int done = (int)HGET(H_DONE);
    const int target = (int)HGET(H_TARGET);
    uint32_t alloc = HGET(H_ALLOC), errf = 0, maxdep = HGET(H_MAXDEPTH);
    uint32_t root_base = HGET(H_ROOTBASE);
    int root_cnt = (int)HGET(H_ROOTCNT);
    const int root_N = (int)HGET(H_ROOTN);
    const int side0 = (flags & F_SIDE) ? 1 : 0, rr0 = (int)HGET(H_RR);
    int pend = (int)F_PEND(flags);
    uint32_t live = 0u;               // slots whose leaf goes to the network after this launch
    // the network row that holds the evaluation of (game, slot): the slot's own row, or the dense row the compaction gave it
#define NN_ROW(idx_) (E.compact ? (size_t)E.row_map[idx_] : (size_t)(idx_))
    int iter = (int)__shfl_sync(CZ_FULL, fw, FI_ITER), ncur = (int)__shfl_sync(CZ_FULL, fw, FI_NCUR);
    int nq = (int)__shfl_sync(CZ_FULL, fw, FI_NQ), started = (int)__shfl_sync(CZ_FULL, fw, FI_STARTED);
    {
        const uint32_t cw0 = __shfl_sync(CZ_FULL, fw, (FI_CUR + lane) & 31), qw0 = __shfl_sync(CZ_FULL, fw, (FI_QUEUE + lane) & 31);
        if (lane < 16) reinterpret_cast<uint32_t *>(cur)[lane] = cw0;
        if (lane < 8) reinterpret_cast<uint32_t *>(queue)[lane] = qw0;
    }
    __syncwarp();
    bool dead = false;

    if (pend == 2) {       // the root's evaluation arrived (main.py:475-487; its value is discarded)
        if (lane < 24) reinterpret_cast<uint32_t *>(S.board)[lane] = reinterpret_cast<const uint32_t *>(E.leafK + (size_t)g * K * 96)[lane];
        __syncwarp();
        uint32_t base;
        const int n = expand_reserve(E, S, alloc, base, errf, lane);
        if (n > 0) {
            expand_write(ar, S, logits + NN_ROW((size_t)g * K) * CZ_NLABEL, n, base, lane, true);
            root_base = base; root_cnt = n;
            if (lane == 0) { atomicAdd(E.cnt_expand + g, 1ull); atomicAdd(E.cnt_C + g, (unsigned long long)n); }
        } else { flags &= ~F_ACTIVE; dead = true; }
        pend = 0;
    }
    if (!dead && root_cnt < 0) {
        if (lane < 24) reinterpret_cast<uint32_t *>(S.board)[lane] = rbw;
        __syncwarp();
        store_leaf_at<T>(E.leafK + (size_t)g * K * 96, S, side0, nn_in, (size_t)g * K, lane);
        pend = 2; live = 1u;
    } else if (!dead) {
        if (iter == 0) {   // gather(): the first K playouts acquire the semaphore in iteration 1, the rest wait in FIFO order
            iter = 1; nq = 0;
            ncur = target < K ? target : K;
            started = ncur;
            if (lane < ncur) { cur[lane] = (uint8_t)(lane | (EV_STEP << 6)); E.plenK[(size_t)g * K + lane] = 0; }
            __syncwarp();
        }
        unsigned long long accL = 0, accC = 0;
        BlockRegs R;
        bool need_nn = false;
        for (int it = 0; it < FIFO_MAX_ITERS && !need_nn && done < target; it++) {
            int nnxt = 0;
            for (int e = 0; e < ncur; e++) {
                const uint32_t ev = cur[e & 63];          // (a ring: iteration 1 appends while it runs, at most K entries are live)
                const int slot = (int)(ev & 63u), kind = (int)(ev >> 6);
                const size_t idx = (size_t)g * K + slot;
                if (kind == (int)EV_AHOP) { if (lane == 0) nxt[nnxt] = (uint8_t)(slot | (EV_STEP << 6)); nnxt++; continue; }
                uint2 *path = E.pathK + idx * MAXD;
                int plen = E.plenK[idx];
                bool ended = false;
                if (kind == (int)EV_RESUME) {
                    if (lane < 24) reinterpret_cast<uint32_t *>(S.board)[lane] = reinterpret_cast<const uint32_t *>(E.leafK + idx * 96)[lane];
                    __syncwarp();
                    uint32_t base;
                    const int n = expand_reserve(E, S, alloc, base, errf, lane);
                    if (n > 0) {
                        expand_write(ar, S, logits + NN_ROW(idx) * CZ_NLABEL, n, base, lane, true);
                        if (lane == 0) {
                            expand_link(ar, path[plen - 1], n, base, 0u);               // also clears `claimed`: now_expanding.remove(node)
                            atomicAdd(E.cnt_expand + g, 1ull); atomicAdd(E.cnt_C + g, (unsigned long long)n);
                        }
                    } else if (lane == 0) {
                        const uint2 pe = path[plen - 1];
                        ar[pe.x + 3 * PE_CS(pe)] &= 0x7FFFFFFFu;                         // give the claim back
                    }
                    __syncwarp();
                    warp_unwind_q(path, ar, plen, n > 0 ? -value[NN_ROW(idx)] : 0.0f, lane);   // return value[0] * -1, unwound through every frame
                    ended = true;
                } else {
                    int side, rr, cnt, parentN;
                    uint32_t base;
                    bool go = true;
                    if (plen == 0) {          // a fresh playout: start_tree_search(root)
                        if (lane < 24) reinterpret_cast<uint32_t *>(S.board)[lane] = rbw;
                        side = side0; rr = rr0; base = root_base; cnt = root_cnt; parentN = root_N;
                    } else {                  // re-check after a spin: the node this task stands on
                        if (lane < 24) reinterpret_cast<uint32_t *>(S.board)[lane] = reinterpret_cast<const uint32_t *>(E.leafK + idx * 96)[lane];
                        __syncwarp();
                        side = S.board[90]; rr = S.board[91];
                        const uint2 pe = path[plen - 1];
                        const uint32_t meta = ar[pe.x + 3 * PE_CS(pe)], child = ar[pe.x + 4 * PE_CS(pe)];
                        parentN = (int)ar[pe.x + 2 * PE_CS(pe)];
                        base = child; cnt = (int)((meta >> 16) & 0xFFu);
                        if (meta & 0x80000000u) { if (lane == 0) nxt[nnxt] = (uint8_t)(slot | (EV_AHOP << 6)); nnxt++; go = false; }   // still now_expanding
                        else if (child == NONE) {                                        // (its expansion failed: this task evaluates it)
                            if (lane == 0) { ar[pe.x + 3 * PE_CS(pe)] = meta | 0x80000000u; queue[nq] = (uint8_t)slot; }
                            nq++;
                            store_leaf_at<T>(E.leafK + idx * 96, S, side, nn_in, idx, lane);
                            go = false;
                        }
                    }
                    __syncwarp();
                    while (go) {
                        if (cnt <= 0 || plen >= MAXD) { errf |= cnt <= 0 ? CZ_ERR_NOMOVES : CZ_ERR_DEPTH; warp_unwind_q(path, ar, plen, 0.0f, lane); ended = true; break; }
                        const uint32_t cs = (uint32_t)((cnt + 7) & ~7);
                        uint32_t *blk = ar + base + HDR;
                        load_block<true>(ar, base, cnt, lane, R);
                        const uint32_t c = select_child<2>(R, cnt, parentN, lane);
                        const int owner = c & 31, ke = (int)(c >> 5);
                        const uint32_t meta = __shfl_sync(CZ_FULL, pick(R.meta, ke), owner);
                        const uint32_t child = __shfl_sync(CZ_FULL, pick(R.child, ke), owner);
                        const int eN = (int)__shfl_sync(CZ_FULL, pick(R.N, ke), owner);
                        if (lane == owner) {  // virtual loss (main.py:403-404); Q stays as stored
                            blk[cs + c] = __float_as_uint(__fadd_rn(__uint_as_float(pick(R.W, ke)), -3.0f));
                            blk[2 * cs + c] = (uint32_t)(eN + 3);
                        }
                        if (lane == 0) path[plen] = path_entry(base + HDR + c, cs, meta & 0xFFFFu);
                        plen++;
                        accL += 1; accC += (unsigned)cnt;
                        const int src = meta & 127, dst = (meta >> 7) & 127;
                        const int cap = S.board[dst], mover = S.board[src];
                        __syncwarp();
                        if (lane == 0) { S.board[dst] = (uint8_t)mover; S.board[src] = 0; }
                        __syncwarp();
                        side ^= 1;
                        rr = cap == 0 ? rr + 1 : 0;
                        if (cap == 1 || cap == 8) {                                      // main.py:409-414
                            const float v = cap == 1 ? (side == 1 ? 1.0f : -1.0f) : (side == 1 ? -1.0f : 1.0f);
                            warp_unwind_q(path, ar, plen, -v, lane);
                            ended = true; break;
                        }
                        if (rr >= 60) { warp_unwind_q(path, ar, plen, 0.0f, lane); ended = true; break; }   // 415-416
                        // start_tree_search(child): now_expanding? unexpanded? (main.py:354-357)
                        if (meta & 0x80000000u) {
                            if (lane == 0) { S.board[90] = (uint8_t)side; S.board[91] = (uint8_t)rr; }
                            __syncwarp();
                            if (lane < 24) reinterpret_cast<uint32_t *>(E.leafK + idx * 96)[lane] = reinterpret_cast<const uint32_t *>(S.board)[lane];
                            if (lane == 0) nxt[nnxt] = (uint8_t)(slot | (EV_AHOP << 6));
                            nnxt++;
                            break;
                        }
                        if (child == NONE) {
                            if (lane == 0) { blk[3 * cs + c] = meta | 0x80000000u; queue[nq] = (uint8_t)slot; S.board[91] = (uint8_t)rr; }
                            nq++;
                            store_leaf_at<T>(E.leafK + idx * 96, S, side, nn_in, idx, lane);   // features queued (push_queue, main.py:362-366)
                            break;
                        }
                        base = child;
                        cnt = (int)((meta >> 16) & 0xFFu);
                        parentN = eN + 3;
                    }
                    if ((uint32_t)plen > maxdep) maxdep = (uint32_t)plen;
                }
                __syncwarp();
                if (ended) {              // the task ends; its semaphore release wakes the next waiting playout (FIFO)
                    done++;
                    plen = 0;
                    if (lane == 0) atomicAdd(E.cnt_playout + g, 1ull);
                    if (started < target) {
                        started++;
                        // Iteration 1 runs the first step of EVERY playout's task in index order and the semaphore is a plain counter there:
                        // a playout that ends inside its first step (king capture / 60-move rule right below the root) hands its permit to
                        // the next playout in the SAME iteration, behind the tasks already started.  Later, a release wakes a waiter: next iteration.
                        if (iter == 1) { if (lane == 0) cur[ncur & 63] = (uint8_t)(slot | (EV_STEP << 6)); ncur++; }
                        else { if (lane == 0) nxt[nnxt] = (uint8_t)(slot | (EV_STEP << 6)); nnxt++; }
                    }
                }
                if (lane == 0) E.plenK[idx] = plen;
                __syncwarp();
            }
            if (iter & 1) {               // prediction_worker: last callback of every odd iteration
                if (nq > 0) {
                    if (lane < nq) nxt[nnxt + lane] = (uint8_t)(queue[lane] | (EV_RESUME << 6));
                    live = __reduce_or_sync(CZ_FULL, lane < nq ? (1u << (queue[lane] & 31)) : 0u);
                    nnxt += nq; nq = 0; need_nn = true;
                }
            }
            __syncwarp();
            iter++;
            uint8_t *tsw = cur; cur = nxt; nxt = tsw; ncur = nnxt;
        }
        if (lane == 0 && accL) { atomicAdd(E.cnt_L + g, accL); atomicAdd(E.cnt_c + g, accC); }
        if (done >= target) { iter = 0; ncur = 0; }       // the search is complete: the next begin_search starts a fresh event loop
    }
    __syncwarp();
    // ---- state back ----
    uint32_t cw = lane < 16 ? reinterpret_cast<const uint32_t *>(cur)[lane] : 0u, qw = lane < 8 ? reinterpret_cast<const uint32_t *>(queue)[lane] : 0u;
    if (lane == FI_ITER) fw = (uint32_t)iter;
    if (lane == FI_NCUR) fw = (uint32_t)ncur;
    if (lane == FI_NQ) fw = (uint32_t)nq;
    if (lane == FI_STARTED) fw = (uint32_t)started;
    const uint32_t cws = __shfl_sync(CZ_FULL, cw, (lane - FI_CUR) & 15), qws = __shfl_sync(CZ_FULL, qw, (lane - FI_QUEUE) & 7);
    if (lane >= FI_CUR && lane < FI_CUR + 16) fw = cws;
    if (lane >= FI_QUEUE && lane < FI_QUEUE + 8) fw = qws;
    if (lane < FW) fp[lane] = fw;
    if (E.compact && lane == 0) E.live_mask[g] = live;
#undef NN_ROW
    HSET(H_FLAGS, F_SETPEND(flags, pend));
    HSET(H_DONE, done);
    HSET(H_ALLOC, alloc);
    HSET(H_ROOTBASE, root_base);
    HSET(H_ROOTCNT, root_cnt);
    HSET(H_MAXDEPTH, maxdep);
    if (lane == H_MAXALLOC && alloc > h) h = alloc;
    if (lane == H_ERR) h |= errf;
    if (lane < HW) hp[lane] = h;
}

// ---- row compaction of the search_threads = K network batch ----------------------------------------------------------------
// After k_wave_fifo, only the (game, slot) rows named in live_mask carry a leaf to evaluate (on average ~11 of 16 per searching game,
// none for games whose search is complete).  k_compact_scan numbers them densely in (game, slot) order -- deterministic -- and
// k_compact_rows gathers their input rows from the staging buffer; the network then runs on the first ceil(count / bucket) * bucket
// rows only, and the next k_wave_fifo finds each evaluation through row_map.
__global__ void __launch_bounds__(1024) k_compact_scan(Dev E) {
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int g0 = 0; g0 < E.B; g0 += 1024) {
        const int g = g0 + tid;
        uint32_t m = g < E.B ? E.live_mask[g] : 0u;
        const int c = __popc(m);
        int incl = c;
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(CZ_FULL, incl, o); if (lane >= o) incl += t; }
        if (lane == 31) s_warp[w] = incl;
        __syncthreads();
        if (w == 0) {
            int v = s_warp[lane];
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(CZ_FULL, v, o); if (lane >= o) v += t; }
            s_warp[lane] = v;
        }
        __syncthreads();
        int base = s_carry + (w ? s_warp[w - 1] : 0) + incl - c;
        while (m) {
            const int slot = __ffs(m) - 1;
            m &= m - 1;
            E.row_map[(size_t)g * E.K + slot] = base;
            E.src_of[base] = g * E.K + slot;
            base++;
        }
        __syncthreads();
        if (tid == 0) s_carry += s_warp[31];
        __syncthreads();
    }
    if (tid == 0) E.dense_count[0] = s_carry;
}

// one warp per dense row, 8-byte units
__global__ void __launch_bounds__(256) k_compact_rows(Dev E, const uint2 *__restrict__ stage, uint2 *__restrict__ dense, int units) {
    const int lane = threadIdx.x & 31, n = E.dense_count[0];
    for (int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n; r += gridDim.x * (blockDim.x >> 5)) {
        const uint2 *src = stage + (size_t)E.src_of[r] * units;
        uint2 *dst = dense + (size_t)r * units;
        for (int i = lane; i < units; i += 32) dst[i] = src[i];
    }
}

// ---- GameBoard.reload + MCTS_tree.reload -------------------------------------------------
__global__ void k_reset(Dev E, const uint8_t *mask, const uint8_t *boards, const uint8_t *sides, const int32_t *rr) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= E.B || (mask && !mask[g])) return;
    uint8_t *b = E.root_board + (size_t)g * 96;
    for (int i = 0; i < 90; i++) b[i] = boards ? boards[(size_t)g * 90 + i] : c_start[i];
    for (int i = 90; i < 96; i++) b[i] = 0;
    const int side = sides ? (sides[g] ? 1 : 0) : 0;
    uint32_t *h = E.hdr + (size_t)g * HW;
    const unsigned long long z = zob_board(E.zob, b, side);
    const uint32_t keep_err = h[H_ERR], keep_ma = h[H_MAXALLOC], keep_md = h[H_MAXDEPTH];
    for (int i = 0; i < HW; i++) h[i] = 0;
    h[H_FLAGS] = side ? F_SIDE : 0u;
    h[H_RR] = (uint32_t)(rr ? rr[g] : 0);
    h[H_ROOTCNT] = (uint32_t)-1;
    h[H_HASHLO] = (uint32_t)z; h[H_HASHHI] = (uint32_t)(z >> 32);
    h[H_ERR] = keep_err; h[H_MAXALLOC] = keep_ma; h[H_MAXDEPTH] = keep_md;      // diagnostics live for the engine's lifetime
    if (E.pendK) for (int s = 0; s < E.K; s++) E.pendK[(size_t)g * E.K + s] = 0;
    if (E.fifo) for (int i = 0; i < FW; i++) E.fifo[(size_t)g * FW + i] = 0;
}

__global__ void k_set_meta(Dev E, const uint8_t *mask, const uint8_t *sides, const int32_t *rr) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= E.B || (mask && !mask[g])) return;
    uint32_t *h = E.hdr + (size_t)g * HW;
    if (sides) {
        const int side = sides[g] ? 1 : 0;
        h[H_FLAGS] = (h[H_FLAGS] & ~F_SIDE) | (side ? F_SIDE : 0u);
        const unsigned long long z = zob_board(E.zob, E.root_board + (size_t)g * 96, side);
        h[H_HASHLO] = (uint32_t)z; h[H_HASHHI] = (uint32_t)(z >> 32);
    }
    if (rr) h[H_RR] = (uint32_t)rr[g];
}

__global__ void k_begin(Dev E, const uint8_t *mask, int playouts) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= E.B) return;
    uint32_t *h = E.hdr + (size_t)g * HW;
    const uint32_t f = h[H_FLAGS];
    if (mask ? !mask[g] : F_TERM(f) != 0) return;
    h[H_DONE] = 0;
    h[H_TARGET] = (uint32_t)playouts;
    h[H_FLAGS] = f | F_ACTIVE;
    if (E.fifo) E.fifo[(size_t)g * FW + FI_ITER] = 0;      // a fresh event loop for this search (MCTS_tree.main creates new coroutines)
}

__global__ void k_unfinished(Dev E, int32_t *out) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    int u = 0;
    if (g < E.B) {
        const uint32_t *h = E.hdr + (size_t)g * HW;
        const uint32_t f = h[H_FLAGS];
        if (f & F_ACTIVE) {
            u = (F_PEND(f) || (int)h[H_ROOTCNT] < 0 || (int)h[H_DONE] < (int)h[H_TARGET]) ? 1 : 0;
            if (E.pendK) for (int s = 0; s < E.K; s++) u |= E.pendK[(size_t)g * E.K + s] ? 1 : 0;
        }
    }
    u = __reduce_add_sync(CZ_FULL, u);
    if ((threadIdx.x & 31) == 0 && u) atomicAdd(out, u);
}

// ---- root statistics -> dense staging ---------------------------------------------------
__global__ void k_root_children(Dev E) {
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (g >= E.B) return;
    const uint32_t *h = E.hdr + (size_t)g * HW;
    const int cnt = (int)h[H_ROOTCNT];
    if (lane == 0) E.st_n[g] = cnt;
    if (cnt <= 0) return;
    const uint32_t cs = (uint32_t)((cnt + 7) & ~7);
    const uint32_t *blk = arena_half(E, g, (h[H_FLAGS] & F_CUR) ? 1 : 0) + h[H_ROOTBASE] + HDR;
    for (int i = lane; i < cnt; i += 32) {
        const float W = __uint_as_float(blk[cs + i]);
        const int N = (int)blk[2 * cs + i];
        const size_t o = (size_t)g * CZ_MAXCHILD + i;
        E.st_p[o] = __uint_as_float(blk[i]);
        E.st_w[o] = W;
        E.st_visits[o] = N;
        E.st_q[o] = E.narr == 6 ? __uint_as_float(blk[5 * cs + i]) : (N > 0 ? __fdiv_rn(W, (float)N) : 0.0f);
        E.st_moves[o] = (uint16_t)(blk[3 * cs + i] & 0xFFFFu);
    }
}

// packed game status record (cchess_main.check_end + GameBoard fields), CZ_STATUS_BYTES per game:
//   [0,90) board | 90 side | 91 terminal | 92 winner (int8) | 96 ply i32 | 100 restrict_round i32 | 104 q f32 | 108 root N i32
__device__ __forceinline__ void write_status(const Dev &E, int g, const uint32_t *h, const uint8_t *b, float q, int lane) {
    uint8_t *o = E.st_status + (size_t)g * CZ_STATUS_BYTES;
    for (int i = lane; i < 90; i += 32) o[i] = b[i];
    if (lane == 0) {
        const uint32_t f = h[H_FLAGS];
        o[90] = (f & F_SIDE) ? 1 : 0;
        o[91] = (uint8_t)F_TERM(f);
        o[92] = (uint8_t)(int8_t)F_WIN(f);
        o[93] = o[94] = o[95] = 0;
        int32_t *w = reinterpret_cast<int32_t *>(o + 96);
        w[0] = (int32_t)h[H_PLY];
        w[1] = (int32_t)h[H_RR];
        w[2] = __float_as_int(q);
        w[3] = (int32_t)h[H_ROOTN];
    }
}
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK) k_status(Dev E) {
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (g >= E.B) return;
    write_status(E, g, E.hdr + (size_t)g * HW, E.root_board + (size_t)g * 96, 0.0f, lane);
}

// ---- play a move: board update + MCTS_tree.update_tree with subtree compaction ------------
// Cheney-style breadth-first copy of the chosen child's subtree into the other arena half.  Also leaves the game's
// packed status record (with Q of the move played = mcts.Q(act), main.py:1350) in st_status.
// One node block (a multiple of 8 words at an 8-word-aligned offset) from the old arena half to the new one: 16-byte accesses, up to four
// loads in flight per lane before the first store (a word-by-word loop serialises a memory round trip per 32 words: the re-root was
// 6 ms per ply for 1024 games that way).
__device__ __forceinline__ void copy_block(uint32_t *__restrict__ dst, const uint32_t *__restrict__ src, uint32_t words, int lane) {
    const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
    uint4 *d4 = reinterpret_cast<uint4 *>(dst);
    const uint32_t n4 = words >> 2;
    for (uint32_t j0 = 0; j0 < n4; j0 += 128) {
        uint4 v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) { const uint32_t j = j0 + (uint32_t)(k * 32 + lane); if (j < n4) v[k] = __ldg(s4 + j); }
#pragma unroll
        for (int k = 0; k < 4; k++) { const uint32_t j = j0 + (uint32_t)(k * 32 + lane); if (j < n4) d4[j] = v[k]; }
    }
}

// Plays root child `choice` (0 <= choice < rcnt = the root's child count) of game g: the whole of update_tree + the board update,
// shared by k_play (child index) and k_play_moves (move code).
__device__ __forceinline__ void play_child(const Dev &E, int g, uint32_t *h, uint8_t *b, int choice, int rcnt, int lane) {
    const uint32_t flags = h[H_FLAGS];
    const int cur = (flags & F_CUR) ? 1 : 0;
    const uint32_t *old = arena_half(E, g, cur);
    uint32_t *neu = arena_half(E, g, cur ^ 1);
    const uint32_t rcs = (uint32_t)((rcnt + 7) & ~7);
    const uint32_t *rblk = old + h[H_ROOTBASE] + HDR;
    const uint32_t meta = rblk[3 * rcs + choice], child = rblk[4 * rcs + choice];
    const int N = (int)rblk[2 * rcs + choice];
    const float Wc = __uint_as_float(rblk[rcs + choice]);
    const float q = E.narr == 6 ? __uint_as_float(rblk[5 * rcs + choice]) : (N > 0 ? __fdiv_rn(Wc, (float)N) : 0.0f);
    const int src = meta & 127, dst = (meta >> 7) & 127;
    const int cap = b[dst], mover = b[src];
    const int rr_old = (int)h[H_RR], ply_old = (int)h[H_PLY];
    const unsigned long long z_old = (unsigned long long)h[H_HASHLO] | ((unsigned long long)h[H_HASHHI] << 32);
    __syncwarp();
    uint32_t alloc = 0;
    int ncnt = -1;
    if (child != NONE) {
        ncnt = (int)((meta >> 16) & 0xFFu);
        uint32_t size = HDR + (uint32_t)E.narr * (uint32_t)((ncnt + 7) & ~7);
        copy_block(neu, old + child, size, lane);
        alloc = size;
        __syncwarp();
        uint32_t scan = 0;
        while (scan < alloc) {
            const int c = (int)neu[scan];
            const uint32_t cs = (uint32_t)((c + 7) & ~7);
            uint32_t *blk = neu + scan + HDR;
            for (int i0 = 0; i0 < c; i0 += 32) {
                const int i = i0 + lane;
                uint32_t oc = NONE, sz = 0;
                if (i < c) {
                    oc = blk[4 * cs + i];
                    if (oc != NONE) sz = HDR + (uint32_t)E.narr * ((((blk[3 * cs + i] >> 16) & 0xFFu) + 7) & ~7u);
                }
                int tot;
                const uint32_t off = alloc + (uint32_t)cz::warp_excl_scan((int)sz, lane, tot);
                if (oc != NONE) blk[4 * cs + i] = off;
                unsigned m = __ballot_sync(CZ_FULL, oc != NONE);
                while (m) {
                    const int l = __ffs(m) - 1;
                    m &= m - 1;
                    const uint32_t so = __shfl_sync(CZ_FULL, oc, l), dn = __shfl_sync(CZ_FULL, off, l), n = __shfl_sync(CZ_FULL, sz, l);
                    copy_block(neu + dn, old + so, n, lane);
                }
                alloc += (uint32_t)tot;
                __syncwarp();
            }
            scan += HDR + (uint32_t)E.narr * cs;
        }
    }
    __syncwarp();
    if (lane == 0) {
        b[dst] = (uint8_t)mover;
        b[src] = 0;
        const int side = (flags & F_SIDE) ? 0 : 1;
        const int rr = cap == 0 ? rr_old + 1 : 0;
        uint32_t f = (flags & ~(F_ACTIVE | 6u | F_SIDE | F_CUR)) | (side ? F_SIDE : 0u) | (cur ? 0u : F_CUR);
        // main.py:1532-1545: king missing -> winner, else restrict_round >= 60 -> tie
        if (cap == 1) f = (f & ~0xF00u) | (1u << 8) | (2u << 10);          // 'K' captured: black wins
        else if (cap == 8) f = (f & ~0xF00u) | (1u << 8) | (1u << 10);     // 'k' captured: red wins
        else if (rr >= 60) f = (f & ~0xF00u) | (2u << 8);
        const unsigned long long z = z_old ^ E.zob[mover * 96 + src] ^ E.zob[mover * 96 + dst] ^ E.zob[95] ^ (cap ? E.zob[cap * 96 + dst] : 0ull);
        h[H_FLAGS] = f;
        h[H_RR] = (uint32_t)rr;
        h[H_PLY] = (uint32_t)(ply_old + 1);
        h[H_ROOTN] = (uint32_t)N;
        h[H_ROOTCNT] = (uint32_t)ncnt;
        h[H_ROOTBASE] = 0;
        h[H_ALLOC] = alloc;
        h[H_DONE] = 0;
        h[H_TARGET] = 0;
        h[H_PLEN] = 0;
        h[H_HASHLO] = (uint32_t)z; h[H_HASHHI] = (uint32_t)(z >> 32);
        if (alloc > h[H_MAXALLOC]) h[H_MAXALLOC] = alloc;
    }
    __syncwarp();
    write_status(E, g, h, b, q, lane);
}

__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK) k_play(Dev E) {
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (g >= E.B) return;
    uint32_t *h = E.hdr + (size_t)g * HW;
    uint8_t *b = E.root_board + (size_t)g * 96;
    const int choice = E.st_choice[g];
    if (choice < 0) { write_status(E, g, h, b, 0.0f, lane); return; }
    const int rcnt = (int)h[H_ROOTCNT];
    if (rcnt <= 0 || choice >= rcnt) { if (lane == 0) atomicOr(h + H_ERR, CZ_ERR_NOMOVES); write_status(E, g, h, b, 0.0f, lane); return; }
    play_child(E, g, h, b, choice, rcnt, lane);
}

// update_tree(act) keyed by the move (main.py:272-276): the root child whose META move equals st_choice[g] (CZ_NOMOVE = leave the
// game alone) is found by a lane-parallel scan of the root block, first match by ballot, and played as k_play plays it.  A move
// that is not a child -- or any move at an unexpanded root -- raises CZ_ERR_NOCHILD (the reference's KeyError) and leaves the game
// untouched; its status record is written either way.
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK) k_play_moves(Dev E) {
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
    if (g >= E.B) return;
    uint32_t *h = E.hdr + (size_t)g * HW;
    uint8_t *b = E.root_board + (size_t)g * 96;
    const uint32_t mv = (uint32_t)E.st_choice[g];
    if (mv == CZ_NOMOVE) { write_status(E, g, h, b, 0.0f, lane); return; }
    const int rcnt = (int)h[H_ROOTCNT];
    int choice = -1;
    if (rcnt > 0) {
        const uint32_t rcs = (uint32_t)((rcnt + 7) & ~7);
        const uint32_t *meta = arena_half(E, g, (h[H_FLAGS] & F_CUR) ? 1 : 0) + h[H_ROOTBASE] + HDR + 3 * rcs;
        for (int i0 = 0; i0 < rcnt && choice < 0; i0 += 32) {          // (choice is warp-uniform: it comes from a ballot)
            const int i = i0 + lane;
            const unsigned m = __ballot_sync(CZ_FULL, i < rcnt && (meta[i] & 0xFFFFu) == mv);
            if (m) choice = i0 + __ffs(m) - 1;
        }
    }
    if (choice < 0) { if (lane == 0) atomicOr(h + H_ERR, CZ_ERR_NOCHILD); write_status(E, g, h, b, 0.0f, lane); return; }
    play_child(E, g, h, b, choice, rcnt, lane);
}

// ---- stateless batched rules ------------------------------------------------------------
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK) k_legal_moves(const uint8_t *boards, const uint8_t *sides, int n, uint16_t *moves, int32_t *counts) {
    __shared__ WarpSmem smem[WARPS_PER_BLOCK];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, g = blockIdx.x * WARPS_PER_BLOCK + w;
    if (g >= n) return;
    WarpSmem &S = smem[w];
    for (int i = lane; i < 90; i += 32) S.board[i] = boards[(size_t)g * 90 + i];
    __syncwarp();
    int c = cz::warp_legal_moves(S.board, sides[g], S.moves, S.scratch, lane);
    if (lane == 0) counts[g] = c;
    if (c > CZ_MAXCHILD) c = CZ_MAXCHILD;
    for (int i = lane; i < CZ_MAXCHILD; i += 32) moves[(size_t)g * CZ_MAXCHILD + i] = i < c ? S.moves[i] : (uint16_t)0;
}

template <typename T>
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK) k_encode(const uint8_t *boards, const uint8_t *sides, int n, T *out) {
    __shared__ WarpSmem smem[WARPS_PER_BLOCK];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, g = blockIdx.x * WARPS_PER_BLOCK + w;
    if (g >= n) return;
    WarpSmem &S = smem[w];
    for (int i = lane; i < 90; i += 32) S.board[i] = boards[(size_t)g * 90 + i];
    __syncwarp();
    cz::warp_encode<T>(S.board, sides[g], out + (size_t)g * CZ_ENC_LEN, lane);
}

__global__ void k_apply(uint8_t *boards, const uint16_t *moves, int n, uint8_t *captured) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n) return;
    uint8_t *b = boards + (size_t)g * 90;
    const int src = moves[g] & 127, dst = (moves[g] >> 7) & 127;
    captured[g] = b[dst];
    b[dst] = b[src];
    b[src] = 0;
}

const int16_t *device_label_table(int device) {
    static const int16_t *tab[64] = {nullptr};
    if (device < 0 || device >= 64) return nullptr;
    if (!tab[device]) {
        int16_t *p = nullptr;
        if (cudaMalloc(&p, sizeof(labels().of)) != cudaSuccess) return nullptr;
        if (cudaMemcpy(p, labels().of, sizeof(labels().of), cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
        tab[device] = p;
    }
    return tab[device];
}

// Zobrist keys: 16 piece codes x 96 squares of splitmix64 output (fixed seed), entry [0][95] = side to move.
const unsigned long long *device_zobrist_table(int device) {
    static const unsigned long long *tab[64] = {nullptr};
    if (device < 0 || device >= 64) return nullptr;
    if (!tab[device]) {
        std::vector<unsigned long long> z(16 * 96);
        unsigned long long x = 0x9E3779B97F4A7C15ull;
        for (auto &v : z) {
            x += 0x9E3779B97F4A7C15ull;
            unsigned long long t = x;
            t = (t ^ (t >> 30)) * 0xBF58476D1CE4E5B9ull;
            t = (t ^ (t >> 27)) * 0x94D049BB133111EBull;
            v = t ^ (t >> 31);
        }
        unsigned long long *p = nullptr;
        if (cudaMalloc(&p, z.size() * 8) != cudaSuccess) return nullptr;
        if (cudaMemcpy(p, z.data(), z.size() * 8, cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
        tab[device] = p;
    }
    return tab[device];
}

inline int nblk(int n, int per) { return (n + per - 1) / per; }

}  // namespace

struct cz_engine {
    Dev d;
    int device;
    int wpb = WARPS_PER_BLOCK;   // warps per CTA of the wave kernels: ceil(B / #SMs) clamped to [1, MAX_WPB]
    std::vector<void *> allocs;
    // pinned host staging
    int32_t *h_n = nullptr, *h_visits = nullptr, *h_choice = nullptr, *h_i32 = nullptr;
    uint16_t *h_moves = nullptr;
    float *h_f = nullptr;
    uint8_t *h_status = nullptr;
    uint32_t *h_hdr = nullptr;
    uint8_t *d_mask = nullptr, *d_boards = nullptr, *d_sides = nullptr;
    int32_t *d_rr = nullptr;
};

extern "C" {

const char *cz_last_error(void) { return g_err.c_str(); }
int cz_version(void) { return 2; }

int cz_labels(char *out) {
    if (!out) return fail(CZ_EINVAL, "cz_labels: null");
    memcpy(out, labels().text, sizeof(labels().text));
    return CZ_OK;
}
int cz_label_index(int s, int d) {
    if (s < 0 || s >= CZ_NSQ || d < 0 || d >= CZ_NSQ) return -1;
    return labels().of[s * CZ_NSQ + d];
}
int cz_unflipped_index(int32_t *out) {
    if (!out) return fail(CZ_EINVAL, "cz_unflipped_index: null");
    memcpy(out, labels().unflipped, sizeof(labels().unflipped));
    return CZ_OK;
}

int cz_from_state(const char *s, uint8_t *board) {
    if (!s || !board) return fail(CZ_EINVAL, "cz_from_state: null");
    static const char *pc = ".KARBNPCkarbnpc";
    int sq = 0;
    for (; *s; s++) {
        const char c = *s;
        if (c == '/') continue;
        if (c >= '1' && c <= '9') {
            for (int k = 0; k < c - '0'; k++) { if (sq >= CZ_NSQ) return fail(CZ_EINVAL, "cz_from_state: too many squares"); board[sq++] = 0; }
            continue;
        }
        char cc = c;  // aliases accepted by the reference's move generator (main.py:835, 846, 857, 873)
        if (cc == 'h') cc = 'n'; else if (cc == 'H') cc = 'N'; else if (cc == 'e') cc = 'b'; else if (cc == 'E') cc = 'B';
        const char *f = strchr(pc + 1, cc);
        if (!f || sq >= CZ_NSQ) return fail(CZ_EINVAL, "cz_from_state: bad character");
        board[sq++] = (uint8_t)(f - pc);
    }
    return sq == CZ_NSQ ? CZ_OK : fail(CZ_EINVAL, "cz_from_state: not 90 squares");
}

int cz_to_state(const uint8_t *board, char *out) {
    if (!out || !board) return fail(CZ_EINVAL, "cz_to_state: null");
    static const char *pc = ".KARBNPCkarbnpc";
    int n = 0;
    for (int y = 0; y < 10; y++) {
        int run = 0;
        for (int x = 0; x < 9; x++) {
            const int p = board[y * 9 + x];
            if (p > 14) return fail(CZ_EINVAL, "cz_to_state: bad piece code");
            if (!p) { run++; continue; }
            if (run) { out[n++] = char('0' + run); run = 0; }
            out[n++] = pc[p];
        }
        if (run) out[n++] = char('0' + run);
        if (y < 9) out[n++] = '/';
    }
    out[n] = 0;
    return CZ_OK;
}

int cz_legal_moves_dev(const uint8_t *boards, const uint8_t *sides, int n, uint16_t *moves, int32_t *counts, void *stream) {
    if (n <= 0) return CZ_OK;
    k_legal_moves<<<nblk(n, WARPS_PER_BLOCK), 32 * WARPS_PER_BLOCK, 0, (cudaStream_t)stream>>>(boards, sides, n, moves, counts);
    CUDA_TRY(cudaGetLastError());
    return CZ_OK;
}

int cz_encode_dev(const uint8_t *boards, const uint8_t *sides, int n, void *out, int dtype, void *stream) {
    if (n <= 0) return CZ_OK;
    dim3 gr(nblk(n, WARPS_PER_BLOCK)), bl(32 * WARPS_PER_BLOCK);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == CZ_F32) k_encode<float><<<gr, bl, 0, st>>>(boards, sides, n, (float *)out);
    else if (dtype == CZ_BF16) k_encode<__nv_bfloat16><<<gr, bl, 0, st>>>(boards, sides, n, (__nv_bfloat16 *)out);
    else if (dtype == CZ_F16) k_encode<__half><<<gr, bl, 0, st>>>(boards, sides, n, (__half *)out);
    else return fail(CZ_EINVAL, "cz_encode_dev: dtype");
    CUDA_TRY(cudaGetLastError());
    return CZ_OK;
}

extern "C++" {
// frees the scratch device buffers of the stateless batch entry points on every exit path
struct DevBufs {
    std::vector<void *> p;
    ~DevBufs() { for (void *q : p) cudaFree(q); }
    template <typename T> cudaError_t alloc(T **out, size_t bytes) {
        void *q = nullptr;
        cudaError_t e = cudaMalloc(&q, bytes);
        if (e == cudaSuccess) { p.push_back(q); *out = (T *)q; }
        return e;
    }
};
}  // extern "C++"

static int batch_io(DevBufs &bufs, int device, const uint8_t *boards, const uint8_t *sides, int n, uint8_t **db, uint8_t **ds) {
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(bufs.alloc(db, (size_t)n * 90));
    CUDA_TRY(cudaMemcpy(*db, boards, (size_t)n * 90, cudaMemcpyHostToDevice));
    if (sides) {
        CUDA_TRY(bufs.alloc(ds, (size_t)n));
        CUDA_TRY(cudaMemcpy(*ds, sides, (size_t)n, cudaMemcpyHostToDevice));
    }
    return CZ_OK;
}

int cz_legal_moves_batch(int device, const uint8_t *boards, const uint8_t *sides, int n, uint16_t *moves, int32_t *counts) {
    if (n < 0 || (n && (!boards || !sides || !moves || !counts))) return fail(CZ_EINVAL, "cz_legal_moves_batch: null");
    if (n == 0) return CZ_OK;
    DevBufs bufs;
    uint8_t *db = nullptr, *ds = nullptr;
    uint16_t *dm = nullptr;
    int32_t *dc = nullptr;
    int rc = batch_io(bufs, device, boards, sides, n, &db, &ds);
    if (rc) return rc;
    CUDA_TRY(bufs.alloc(&dm, (size_t)n * CZ_MAXCHILD * 2));
    CUDA_TRY(bufs.alloc(&dc, (size_t)n * 4));
    rc = cz_legal_moves_dev(db, ds, n, dm, dc, nullptr);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpy(moves, dm, (size_t)n * CZ_MAXCHILD * 2, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(counts, dc, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return CZ_OK;
}

int cz_apply_moves_batch(int device, uint8_t *boards, const uint16_t *moves, int n, uint8_t *captured) {
    if (n < 0 || (n && (!boards || !moves || !captured))) return fail(CZ_EINVAL, "cz_apply_moves_batch: null");
    if (n == 0) return CZ_OK;
    DevBufs bufs;
    uint8_t *db = nullptr, *ds = nullptr, *dcap = nullptr;
    uint16_t *dm = nullptr;
    int rc = batch_io(bufs, device, boards, nullptr, n, &db, &ds);
    if (rc) return rc;
    CUDA_TRY(bufs.alloc(&dm, (size_t)n * 2));
    CUDA_TRY(bufs.alloc(&dcap, (size_t)n));
    CUDA_TRY(cudaMemcpy(dm, moves, (size_t)n * 2, cudaMemcpyHostToDevice));
    k_apply<<<nblk(n, 128), 128>>>(db, dm, n, dcap);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpy(boards, db, (size_t)n * 90, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(captured, dcap, (size_t)n, cudaMemcpyDeviceToHost));
    return CZ_OK;
}

int cz_encode_batch(int device, const uint8_t *boards, const uint8_t *sides, int n, float *out) {
    if (n < 0 || (n && (!boards || !sides || !out))) return fail(CZ_EINVAL, "cz_encode_batch: null");
    if (n == 0) return CZ_OK;
    DevBufs bufs;
    uint8_t *db = nullptr, *ds = nullptr;
    float *dout = nullptr;
    int rc = batch_io(bufs, device, boards, sides, n, &db, &ds);
    if (rc) return rc;
    CUDA_TRY(bufs.alloc(&dout, (size_t)n * CZ_ENC_LEN * 4));
    rc = cz_encode_dev(db, ds, n, dout, CZ_F32, nullptr);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpy(out, dout, (size_t)n * CZ_ENC_LEN * 4, cudaMemcpyDeviceToHost));
    return CZ_OK;
}

// ------------------------------------------------------------------------------------------
extern "C++" {
template <typename T>
static int dalloc(cz_engine *e, T **p, size_t count, bool zero = true) {
    void *q = nullptr;
    cudaError_t ce = cudaMalloc(&q, count * sizeof(T));
    if (ce != cudaSuccess) return fail(CZ_ENOMEM, "cudaMalloc", ce);
    if (zero) cudaMemset(q, 0, count * sizeof(T));
    e->allocs.push_back(q);
    *p = (T *)q;
    return CZ_OK;
}
// every exit of cz_engine_create_ex after `new` goes through here: nothing (arena, pinned staging) leaks on failure
static int create_failed(cz_engine *e, int code, const char *what, cudaError_t ce = cudaSuccess) {
    const int rc = fail(code, what, ce);
    const std::string keep = g_err;
    cz_engine_destroy(e);
    g_err = keep;
    return rc;
}
}  // extern "C++"

int cz_engine_create(int n_games, int64_t arena_words, int device, cz_engine **out) {
    return cz_engine_create_ex(n_games, arena_words, device, 1, out);
}

int cz_engine_leaves(const cz_engine *e) { return e ? e->d.K : CZ_EINVAL; }

extern "C++" { static int create_engine(int n_games, int64_t arena_words, int device, int leaves, bool fifo, cz_engine **out); }

int cz_engine_create_ex(int n_games, int64_t arena_words, int device, int leaves, cz_engine **out) {
    return create_engine(n_games, arena_words, device, leaves, false, out);
}
int cz_engine_create_fifo(int n_games, int64_t arena_words, int device, int search_threads, cz_engine **out) {
    if (search_threads < 1 || search_threads > 32) return fail(CZ_EINVAL, "cz_engine_create_fifo: search_threads must be 1..32");
    return create_engine(n_games, arena_words, device, search_threads, true, out);
}
int cz_engine_is_fifo(const cz_engine *e) { return e ? (e->d.fifo != nullptr) : CZ_EINVAL; }

extern "C++" {
static int create_engine(int n_games, int64_t arena_words, int device, int leaves, bool fifo, cz_engine **out) {
    if (n_games <= 0 || !out) return fail(CZ_EINVAL, "cz_engine_create: bad arguments");
    const bool multi = fifo || leaves != 1;    // leaves == -1: the leaf-parallel kernel with one slot (test hook)
    const int K = leaves < 0 ? -leaves : leaves;
    if (K < 1 || K > 64) return fail(CZ_EINVAL, "cz_engine_create_ex: leaves must be 1..64");
    if (arena_words <= 0) arena_words = 2ll << 20;     // 8 MiB per half: 2.7x the high-water mark of a 1200-playout self-play soak (0.74 Mi words)
    if (arena_words < 4096 || arena_words >= (1ll << 31)) return fail(CZ_EINVAL, "cz_engine_create: arena_words out of range");
    arena_words = (arena_words + 31) & ~31ll;
    CUDA_TRY(cudaSetDevice(device));
    cz_engine *e = new cz_engine();
    e->device = device;
    Dev &d = e->d;
    memset(&d, 0, sizeof(d));
    d.B = n_games;
    d.A = arena_words;
    d.K = K;
    d.narr = fifo ? 6 : 5;
    {
        int sms = 148;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms <= 0) sms = 148;
        int w = (n_games + sms - 1) / sms;
        e->wpb = w < 1 ? 1 : (w > MAX_WPB ? MAX_WPB : w);
    }
    const size_t B = (size_t)n_games;
    int rc = 0;
#define AL(ptr, cnt) if (!rc) rc = dalloc(e, &ptr, cnt)
    AL(d.hdr, B * HW); AL(d.root_board, B * 96); AL(d.leaf_board, B * 96); AL(d.path, B * MAXD);
    AL(d.cnt_expand, B); AL(d.cnt_playout, B); AL(d.cnt_L, B); AL(d.cnt_c, B); AL(d.cnt_C, B); AL(d.leaf_hash, B * K);
    AL(d.st_n, B); AL(d.st_visits, B * CZ_MAXCHILD); AL(d.st_choice, B); AL(d.st_moves, B * CZ_MAXCHILD);
    AL(d.st_w, B * CZ_MAXCHILD); AL(d.st_p, B * CZ_MAXCHILD); AL(d.st_q, B * CZ_MAXCHILD); AL(d.st_count, 8); AL(d.st_status, B * CZ_STATUS_BYTES);
    AL(e->d_mask, B); AL(e->d_boards, B * 90); AL(e->d_sides, B); AL(e->d_rr, B);
    if (multi) { AL(d.pendK, B * K); AL(d.plenK, B * K); AL(d.pathK, B * K * MAXD); AL(d.leafK, B * K * 96); }
    if (fifo) { AL(d.fifo, B * FW); AL(d.live_mask, B); AL(d.row_map, B * K); AL(d.src_of, B * K); AL(d.dense_count, 8); }
    if (!rc) { uint32_t *a = nullptr; rc = dalloc(e, &a, B * 2 * (size_t)arena_words, false); d.arena = a; }
#undef AL
    if (rc) { const std::string keep = g_err; cz_engine_destroy(e); g_err = keep; return rc; }
    d.label_of = device_label_table(device);
    d.zob = device_zobrist_table(device);
    if (!d.label_of || !d.zob) return create_failed(e, CZ_ECUDA, "label / zobrist table upload");
    const size_t hb = B * CZ_MAXCHILD;
    if (cudaMallocHost(&e->h_n, B * 4) || cudaMallocHost(&e->h_visits, hb * 4) || cudaMallocHost(&e->h_choice, B * 4) ||
        cudaMallocHost(&e->h_moves, hb * 2) || cudaMallocHost(&e->h_f, hb * 4 * 3) || cudaMallocHost(&e->h_status, B * CZ_STATUS_BYTES) ||
        cudaMallocHost(&e->h_i32, 64) || cudaMallocHost(&e->h_hdr, B * HW * 4))
        return create_failed(e, CZ_ENOMEM, "cudaMallocHost");
    {
        uint8_t sb[96] = {0};
        if (cz_from_state("RNBAKABNR/9/1C5C1/P1P1P1P1P/9/9/p1p1p1p1p/1c5c1/9/rnbakabnr", sb) != CZ_OK) return create_failed(e, CZ_EINVAL, "start position");
        cudaError_t ce = cudaMemcpyToSymbol(c_start, sb, 96);   // GameBoard.__init__ state, main.py:585
        if (ce != cudaSuccess) return create_failed(e, CZ_ECUDA, "cudaMemcpyToSymbol(c_start)", ce);
    }
    k_reset<<<nblk(n_games, 128), 128>>>(d, nullptr, nullptr, nullptr, nullptr);
    cudaError_t ce = cudaDeviceSynchronize();
    if (ce != cudaSuccess) return create_failed(e, CZ_ECUDA, "k_reset", ce);
    *out = e;
    return CZ_OK;
}
}  // extern "C++"

int cz_engine_destroy(cz_engine *e) {
    if (!e) return CZ_OK;
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    for (void *p : e->allocs) cudaFree(p);
    cudaFreeHost(e->h_n); cudaFreeHost(e->h_visits); cudaFreeHost(e->h_choice); cudaFreeHost(e->h_moves);
    cudaFreeHost(e->h_f); cudaFreeHost(e->h_status); cudaFreeHost(e->h_i32); cudaFreeHost(e->h_hdr);
    delete e;
    return CZ_OK;
}

int cz_engine_n_games(const cz_engine *e) { return e ? e->d.B : CZ_EINVAL; }

int cz_engine_reset(cz_engine *e, void *stream, const uint8_t *mask, const uint8_t *boards, const uint8_t *sides, const int32_t *rr) {
    if (!e) return fail(CZ_EINVAL, "null engine");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t B = (size_t)e->d.B;
    CUDA_TRY(cudaSetDevice(e->device));
    if (mask) CUDA_TRY(cudaMemcpyAsync(e->d_mask, mask, B, cudaMemcpyHostToDevice, st));
    if (boards) CUDA_TRY(cudaMemcpyAsync(e->d_boards, boards, B * 90, cudaMemcpyHostToDevice, st));
    if (sides) CUDA_TRY(cudaMemcpyAsync(e->d_sides, sides, B, cudaMemcpyHostToDevice, st));
    if (rr) CUDA_TRY(cudaMemcpyAsync(e->d_rr, rr, B * 4, cudaMemcpyHostToDevice, st));
    k_reset<<<nblk(e->d.B, 128), 128, 0, st>>>(e->d, mask ? e->d_mask : nullptr, boards ? e->d_boards : nullptr,
                                               sides ? e->d_sides : nullptr, rr ? e->d_rr : nullptr);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(st));   // host buffers may be pageable: do not return before they are consumed
    return CZ_OK;
}

int cz_engine_set_root_meta(cz_engine *e, void *stream, const uint8_t *mask, const uint8_t *sides, const int32_t *rr) {
    if (!e) return fail(CZ_EINVAL, "null engine");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t B = (size_t)e->d.B;
    CUDA_TRY(cudaSetDevice(e->device));
    if (mask) CUDA_TRY(cudaMemcpyAsync(e->d_mask, mask, B, cudaMemcpyHostToDevice, st));
    if (sides) CUDA_TRY(cudaMemcpyAsync(e->d_sides, sides, B, cudaMemcpyHostToDevice, st));
    if (rr) CUDA_TRY(cudaMemcpyAsync(e->d_rr, rr, B * 4, cudaMemcpyHostToDevice, st));
    k_set_meta<<<nblk(e->d.B, 128), 128, 0, st>>>(e->d, mask ? e->d_mask : nullptr, sides ? e->d_sides : nullptr, rr ? e->d_rr : nullptr);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(st));
    return CZ_OK;
}

int cz_engine_begin_search(cz_engine *e, void *stream, const uint8_t *mask, int playouts) {
    if (!e || playouts < 0) return fail(CZ_EINVAL, "cz_engine_begin_search: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(e->device));
    if (mask) CUDA_TRY(cudaMemcpyAsync(e->d_mask, mask, (size_t)e->d.B, cudaMemcpyHostToDevice, st));
    k_begin<<<nblk(e->d.B, 128), 128, 0, st>>>(e->d, mask ? e->d_mask : nullptr, playouts);
    CUDA_TRY(cudaGetLastError());
    if (mask) CUDA_TRY(cudaStreamSynchronize(st));
    return CZ_OK;
}

extern "C++" {
template <bool X, bool S>
static int launch_wave(cz_engine *e, void *stream, void *nn_in, int dt, const float *logits, const float *value) {
    dim3 gr(nblk(e->d.B, e->wpb)), bl(32 * e->wpb);
    const size_t sm = (size_t)e->wpb * sizeof(WarpSmem);
    cudaStream_t st = (cudaStream_t)stream;
    if (dt == CZ_F32) k_wave<float, X, S><<<gr, bl, sm, st>>>(e->d, (float *)nn_in, logits, value);
    else if (dt == CZ_BF16) k_wave<__nv_bfloat16, X, S><<<gr, bl, sm, st>>>(e->d, (__nv_bfloat16 *)nn_in, logits, value);
    else if (dt == CZ_F16) k_wave<__half, X, S><<<gr, bl, sm, st>>>(e->d, (__half *)nn_in, logits, value);
    else if (dt == CZ_BOARD) k_wave<uint8_t, X, S><<<gr, bl, sm, st>>>(e->d, (uint8_t *)nn_in, logits, value);
    else return fail(CZ_EINVAL, "wave: nn_dtype");
    CUDA_TRY(cudaGetLastError());
    return CZ_OK;
}
}  // extern "C++"

int cz_engine_wave(cz_engine *e, void *stream, void *nn_in, int nn_dtype, const float *logits, const float *value) {
    if (!e || !nn_in || !logits || !value) return fail(CZ_EINVAL, "cz_engine_wave: null");
    if (e->d.fifo) {    // search_threads = K schedule of the reference (canonical FIFO form)
        dim3 gr(nblk(e->d.B, e->wpb)), bl(32 * e->wpb);
        const size_t sm = (size_t)e->wpb * sizeof(WarpSmem);
        cudaStream_t st = (cudaStream_t)stream;
        if (nn_dtype == CZ_F32) k_wave_fifo<float><<<gr, bl, sm, st>>>(e->d, (float *)nn_in, logits, value);
        else if (nn_dtype == CZ_BF16) k_wave_fifo<__nv_bfloat16><<<gr, bl, sm, st>>>(e->d, (__nv_bfloat16 *)nn_in, logits, value);
        else if (nn_dtype == CZ_F16) k_wave_fifo<__half><<<gr, bl, sm, st>>>(e->d, (__half *)nn_in, logits, value);
        else if (nn_dtype == CZ_BOARD) k_wave_fifo<uint8_t><<<gr, bl, sm, st>>>(e->d, (uint8_t *)nn_in, logits, value);
        else return fail(CZ_EINVAL, "wave: nn_dtype");
        CUDA_TRY(cudaGetLastError());
        return CZ_OK;
    }
    if (e->d.pendK) {   // leaf-parallel engine
        dim3 gr(nblk(e->d.B, e->wpb)), bl(32 * e->wpb);
        const size_t sm = (size_t)e->wpb * sizeof(WarpSmem);
        cudaStream_t st = (cudaStream_t)stream;
        if (nn_dtype == CZ_F32) k_wave_multi<float><<<gr, bl, sm, st>>>(e->d, (float *)nn_in, logits, value);
        else if (nn_dtype == CZ_BF16) k_wave_multi<__nv_bfloat16><<<gr, bl, sm, st>>>(e->d, (__nv_bfloat16 *)nn_in, logits, value);
        else if (nn_dtype == CZ_F16) k_wave_multi<__half><<<gr, bl, sm, st>>>(e->d, (__half *)nn_in, logits, value);
        else if (nn_dtype == CZ_BOARD) k_wave_multi<uint8_t><<<gr, bl, sm, st>>>(e->d, (uint8_t *)nn_in, logits, value);
        else return fail(CZ_EINVAL, "wave: nn_dtype");
        CUDA_TRY(cudaGetLastError());
        return CZ_OK;
    }
    return launch_wave<true, true>(e, stream, nn_in, nn_dtype, logits, value);
}
// search_threads = K engines: one wave with row compaction.  nn_stage [B*K rows] receives every slot's input row as cz_engine_wave
// would write it; nn_dense [B*K rows] receives the rows that need an evaluation, densely, in (game, slot) order; logits / value are
// read through the row map of the PREVIOUS cz_engine_wave_compact call (so the caller evaluates nn_dense[0 .. n) into
// logits[0 .. n) / value[0 .. n), n from cz_engine_live_rows, between two calls).  Do not mix with cz_engine_wave inside a search.
int cz_engine_wave_compact(cz_engine *e, void *stream, void *nn_stage, void *nn_dense, int nn_dtype, const float *logits, const float *value) {
    if (!e || !nn_stage || !nn_dense || !logits || !value) return fail(CZ_EINVAL, "cz_engine_wave_compact: null");
    if (!e->d.fifo) return fail(CZ_EINVAL, "cz_engine_wave_compact: needs a search_threads engine (cz_engine_create_fifo)");
    const int row_bytes = nn_dtype == CZ_BOARD ? 96 : nn_dtype == CZ_F32 ? 1260 * 4 : (nn_dtype == CZ_F16 || nn_dtype == CZ_BF16) ? 1260 * 2 : 0;
    if (!row_bytes) return fail(CZ_EINVAL, "wave: nn_dtype");
    cudaStream_t st = (cudaStream_t)stream;
    e->d.compact = 1;
    const int rc = cz_engine_wave(e, stream, nn_stage, nn_dtype, logits, value);
    e->d.compact = 0;
    if (rc) return rc;
    k_compact_scan<<<1, 1024, 0, st>>>(e->d);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->device);
    k_compact_rows<<<2 * sms, 256, 0, st>>>(e->d, (const uint2 *)nn_stage, (uint2 *)nn_dense, row_bytes / 8);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(e->h_i32 + 8, e->d.dense_count, 4, cudaMemcpyDeviceToHost, st));
    return CZ_OK;
}
// Rows of the dense batch the last cz_engine_wave_compact produced (synchronises the stream).
int cz_engine_live_rows(cz_engine *e, void *stream, int32_t *out_rows) {
    if (!e || !out_rows) return fail(CZ_EINVAL, "cz_engine_live_rows: null");
    CUDA_TRY(cudaSetDevice(e->device));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    *out_rows = e->h_i32[8];
    return CZ_OK;
}

int cz_engine_select(cz_engine *e, void *stream, void *nn_in, int nn_dtype) {
    if (!e || !nn_in) return fail(CZ_EINVAL, "cz_engine_select: null");
    if (e->d.pendK) return fail(CZ_EINVAL, "cz_engine_select: leaf-parallel engines only support cz_engine_wave");
    return launch_wave<false, true>(e, stream, nn_in, nn_dtype, nullptr, nullptr);
}
int cz_engine_expand_backup(cz_engine *e, void *stream, const float *logits, const float *value) {
    if (!e || !logits || !value) return fail(CZ_EINVAL, "cz_engine_expand_backup: null");
    if (e->d.pendK) return fail(CZ_EINVAL, "cz_engine_expand_backup: leaf-parallel engines only support cz_engine_wave");
    return launch_wave<true, false>(e, stream, (void *)logits, CZ_F32, logits, value);
}

int cz_engine_enable_hashing(cz_engine *e, int on) {
    if (!e) return fail(CZ_EINVAL, "null engine");
    e->d.hash_on = on ? 1 : 0;   // read by every wave launched (or captured) afterwards
    return CZ_OK;
}
int cz_engine_leaf_hashes(cz_engine *e, uint64_t **dev_keys) {
    if (!e || !dev_keys) return fail(CZ_EINVAL, "cz_engine_leaf_hashes: null");
    *dev_keys = (uint64_t *)e->d.leaf_hash;
    return CZ_OK;
}

int cz_engine_unfinished_async(cz_engine *e, void *stream, int32_t *dev_count) {
    if (!e || !dev_count) return fail(CZ_EINVAL, "cz_engine_unfinished_async: null");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(dev_count, 0, 4, st));
    k_unfinished<<<nblk(e->d.B, 128), 128, 0, st>>>(e->d, dev_count);
    CUDA_TRY(cudaGetLastError());
    return CZ_OK;
}

int cz_engine_unfinished(cz_engine *e, void *stream, int32_t *out_count) {
    if (!e || !out_count) return fail(CZ_EINVAL, "cz_engine_unfinished: null");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(e->device));
    int rc = cz_engine_unfinished_async(e, stream, e->d.st_count);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(e->h_i32, e->d.st_count, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    *out_count = e->h_i32[0];
    return CZ_OK;
}

int cz_engine_root_children(cz_engine *e, void *stream, int32_t *n_children, uint16_t *moves, int32_t *visits, float *w, float *p, float *q) {
    if (!e) return fail(CZ_EINVAL, "null engine");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t B = (size_t)e->d.B, hb = B * CZ_MAXCHILD;
    CUDA_TRY(cudaSetDevice(e->device));
    k_root_children<<<nblk(e->d.B, WARPS_PER_BLOCK), 32 * WARPS_PER_BLOCK, 0, st>>>(e->d);
    CUDA_TRY(cudaGetLastError());
    if (n_children) CUDA_TRY(cudaMemcpyAsync(e->h_n, e->d.st_n, B * 4, cudaMemcpyDeviceToHost, st));
    if (moves) CUDA_TRY(cudaMemcpyAsync(e->h_moves, e->d.st_moves, hb * 2, cudaMemcpyDeviceToHost, st));
    if (visits) CUDA_TRY(cudaMemcpyAsync(e->h_visits, e->d.st_visits, hb * 4, cudaMemcpyDeviceToHost, st));
    if (w) CUDA_TRY(cudaMemcpyAsync(e->h_f, e->d.st_w, hb * 4, cudaMemcpyDeviceToHost, st));
    if (p) CUDA_TRY(cudaMemcpyAsync(e->h_f + hb, e->d.st_p, hb * 4, cudaMemcpyDeviceToHost, st));
    if (q) CUDA_TRY(cudaMemcpyAsync(e->h_f + 2 * hb, e->d.st_q, hb * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (n_children) memcpy(n_children, e->h_n, B * 4);
    if (moves) memcpy(moves, e->h_moves, hb * 2);
    if (visits) memcpy(visits, e->h_visits, hb * 4);
    if (w) memcpy(w, e->h_f, hb * 4);
    if (p) memcpy(p, e->h_f + hb, hb * 4);
    if (q) memcpy(q, e->h_f + 2 * hb, hb * 4);
    return CZ_OK;
}

int cz_engine_play_status(cz_engine *e, void *stream, const int32_t *child_index, uint8_t *status) {
    if (!e || !child_index) return fail(CZ_EINVAL, "cz_engine_play: null");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t B = (size_t)e->d.B;
    CUDA_TRY(cudaSetDevice(e->device));
    memcpy(e->h_choice, child_index, B * 4);
    CUDA_TRY(cudaMemcpyAsync(e->d.st_choice, e->h_choice, B * 4, cudaMemcpyHostToDevice, st));
    k_play<<<nblk(e->d.B, WARPS_PER_BLOCK), 32 * WARPS_PER_BLOCK, 0, st>>>(e->d);
    CUDA_TRY(cudaGetLastError());
    if (status) CUDA_TRY(cudaMemcpyAsync(e->h_status, e->d.st_status, B * CZ_STATUS_BYTES, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));   // h_choice is reused by the next call
    if (status) memcpy(status, e->h_status, B * CZ_STATUS_BYTES);
    return CZ_OK;
}

int cz_engine_play(cz_engine *e, void *stream, const int32_t *child_index) { return cz_engine_play_status(e, stream, child_index, nullptr); }

int cz_engine_play_moves(cz_engine *e, void *stream, const uint16_t *moves, uint8_t *status) {
    if (!e || !moves) return fail(CZ_EINVAL, "cz_engine_play_moves: null");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t B = (size_t)e->d.B;
    CUDA_TRY(cudaSetDevice(e->device));
    for (size_t g = 0; g < B; g++) e->h_choice[g] = (int32_t)moves[g];     // the move codes travel in the child-index buffer
    CUDA_TRY(cudaMemcpyAsync(e->d.st_choice, e->h_choice, B * 4, cudaMemcpyHostToDevice, st));
    k_play_moves<<<nblk(e->d.B, WARPS_PER_BLOCK), 32 * WARPS_PER_BLOCK, 0, st>>>(e->d);
    CUDA_TRY(cudaGetLastError());
    if (status) CUDA_TRY(cudaMemcpyAsync(e->h_status, e->d.st_status, B * CZ_STATUS_BYTES, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));   // h_choice is reused by the next call
    if (status) memcpy(status, e->h_status, B * CZ_STATUS_BYTES);
    return CZ_OK;
}

int cz_engine_status_packed(cz_engine *e, void *stream, uint8_t *status) {
    if (!e || !status) return fail(CZ_EINVAL, "cz_engine_status_packed: null");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t B = (size_t)e->d.B;
    CUDA_TRY(cudaSetDevice(e->device));
    k_status<<<nblk(e->d.B, WARPS_PER_BLOCK), 32 * WARPS_PER_BLOCK, 0, st>>>(e->d);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(e->h_status, e->d.st_status, B * CZ_STATUS_BYTES, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    memcpy(status, e->h_status, B * CZ_STATUS_BYTES);
    return CZ_OK;
}

int cz_engine_status(cz_engine *e, void *stream, uint8_t *terminal, int8_t *winner, int32_t *ply, int32_t *rr, uint8_t *side, uint8_t *boards) {
    if (!e) return fail(CZ_EINVAL, "null engine");
    const size_t B = (size_t)e->d.B;
    std::vector<uint8_t> rec(B * CZ_STATUS_BYTES);
    int rc = cz_engine_status_packed(e, stream, rec.data());   // one kernel, one device->host copy, one synchronisation
    if (rc) return rc;
    for (size_t g = 0; g < B; g++) {
        const uint8_t *r = rec.data() + g * CZ_STATUS_BYTES;
        int32_t w[4];
        memcpy(w, r + 96, 16);
        if (boards) memcpy(boards + g * 90, r, 90);
        if (side) side[g] = r[90];
        if (terminal) terminal[g] = r[91];
        if (winner) winner[g] = (int8_t)r[92];
        if (ply) ply[g] = w[0];
        if (rr) rr[g] = w[1];
    }
    return CZ_OK;
}

extern "C++" {
static int fetch_headers(cz_engine *e, void *stream) {
    CUDA_TRY(cudaSetDevice(e->device));
    CUDA_TRY(cudaMemcpyAsync(e->h_hdr, e->d.hdr, (size_t)e->d.B * HW * 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    return CZ_OK;
}
}  // extern "C++"

int cz_engine_counters(cz_engine *e, void *stream, int64_t *out) {
    if (!e || !out) return fail(CZ_EINVAL, "cz_engine_counters: null");
    const size_t B = (size_t)e->d.B;
    int rc = fetch_headers(e, stream);
    if (rc) return rc;
    std::vector<unsigned long long> a(B), b(B), c(B), d(B), cc(B);
    CUDA_TRY(cudaMemcpy(a.data(), e->d.cnt_expand, B * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(b.data(), e->d.cnt_playout, B * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(c.data(), e->d.cnt_L, B * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(d.data(), e->d.cnt_c, B * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(cc.data(), e->d.cnt_C, B * 8, cudaMemcpyDeviceToHost));
    for (int i = 0; i < 9; i++) out[i] = 0;
    out[6] = -1;
    for (size_t g = 0; g < B; g++) {
        const uint32_t *h = e->h_hdr + g * HW;
        out[0] += (int64_t)a[g]; out[1] += (int64_t)b[g]; out[2] += (int64_t)c[g]; out[3] += (int64_t)d[g];
        out[4] |= h[H_ERR];
        if (h[H_MAXALLOC] > out[5]) out[5] = h[H_MAXALLOC];
        if (h[H_ERR] && out[6] < 0) out[6] = (int64_t)g;
        if (h[H_MAXDEPTH] > out[7]) out[7] = h[H_MAXDEPTH];
        out[8] += (int64_t)cc[g];
    }
    return CZ_OK;
}

int cz_engine_root_keys(cz_engine *e, void *stream, uint64_t *keys) {
    if (!e || !keys) return fail(CZ_EINVAL, "cz_engine_root_keys: null");
    int rc = fetch_headers(e, stream);
    if (rc) return rc;
    for (int g = 0; g < e->d.B; g++) keys[g] = (uint64_t)e->h_hdr[(size_t)g * HW + H_HASHLO] | ((uint64_t)e->h_hdr[(size_t)g * HW + H_HASHHI] << 32);
    return CZ_OK;
}

int cz_engine_tree_signature(cz_engine *e, void *stream, int game, int64_t *out, int64_t cap, int64_t *n) {
    if (!e || !n || game < 0 || game >= e->d.B) return fail(CZ_EINVAL, "cz_engine_tree_signature: bad arguments");
    int rc = fetch_headers(e, stream);
    if (rc) return rc;
    const uint32_t *h = e->h_hdr + (size_t)game * HW;
    const int cur = (h[H_FLAGS] & F_CUR) ? 1 : 0;
    const uint32_t alloc = h[H_ALLOC], rbase = h[H_ROOTBASE];
    const int32_t rcnt = (int32_t)h[H_ROOTCNT];
    std::vector<uint32_t> ar(alloc);
    if (alloc) CUDA_TRY(cudaMemcpy(ar.data(), e->d.arena + ((size_t)game * 2 + cur) * (size_t)e->d.A, (size_t)alloc * 4, cudaMemcpyDeviceToHost));
    int64_t k = 0;
    struct Fr { uint32_t base; int cnt; int i; };
    std::vector<Fr> stack;
    if (rcnt > 0) stack.push_back({rbase, rcnt, 0});
    const Labels &L = labels();
    while (!stack.empty()) {
        Fr &f = stack.back();
        if (f.i >= f.cnt) { stack.pop_back(); continue; }
        const uint32_t cs = (uint32_t)((f.cnt + 7) & ~7);
        const uint32_t *blk = ar.data() + f.base + HDR;
        const int i = f.i++;
        const uint32_t meta = blk[3 * cs + i], child = blk[4 * cs + i];
        const int N = (int)blk[2 * cs + i];
        float W, Q;
        memcpy(&W, &blk[cs + i], 4);
        Q = N > 0 ? W / (float)N : 0.0f;
        if (e->d.narr == 6) memcpy(&Q, &blk[5 * cs + i], 4);     // FIFO mode: the stored Q of the last back_up_value
        uint32_t qb;
        memcpy(&qb, &Q, 4);
        const int nch = child != NONE ? (int)((meta >> 16) & 0xFFu) : 0;
        if (k < cap && out) {
            int64_t *r = out + 6 * k;
            r[0] = L.of[(meta & 127) * CZ_NSQ + ((meta >> 7) & 127)];
            float P;
            memcpy(&P, &blk[i], 4);
            r[1] = N;
            r[2] = W != W ? 0x7FC00000u : blk[cs + i];   // NaN payloads are not part of parity
            r[3] = P != P ? 0x7FC00000u : blk[i];
            r[4] = Q != Q ? 0x7FC00000u : qb;
            r[5] = nch;
        }
        k++;
        if (nch > 0) stack.push_back({child, nch, 0});
    }
    *n = k;
    return CZ_OK;
}

}  // extern "C"
