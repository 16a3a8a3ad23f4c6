// mortal_b200 — CUDA kernels (sm_100a) and the C ABI of include/mjx.h.
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/mjx.h"
#include "mjx_sp.cuh"
#include "mjx_policy.cuh"
#include "mjx_replay.cuh"
#include "mjx_invisible.cuh"
#include "mjx_state.cuh"
#include "mjx_nn.cuh"
#include "mjx_select.cuh"
#include "mjx_tables_host.h"

using namespace mjx;

// ================================================================ kernels
constexpr int STEP_WARPS = 4;  // tables per CTA

// One warp = one table: record HBM -> smem (uint4, coalesced), step, smem -> HBM.
__global__ void __launch_bounds__(STEP_WARPS * 32) k_step(EnvView V, Tables T) {
    __shared__ __align__(16) unsigned char s_tab[STEP_WARPS][sizeof(TableState)];
    __shared__ WarpScratch s_scratch[STEP_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int table = blockIdx.x * STEP_WARPS + warp;
    if (table >= V.n_tables) return;
    TableState* g = V.tables + table;
    // cheap liveness probe before moving 2 KB
    if (!(g->gflags & GF_ALIVE)) return;
    constexpr int NV = sizeof(TableState) / 16;
    uint4* dst = reinterpret_cast<uint4*>(s_tab[warp]);
    const uint4* src = reinterpret_cast<const uint4*>(g);
    for (int i = lane; i < NV; i += 32) dst[i] = src[i];
    __syncwarp();
    Ctx c;
    c.S = reinterpret_cast<TableState*>(s_tab[warp]);
    c.W = &s_scratch[warp];
    c.T = T;
    c.lane = lane;
    c.df = s_scratch[warp].dora_factor;
    if (V.log) { c.log = V.log + (size_t)table * V.log_cap; c.log_n = V.log_len + table; c.log_cap = V.log_cap; }
    if (V.grp) { c.grp = V.grp + (size_t)table * V.grp_cap * 7; c.grp_n = V.grp_len + table; c.grp_cap = V.grp_cap; }
    const i32 err_before = c.S->err;
    const bool live = step_table(c, V, table);
    __syncwarp();
    uint4* gdst = reinterpret_cast<uint4*>(g);
    for (int i = lane; i < NV; i += 32) gdst[i] = dst[i];
    if (lane == 0 && live) {
        atomicAdd(&V.counters[0], 1ull);
        atomicAdd(&V.counters[1], 1ull);
    }
    if (lane == 0 && err_before == 0 && c.S->err != 0) atomicAdd(&V.counters[2], 1ull);  // tables that failed so far (mjx_env_poll)
}

// Log replay (csrc/mjx_replay.cuh): one warp = one (game log, player) job, advanced to its next logged decision.
__global__ void __launch_bounds__(STEP_WARPS * 32) k_replay_step(EnvView V, ReplayView R, Tables T) {
    __shared__ __align__(16) unsigned char s_tab[STEP_WARPS][sizeof(TableState)];
    __shared__ WarpScratch s_scratch[STEP_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int job = blockIdx.x * STEP_WARPS + warp;
    if (job >= V.n_tables) return;
    TableState* g = V.tables + job;
    if (!(g->gflags & GF_ALIVE)) return;
    constexpr int NV = sizeof(TableState) / 16;
    uint4* dst = reinterpret_cast<uint4*>(s_tab[warp]);
    const uint4* src = reinterpret_cast<const uint4*>(g);
    for (int i = lane; i < NV; i += 32) dst[i] = src[i];
    __syncwarp();
    Ctx c;
    c.S = reinterpret_cast<TableState*>(s_tab[warp]);
    c.W = &s_scratch[warp];
    c.T = T;
    c.lane = lane;
    c.df = s_scratch[warp].dora_factor;
    const bool live = replay_table(c, V, R, job);
    __syncwarp();
    uint4* gdst = reinterpret_cast<uint4*>(g);
    for (int i = lane; i < NV; i += 32) gdst[i] = dst[i];
    if (lane == 0 && live) atomicAdd(&V.counters[0], 1ull);
}

__global__ void k_begin_step(EnvView V) {
    *V.n_rows = 0;
    V.counters[0] = 0;
}

__global__ void k_init_tables(TableState* tabs, int n, const u64* nonces, const u64* keys, int shuffle_kind, i32* done,
                              i32* steps, i32* err) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    TableState* S = tabs + t;
    unsigned char* p = reinterpret_cast<unsigned char*>(S);
    for (size_t i = 0; i < sizeof(TableState); i++) p[i] = 0;
    S->nonce = nonces[t];
    S->key = keys[t];
    for (int i = 0; i < 4; i++) {
        S->scores[i] = 25000;  // game.rs:225
        S->row_of_seat[i] = -1;
        S->kan_row_of_seat[i] = -1;
        S->auto_action[i] = -1;
    }
    S->shuffle_kind = (u8)shuffle_kind;
    S->gflags = GF_ALIVE;
    done[t] = 0;
    steps[t] = 0;
    err[t] = 0;
}

// Observation encoder, stage 1: one warp = one feature group (ENC_N_PARTS row ranges) of one decision row. Stage the
// table record, derive that part of the compact form (row masks + value rows, csrc/mjx_obs.cuh) in shared memory,
// copy it out coalesced (10,944 B per row for v4). Items are ordered part-major: neighbouring warps run the same code.
// largest per-part window of the compact form (mask rows * 8 + value rows * 136 bytes): what one warp stages
constexpr int enc_max_window_bytes(int ver) {
    const ObsLayout L = make_layout(ver);
    int best = 0;
    for (int q = 0; q < ENC_N_PARTS; q++) {
        const int b = (L.part_row[q + 1] - L.part_row[q]) * 8 + (L.part_sv[q + 1] - L.part_sv[q]) * OBS_COLS * 4;
        if (b > best) best = b;
    }
    return best;
}
template <int VER> struct EncF {
    static constexpr int COMPACT = enc_compact_bytes(VER);
    static constexpr int WINDOW_PAD = (enc_max_window_bytes(VER) + 15) & ~15;          // the staged record wants 16-byte alignment
    static constexpr int WARP_BYTES = WINDOW_PAD + (int)sizeof(TableState) + 48;        // + record + dora factors
    static constexpr int WARPS = 232448 / WARP_BYTES >= 20 ? 20 : 232448 / WARP_BYTES;  // one CTA per SM, register-limited
    static constexpr size_t SMEM = (size_t)WARPS * WARP_BYTES;
    static_assert(COMPACT % 8 == 0 && WARP_BYTES % 16 == 0, "vector copies");
};

template <int VER>
__global__ void __launch_bounds__(EncF<VER>::WARPS * 32, 1) k_encode_features(EnvView V, Tables T, unsigned char* __restrict__ compact, int* __restrict__ work) {
    constexpr ObsLayout L = make_layout(VER);
    constexpr int COMPACT = EncF<VER>::COMPACT, WARPS = EncF<VER>::WARPS;
    extern __shared__ __align__(128) unsigned char s_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char* base = s_raw + (size_t)warp * EncF<VER>::WARP_BYTES;
    u64* win = reinterpret_cast<u64*>(base);  // this part's window: its mask rows, then its value rows
    TableState* s_state = reinterpret_cast<TableState*>(base + EncF<VER>::WINDOW_PAD);
    u8* df = base + EncF<VER>::WINDOW_PAD + sizeof(TableState);
    const int n_rows = *V.n_rows;
    const int n_items = n_rows * ENC_N_PARTS;
    // Items are handed out dynamically, longest first: the action block (part 3: discard candidates, unconditional-tenpai
    // scan, L2 table gathers) of every row, then the ponds, the counters/overview group and the cheap hand/scalar group,
    // so that the expensive rows do not form the tail. `work` is reset by k_encode_store, which always runs next.
    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(work, 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n_items) break;
        const int ord = item / n_rows, row = item - ord * n_rows;
        const int part = ord == 0 ? 3 : ord == 1 ? 1 : ord == 2 ? 2 : 0;
        // this part's window of the compact form, in 8-byte words (mask rows, then the value rows as 17 words each)
        int bm_lo = 0, bm_hi = 0, slot_lo = 0, slot_hi = 0;
#pragma unroll
        for (int q = 0; q < ENC_N_PARTS; q++)
            if (q == part) { bm_lo = L.part_row[q]; bm_hi = L.part_row[q + 1]; slot_lo = L.part_sv[q]; slot_hi = L.part_sv[q + 1]; }
        const int n_bm = bm_hi - bm_lo, n_win = n_bm + (slot_hi - slot_lo) * 17;  // window size in 8-byte words
        // biased pointers: bm[row] / sv[slot * 34 + col] address the window for the rows / slots of this part
        u64* bm = win - bm_lo;
        float* sv = reinterpret_cast<float*>(win + n_bm) - slot_lo * OBS_COLS;
        {
            const uint4* src = reinterpret_cast<const uint4*>(V.tables + V.row_table[row]);
            uint4* dst = reinterpret_cast<uint4*>(s_state);
            for (int i = lane; i < (int)(sizeof(TableState) / 16); i += 32) dst[i] = __ldg(src + i);
            for (int i = lane; i < n_win; i += 32) win[i] = 0;
        }
        __syncwarp();
        const TableState* S = s_state;
        {   // dora factors: lane k resolves indicator k once, every lane counts its own tile kinds
            const int nd = S->n_dora;
            const int d = lane < nd ? tile_next(S->wall[60 - lane]) : -1;
            int f0 = 0, f1 = 0;
            for (int k = 0; k < nd; k++) {
                const int dk = __shfl_sync(0xffffffffu, d, k);
                f0 += dk == lane;
                f1 += dk == lane + 32;
            }
            df[lane] = (u8)f0;
            if (lane < 2) df[32 + lane] = (u8)f1;
        }
        __syncwarp();
        const u8 rs = V.row_seat[row];
        EncCtx e;
        e.S = S; e.T = T; e.bm = bm; e.sv = sv; e.seat = rs & 3; e.kan_select = (rs >> 2) & 1;
        e.lane = lane; e.dora_factor = df; e.parts = 1u << part;
        Ctx c;
        c.S = s_state; c.W = nullptr; c.T = T; c.lane = lane; c.df = df;
        encode_obs<VER>(e, c, nullptr);
        __syncwarp();
        u64* out = reinterpret_cast<u64*>(compact + (size_t)row * COMPACT);
        for (int i = lane; i < n_bm; i += 32) out[bm_lo + i] = win[i];
        for (int i = n_bm + lane; i < n_win; i += 32) out[L.bm_rows + slot_lo * 17 + (i - n_bm)] = win[i];
        __syncwarp();
    }
}

// Stage 2, the HBM-bound one: one warp = one slice of one observation at a time. Clear a shared-memory tile, light
// the non-zero rows from the compact form, hand the tile to the copy engine as one bulk async store (TMA). Two tiles
// per warp: the next slice is built while the copy engine still reads the previous one.
constexpr int ENCS_WARPS = 16;
constexpr int ENC_SLICE_BYTES = OBS_SLICE_ROWS * OBS_COLS * (int)sizeof(float);  // 6,256
constexpr size_t ENCS_SMEM_BYTES = (size_t)ENCS_WARPS * 2 * ENC_SLICE_BYTES;     // 200,192
static_assert(ENC_SLICE_BYTES % 16 == 0, "bulk copies need 16-byte alignment");
static_assert(ENCS_SMEM_BYTES <= 232448, "one CTA per SM");

struct EncStoreArgs { int rows, bm_rows, n_sv, compact_bytes, n_slices, ver; };
__constant__ short c_sv_row[4][OBS_MAX_SV];  // ObsLayout::sv_row of versions 1..4

__global__ void __launch_bounds__(ENCS_WARPS * 32, 1) k_encode_store(EnvView V, EncStoreArgs A, const unsigned char* __restrict__ compact,
                                                                     float* __restrict__ obs, int* __restrict__ work) {
    extern __shared__ __align__(128) unsigned char s_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (blockIdx.x == 0 && threadIdx.x == 0) *work = 0;  // re-arm k_encode_features' work counter for the next step
    unsigned char* base = s_raw + (size_t)warp * 2 * ENC_SLICE_BYTES;
    const int n_items = *V.n_rows * A.n_slices;
    const int stride = gridDim.x * ENCS_WARPS;
    const short* sv_row = c_sv_row[A.ver - 1];
    // the 0.5 GB of observations stream through L2 as evict-first so that they do not push out the compact form
    // this kernel is reading (44 MB, written by k_encode_features just before)
    unsigned long long evict_first;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(evict_first));
    int item = blockIdx.x * ENCS_WARPS + warp;
    u64 m0 = 0, m1 = 0;
    if (item < n_items) {
        const int row = item / A.n_slices;
        enc_load_masks(reinterpret_cast<const u64*>(compact + (size_t)row * A.compact_bytes), A.bm_rows,
                       (item - row * A.n_slices) * OBS_SLICE_ROWS, lane, m0, m1);
    }
    for (int buf = 0; item < n_items; item += stride, buf ^= 1) {
        const int row = item / A.n_slices, slice = item - row * A.n_slices;
        const int row_lo = slice * OBS_SLICE_ROWS, row_hi = min(row_lo + OBS_SLICE_ROWS, A.rows);
        // the next item's row masks are requested now and consumed one iteration later
        u64 n0 = 0, n1 = 0;
        if (item + stride < n_items) {
            const int nrow = (item + stride) / A.n_slices;
            enc_load_masks(reinterpret_cast<const u64*>(compact + (size_t)nrow * A.compact_bytes), A.bm_rows,
                           (item + stride - nrow * A.n_slices) * OBS_SLICE_ROWS, lane, n0, n1);
        }
        float* tile = reinterpret_cast<float*>(base + buf * ENC_SLICE_BYTES);
        // the store that last used this tile (two items ago) must have finished reading it
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncwarp();
        const unsigned char* cf = compact + (size_t)row * A.compact_bytes;
        enc_materialize(reinterpret_cast<const float*>(cf + A.bm_rows * 8), sv_row, A.n_sv, lane, tile, row_lo, row_hi, m0, m1);
        // make the generic-proxy smem writes visible to the async proxy, then one lane issues the bulk store
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
            float* dst = obs + ((size_t)row * A.rows + row_lo) * OBS_COLS;
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                         :: "l"(dst), "r"((unsigned)__cvta_generic_to_shared(tile)),
                            "r"((unsigned)((row_hi - row_lo) * OBS_COLS * (int)sizeof(float))), "l"(evict_first)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        m0 = n0; m1 = n1;
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    __syncwarp();
}

// invisible (oracle) observation of every row of the step: one warp per row (csrc/mjx_invisible.cuh)
__global__ void __launch_bounds__(128) k_encode_invisible(EnvView V, int version, float* __restrict__ out, int all_yama) {
    const int lane = threadIdx.x & 31, gwarp = blockIdx.x * 4 + (threadIdx.x >> 5), nwarps = gridDim.x * 4;
    const int n_rows = *V.n_rows, rows = oracle_obs_rows(version);
    for (int row = gwarp; row < n_rows; row += nwarps)
        encode_invisible(V.tables + V.row_table[row], V.row_seat[row] & 3, version, out + (size_t)row * rows * OBS_COLS, lane, all_yama != 0);
}

__global__ void k_set_seeds(TableState* tabs, int n, const u64* nonces, const u64* keys, int shuffle_kind) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) { tabs[t].nonce = nonces[t]; tabs[t].key = keys[t]; tabs[t].shuffle_kind = (u8)shuffle_kind; }
}

// ---- libriichi.state.PlayerState batch (csrc/mjx_state.cuh): one warp = one state, record staged in shared memory
#define STATE_KERNEL_PROLOGUE                                                                                     \
    __shared__ __align__(16) unsigned char s_tab[STEP_WARPS][sizeof(TableState)];                                \
    __shared__ WarpScratch s_scratch[STEP_WARPS];                                                                 \
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;                                                   \
    const int i = blockIdx.x * STEP_WARPS + warp;                                                                 \
    if (i >= V.n_tables) return;                                                                                  \
    TableState* g = V.tables + i;                                                                                 \
    constexpr int NV = sizeof(TableState) / 16;                                                                   \
    uint4* dst = reinterpret_cast<uint4*>(s_tab[warp]);                                                           \
    for (int q = lane; q < NV; q += 32) dst[q] = reinterpret_cast<const uint4*>(g)[q];                            \
    __syncwarp();                                                                                                 \
    Ctx c; c.S = reinterpret_cast<TableState*>(s_tab[warp]); c.W = &s_scratch[warp]; c.T = T; c.lane = lane;     \
    c.df = s_scratch[warp].dora_factor;                                                                           \
    recompute_dora_factor(c);

__global__ void k_state_init(TableState* tabs, int n, const u8* player_ids) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) { tabs[t].viewer1 = (u8)(player_ids[t] + 1); tabs[t].gflags = GF_ALIVE; tabs[t].last_kawa_tile = T_NONE;
                 for (int s = 0; s < 4; s++) tabs[t].priv[s].last_self_tsumo = T_NONE; }
}

__global__ void __launch_bounds__(STEP_WARPS * 32) k_state_update(EnvView V, Tables T, const u64* __restrict__ words,
                                                                    const u64* __restrict__ payload, u32* __restrict__ cans) {
    STATE_KERNEL_PROLOGUE
    const u64 w = words[i];
    const int p = c.S->viewer1 - 1;
    if (w != 0) {
        apply_event(c, w, payload ? payload + (size_t)i * REPLAY_KYOKU_WORDS : nullptr, false);
        __syncwarp();
        for (int q = lane; q < NV; q += 32) reinterpret_cast<uint4*>(g)[q] = dst[q];
    }
    if (lane == 0) cans[i] = (u32)c.S->priv[p].cans | ((u32)c.S->priv[p].target_actor << 16);
}

__global__ void __launch_bounds__(STEP_WARPS * 32) k_state_view(EnvView V, Tables T, int index, mjx_player_view* out) {
    STATE_KERNEL_PROLOGUE
    if (i != index) return;
    if (lane == 0) state_view(c, c.S->viewer1 - 1, out);
}

// one decision row per state: row i = state i (obs_repr.rs:776-790 encode_obs(version, at_kan_select))
__global__ void __launch_bounds__(STEP_WARPS * 32) k_state_rows(EnvView V, Tables T, const u8* __restrict__ at_kan_select) {
    STATE_KERNEL_PROLOGUE
    const int p = c.S->viewer1 - 1;
    const bool kan = at_kan_select && at_kan_select[i];
    const u16 cans_bits = c.S->priv[p].cans;
    const u64 discards = (cans_bits & CAN_DISCARD) ? discard_candidates(c, p) : 0;
    write_mask_row(c, V, i, legal_mask(c, p, kan, discards));
    if (lane == 0) { V.row_table[i] = i; V.row_seat[i] = (u8)(p | (kan ? 4 : 0)); V.row_step[i] = 0; if (i == 0) *V.n_rows = V.n_tables; }
}

__global__ void __launch_bounds__(STEP_WARPS * 32) k_state_query(EnvView V, Tables T, int index, int what, const i32* __restrict__ args,
                                                                   i32* __restrict__ out) {
    STATE_KERNEL_PROLOGUE
    if (i != index) return;
    const int p = c.S->viewer1 - 1;
    if (what == 0) {
        u8 ura[5];
        const int n_ura = min(max(args[1], 0), 5);
        for (int k = 0; k < n_ura; k++) ura[k] = (u8)args[2 + k];
        bool ok;
        const Point pt = agari_points_ura(c, p, args[0] != 0, ura, n_ura, &ok);
        if (lane == 0) { out[0] = pt.ron; out[1] = pt.tsumo_ko; out[2] = pt.tsumo_oya; out[3] = ok ? 1 : 0; }
    } else if (what == 1) {
        const bool r = rule_based_agari(c, p);
        if (lane == 0) out[0] = r ? 1 : 0;
    } else if (what == 2) {
        const u64 m = discard_candidates(c, p);
        if (lane == 0) { out[0] = (i32)(u32)m; out[1] = (i32)(u32)(m >> 32); }
    } else if (what == 3) {
        EncCtx e; e.S = c.S; e.T = T; e.bm = nullptr; e.sv = nullptr; e.seat = p; e.kan_select = false; e.lane = lane;
        e.dora_factor = c.df; e.parts = 0;
        const u64 m = unconditional_tenpai_discards(e, c);
        if (lane == 0) { out[0] = (i32)(u32)m; out[1] = (i32)(u32)(m >> 32); }
    } else if (what == 4) {
        Reaction r;
        i32 err = 0;
        const bool okd = decode_action(c.S, p, args[0], args[1], r, &err);
        if (lane == 0) {
            u64 w = 0;
            if (okd) {
                const int ty = r.type == R_DAHAI ? LOG_DAHAI : r.type == R_CHI ? LOG_CHI : r.type == R_PON ? LOG_PON :
                               r.type == R_DAIMINKAN ? LOG_DAIMINKAN : r.type == R_KAKAN ? LOG_KAKAN : r.type == R_ANKAN ? LOG_ANKAN :
                               r.type == R_REACH ? LOG_REACH : r.type == R_HORA ? LOG_HORA : r.type == R_RYUKYOKU ? LOG_RYUKYOKU : 0;
                w = log_word(ty, r.actor, r.target, r.pai, r.tsumogiri, 0, r.consumed[0], r.consumed[1], r.consumed[2], r.consumed[3], 0);
            }
            out[0] = (i32)(u32)w; out[1] = (i32)(u32)(w >> 32); out[2] = okd ? 0 : (err ? err : ERR_ILLEGAL_ACTION);
        }
    }
}

// ---- single-player tables: level-synchronous DP over all rows of the step (csrc/mjx_sp.cuh)
constexpr int SP_WARPS = 4;
constexpr int MJX_HOST_COPY_GROUPS = 4;
constexpr int MJX_SP_MAX_LANES = 4;  // mjx_env_encode_obs_host: row groups of the SP block / D2H pipeline

__global__ void k_sp_begin(SpGlobal G) {
    if (threadIdx.x < SP_SLOTS) G.wl_count[threadIdx.x] = 0;
    if (threadIdx.x == 0) {
        if (G.counters[2]) G.counters[3] += 1;  // an overflow happened in the previous block
        G.counters[0] = 0; G.counters[1] = 0; G.counters[2] = 0; G.counters[4] = 0; G.counters[5] = 0;
    }
}

// one warp per observation row (init / finalize)
#define SP_ROW_PROLOGUE                                                                         \
    __shared__ u8 s_df[SP_WARPS][40];                                                           \
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;                                 \
    const int gwarp = blockIdx.x * SP_WARPS + warp, nwarps = gridDim.x * SP_WARPS;              \
    SpCtx s; s.G = G; s.T = T; s.df = s_df[warp]; s.lane = lane;

// rows [row_lo, min(n_rows, row_hi)) of the step, of which this launch takes the `part`-th of `parts` equal shares (the step's row
// count only exists on the device, so concurrent DP lanes name their share as a fraction)
#define SP_ROW_RANGE                                                                            \
    const int span_ = max(min(*V.n_rows, row_hi) - row_lo, 0);                                  \
    const int r0 = row_lo + (int)((long long)span_ * part / parts), r1 = row_lo + (int)((long long)span_ * (part + 1) / parts);

__global__ void __launch_bounds__(SP_WARPS * 32) k_sp_init(SpGlobal G, Tables T, EnvView V, int row_lo, int row_hi, int part, int parts) {
    SP_ROW_PROLOGUE
    SP_ROW_RANGE
    for (int row = r0 + gwarp; row < r1; row += nwarps)
        sp_stage_init(s, V.tables + V.row_table[row], row, V.row_table[row], V.row_seat[row] & 3);
}

// KIND 0: D level, 1: W level, 2: the tenpai W level (csrc/mjx_sp.cuh sp_expand_batch): one CTA = batches of 32 states
template <int KIND>
__global__ void __launch_bounds__(SP_THREADS) k_sp_expand(SpGlobal G, Tables T, int level) {
    __shared__ SpExpandBatch sb;
    SpBlk B; B.tid = threadIdx.x; B.nthr = blockDim.x; B.bid = blockIdx.x; B.nblk = gridDim.x;
    sp_expand_level<KIND>(G, T, sb, B, level);
}

// KIND 0: D level (per-turn best discard), 1: W level above tenpai, 2: the tenpai W level (scores of the winning draws)
template <int KIND>
__global__ void __launch_bounds__(SP_THREADS) k_sp_eval(SpGlobal G, int level) {
    SpBlk B; B.tid = threadIdx.x; B.nthr = blockDim.x; B.bid = blockIdx.x; B.nblk = gridDim.x;
    if (KIND == 0) {
        __shared__ SpEvalDBatch sd;
        sp_eval_d_level(G, sd, B, level);
    } else {
        __shared__ SpEvalWBatch sw[SP_THREADS / 32];
        sp_eval_w_level<KIND == 2>(G, sw, B, level);
    }
}

// the probability table of the W evaluation (csrc/mjx_sp.cuh), built once per process with the reference's operation sequence
__global__ void k_sp_tables(float* p_tab) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < SP_NTS_DIM * SP_NTS_DIM) sp_fill_ptab_block(p_tab + (size_t)i * 4 * SP_TRI, i / SP_NTS_DIM, i % SP_NTS_DIM);
}

__global__ void k_sp_mark(SpGlobal G, int which) { G.counters[4 + which] = min(G.counters[1], G.edge_cap); }

__global__ void __launch_bounds__(256) k_sp_densify(SpGlobal G) {
    SpBlk B; B.tid = threadIdx.x; B.nthr = blockDim.x; B.bid = blockIdx.x; B.nblk = gridDim.x;
    sp_densify(G, B);
}

__global__ void __launch_bounds__(128) k_sp_score(SpGlobal G, Tables T) {
    const int b = G.counters[4], e_end = G.counters[5];
    for (int e = b + blockIdx.x * blockDim.x + threadIdx.x; e < e_end; e += gridDim.x * blockDim.x) sp_score_edge(G, T, e);
}

__global__ void __launch_bounds__(SP_WARPS * 32) k_sp_finalize(SpGlobal G, Tables T, EnvView V, float* __restrict__ obs, int row_lo,
                                                               int row_hi, int part, int parts) {
    SP_ROW_PROLOGUE
    SP_ROW_RANGE
    for (int row = r0 + gwarp; row < r1; row += nwarps)
        sp_stage_finalize(s, row, obs + (size_t)row * OBS_ROWS_V4 * OBS_COLS);
}

__global__ void __launch_bounds__(256) k_sp_release(SpGlobal G) {
    SpBlk B; B.tid = threadIdx.x; B.nthr = blockDim.x; B.bid = blockIdx.x; B.nblk = gridDim.x;
    sp_release(G, B);
}

__global__ void k_policy_test(EnvView V, int kind, i64* actions, i64* trace, float* q_out) {
    const int n_rows = *V.n_rows;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += gridDim.x * blockDim.x) {
        const int t = V.row_table[r], seat = V.row_seat[r] & 3, kan = (V.row_seat[r] >> 2) & 1;
        u64 m = 0;
        for (int i = 0; i < ACTION_SPACE; i++) if (V.masks[(size_t)r * ACTION_SPACE + i]) m |= 1ull << i;
        const TableState* S = V.tables + t;
        const SeatPrivate& P = S->priv[seat];
        u64 h = policy_hash(S->nonce, S->key, (u64)t, V.row_step[r], (u32)seat, (u32)kan);
        int a = test_policy(kind, h, kan != 0, m, P.keep_shanten, P.next_shanten);
        actions[r] = a;
        if (q_out)  // what a masked dueling head would give a uniform policy: 0 on legal actions, -inf elsewhere
            for (int i = 0; i < ACTION_SPACE; i++) q_out[(size_t)r * ACTION_SPACE + i] = ((m >> i) & 1) ? 0.f : -INFINITY;
        if (trace) {
            i64* o = trace + (size_t)r * 6;
            o[0] = t; o[1] = V.row_step[r]; o[2] = seat; o[3] = a; o[4] = kan; o[5] = (i64)m;
        }
    }
}

// ---- standalone: shanten (hands staged through smem so the 34-byte records load coalesced)
constexpr int SH_THREADS = 256;
__global__ void __launch_bounds__(SH_THREADS) k_shanten(Tables T, const u8* __restrict__ tiles, const u8* __restrict__ len_div3,
                                                         i8* __restrict__ out, int n) {
    __shared__ __align__(16) u8 s_tiles[SH_THREADS * 34];
    const int base = blockIdx.x * SH_THREADS;
    const int cnt = min(SH_THREADS, n - base);
    if (cnt <= 0) return;
    const size_t byte0 = (size_t)base * 34;
    const int nbytes = cnt * 34;
    // 34-byte records: block start is 34*256-byte aligned -> 16-byte aligned when base is a multiple of 8
    for (int i = threadIdx.x; i < nbytes; i += SH_THREADS) s_tiles[i] = tiles[byte0 + i];
    __syncthreads();
    if (threadIdx.x < cnt) {
        const u8* h = s_tiles + threadIdx.x * 34;
        u8 loc[34];
#pragma unroll
        for (int i = 0; i < 34; i++) loc[i] = h[i];
        out[base + threadIdx.x] = (i8)shanten_all(T, loc, len_div3[base + threadIdx.x]);
    }
}

__global__ void __launch_bounds__(128) k_agari(Tables T, const mjx_agari_in* __restrict__ in, mjx_agari_out* __restrict__ out,
                                                int n, int mode) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    mjx_agari_in q = in[i];
    AgariQuery a;
    a.tehai = q.tehai;
    a.chis = q.chis; a.pons = q.pons; a.minkans = q.minkans; a.ankans = q.ankans;
    a.n_chis = q.n_chis; a.n_pons = q.n_pons; a.n_minkans = q.n_minkans; a.n_ankans = q.n_ankans;
    a.bakaze = q.bakaze; a.jikaze = q.jikaze; a.winning_tile = q.winning_tile;
    a.is_ron = q.is_ron != 0;
    a.is_menzen = q.n_chis == 0 && q.n_pons == 0 && q.n_minkans == 0;
    mjx_agari_out o;
    o.kind = 0; o.fu = o.han = o.yakuman = 0; o.ron = o.tsumo_ko = o.tsumo_oya = 0;
    if (mode == 2) {
        o.kind = has_yaku(T, a) ? 1 : 0;
    } else if (mode == 3) {  // agari.rs:854-912 check_ankan_after_riichi, strict = false (what update.rs:278 asks)
        o.kind = ankan_after_riichi_ok(T, q.tehai, q.additional_hans, q.winning_tile) ? 1 : 0;
    } else {
        Agari r = mode == 0 ? search_yakus(T, a, false) : agari_with(T, a, q.additional_hans, q.doras);
        if (r.kind != 0) {
            o.kind = r.kind; o.fu = r.fu; o.han = r.han; o.yakuman = r.yakuman;
            bool ok;
            Point p = agari_point(r, q.is_oya != 0, &ok);
            if (ok) { o.ron = p.ron; o.tsumo_ko = p.tsumo_ko; o.tsumo_oya = p.tsumo_oya; }
            else { o.ron = o.tsumo_ko = o.tsumo_oya = -1; }
        }
    }
    out[i] = o;
}

__global__ void k_make_wall(u64 nonce, u64 key, int kyoku, int honba, int kind, u8* out) {
    __shared__ u8 w[136];
    if (threadIdx.x == 0) make_wall(nonce, key, kyoku, honba, kind, w);
    __syncthreads();
    for (int i = threadIdx.x; i < 136; i += blockDim.x) out[i] = w[i];
}

// ================================================================ host side
namespace {

thread_local std::string g_err;
std::mutex g_mu;
bool g_ready = false;
int g_device = -1;
int g_sm_count = 148;
Tables g_T;
const float* g_sp_p_tab = nullptr;  // csrc/mjx_sp.cuh draw-probability table (device)

int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CU(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess)                                                            \
            return fail(MJX_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

template <typename Tp>
int upload(const std::vector<Tp>& v, const Tp** out) {
    Tp* d = nullptr;
    CU(cudaMalloc(&d, v.size() * sizeof(Tp)));
    CU(cudaMemcpy(d, v.data(), v.size() * sizeof(Tp), cudaMemcpyHostToDevice));
    *out = d;
    return 0;
}

}  // namespace

struct mjx_env {
    int n_tables = 0, row_cap = 0, obs_version = 4, shuffle_kind = 0, quick_eval = 1;
    bool first = true;
    EnvView V;
    u64 *d_nonces = nullptr, *d_keys = nullptr;
    i64* d_dummy_actions = nullptr;
    u8* d_guard = nullptr;
    u8* d_quick_eval = nullptr;
    SpGlobal sp;
    int sp_enabled = 1, sp_wanted = 1;
    // concurrent DP lanes of the single-player block (mjx_env_encode_obs): every lane runs on a side stream of its own while the
    // caller's stream runs the two encoder kernels; lane 0 = `sp`, lanes 1.. own a smaller state table each, allocated on first use
    SpGlobal sp_lane[MJX_SP_MAX_LANES - 1];
    int sp_lanes = 1, sp_lanes_alloc = 1;
    int sp_grid_x = 10, sp_grid_e = 16;  // CTAs per SM of the expansion / evaluation launches
    int sp_thr_x = SP_THREADS, sp_thr_e = SP_THREADS;
    long long sp_want_slots = 0;
    cudaStream_t sp_stream[MJX_SP_MAX_LANES] = {};
    cudaEvent_t ev_sp_fork = nullptr, ev_sp_store = nullptr, ev_sp_join[MJX_SP_MAX_LANES] = {};
    unsigned char* d_compact = nullptr;
    cudaEvent_t ev_enc[3] = {nullptr, nullptr, nullptr};  // optional per-kernel timing of the encoder pair (bench.py roofline)
    bool time_encode = false;
    ReplayView R{};  // replay mode (mjx_env_create_replay): device arrays of the jobs
    bool replay = false;
    int* d_enc_work = nullptr;  // k_encode_features' dynamic work counter
    EncStoreArgs enc_args{};
    cudaStream_t copy_stream = nullptr;  // mjx_env_encode_obs_host: D2H overlapped with the SP kernels
    cudaEvent_t ev_rows = nullptr, ev_sp = nullptr, ev_grp[MJX_HOST_COPY_GROUPS] = {};
    long long launches = 0;  // kernels launched on behalf of this env (bench.py's gpu_launches)
    bool is_state = false;   // mjx_state_create: a batch of single-seat PlayerStates
    u64 *d_state_words = nullptr, *d_state_pay = nullptr;
    u32* d_state_cans = nullptr;
    unsigned char* d_state_misc = nullptr;
};

static void set_enc_args(mjx_env* env, int version) {
    const ObsLayout L = make_layout(version);
    env->enc_args.rows = L.rows; env->enc_args.bm_rows = L.bm_rows; env->enc_args.n_sv = L.n_sv;
    env->enc_args.compact_bytes = L.bm_rows * 8 + L.n_sv * OBS_COLS * 4;
    env->enc_args.n_slices = (L.rows + OBS_SLICE_ROWS - 1) / OBS_SLICE_ROWS;
    env->enc_args.ver = version;
}

template <int VER>
static void launch_features(mjx_env* env, cudaStream_t st) {
    k_encode_features<VER><<<g_sm_count, EncF<VER>::WARPS * 32, EncF<VER>::SMEM, st>>>(env->V, g_T, env->d_compact, env->d_enc_work);
}

// device buffers of one DP instance (csrc/mjx_sp.cuh SpGlobal) for about `want` live states; `G.rows` is shared by all instances
static int sp_alloc(SpGlobal& G, long long want) {
    int hc = 1 << 20;
    while (hc < want && hc < (1 << 26)) hc <<= 1;
    G.hash_cap = hc;
    G.p_tab = g_sp_p_tab;
    G.wl_cap = hc / 2;       // per level
    G.edge_cap = hc * 2;
    G.score_cap = hc;
    CU(cudaMalloc(&G.hkey, (size_t)G.hash_cap * sizeof(u64)));
    CU(cudaMalloc(&G.nsig, (size_t)G.hash_cap * sizeof(SpSigP)));
    CU(cudaMalloc(&G.einfo, (size_t)G.hash_cap * sizeof(u64)));
    CU(cudaMalloc(&G.vals, (size_t)G.hash_cap * SP_VALS * sizeof(float)));
    CU(cudaMalloc(&G.sid, (size_t)G.hash_cap * sizeof(u32)));
    CU(cudaMalloc(&G.dkey, (size_t)G.hash_cap * sizeof(u64)));
    CU(cudaMalloc(&G.echild, (size_t)G.edge_cap * sizeof(u32)));
    CU(cudaMalloc(&G.evid, (size_t)G.edge_cap * sizeof(u32)));
    CU(cudaMemset(G.evid, 0, (size_t)G.edge_cap * sizeof(u32)));
    CU(cudaMalloc(&G.emeta, (size_t)G.edge_cap * sizeof(u16)));
    CU(cudaMalloc(&G.eowner, (size_t)G.edge_cap * sizeof(u32)));
    CU(cudaMalloc(&G.leaf_scores, (size_t)G.score_cap * 4 * sizeof(float)));
    CU(cudaMalloc(&G.wl, (size_t)SP_SLOTS * G.wl_cap * sizeof(u32)));
    CU(cudaMalloc(&G.wl_count, SP_SLOTS * sizeof(i32)));
    CU(cudaMalloc(&G.counters, 8 * sizeof(i32)));
    CU(cudaMemset(G.counters, 0, 8 * sizeof(i32)));
    CU(cudaMemset(G.wl_count, 0, SP_SLOTS * sizeof(i32)));
    CU(cudaMemset(G.hkey, 0xFF, (size_t)G.hash_cap * sizeof(u64)));  // SP_EMPTY; afterwards k_sp_release frees what a block used
    return MJX_OK;
}
static SpGlobal& sp_of(mjx_env* env, int lane) { return lane == 0 ? env->sp : env->sp_lane[lane - 1]; }
static void sp_free(SpGlobal& G) {
    cudaFree(G.hkey); cudaFree(G.nsig); cudaFree(G.einfo); cudaFree(G.vals); cudaFree(G.sid); cudaFree(G.dkey); cudaFree(G.echild); cudaFree(G.evid); cudaFree(G.emeta);
    cudaFree(G.eowner); cudaFree(G.leaf_scores); cudaFree(G.wl); cudaFree(G.wl_count); cudaFree(G.counters);
}
// lanes 1..n-1 (lane 0 is env->sp): each expects 1/n of the step's states and gets twice that
static int sp_ensure_lanes(mjx_env* env, int lanes) {
    if (!env->ev_sp_fork) {
        CU(cudaEventCreateWithFlags(&env->ev_sp_fork, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&env->ev_sp_store, cudaEventDisableTiming));
    }
    for (int g = 0; g < lanes; g++)
        if (!env->sp_stream[g]) {
            CU(cudaStreamCreateWithFlags(&env->sp_stream[g], cudaStreamNonBlocking));
            CU(cudaEventCreateWithFlags(&env->ev_sp_join[g], cudaEventDisableTiming));
        }
    for (int g = env->sp_lanes_alloc; g < lanes; g++) {
        SpGlobal& G = env->sp_lane[g - 1];
        memset(&G, 0, sizeof G);
        G.rows = env->sp.rows;
        int rc = sp_alloc(G, env->sp_want_slots * 2 / lanes);
        if (rc) return rc;
        env->sp_lanes_alloc = g + 1;
    }
    return MJX_OK;
}

extern "C" {

const char* mjx_last_error(void) { return g_err.c_str(); }

int mjx_init(const char* data_dir, int device) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_ready) {
        if (device != g_device) return fail(MJX_ERR_ARG, "mjx_init: already initialised on another device");
        return MJX_OK;
    }
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0)
        return fail(MJX_ERR_CUDA, "mjx_init: no CUDA device (this library has no CPU path)");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    g_sm_count = prop.multiProcessorCount;
    HostTables H;
    if (!load_host_tables(data_dir, H)) return fail(MJX_ERR_TABLES, "mjx_init: " + H.error);
    int rc;
    if ((rc = upload(H.suhai, &g_T.suhai))) return rc;
    if ((rc = upload(H.jihai, &g_T.jihai))) return rc;
    if ((rc = upload(H.agari_keys, &g_T.agari_keys))) return rc;
    if ((rc = upload(H.agari_divs, &g_T.agari_divs))) return rc;
    if ((rc = upload(H.agari_ndivs, &g_T.agari_ndivs))) return rc;
    CU(cudaFuncSetAttribute(k_encode_features<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EncF<1>::SMEM));
    CU(cudaFuncSetAttribute(k_encode_features<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EncF<2>::SMEM));
    CU(cudaFuncSetAttribute(k_encode_features<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EncF<3>::SMEM));
    CU(cudaFuncSetAttribute(k_encode_features<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)EncF<4>::SMEM));
    {
        short tab[4][OBS_MAX_SV];
        for (int v = 1; v <= 4; v++) {
            const ObsLayout L = make_layout(v);
            for (int i = 0; i < OBS_MAX_SV; i++) tab[v - 1][i] = i < L.n_sv ? L.sv_row[i] : (short)-1;
        }
        CU(cudaMemcpyToSymbol(c_sv_row, tab, sizeof tab));
    }
    CU(cudaFuncSetAttribute(k_encode_store, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ENCS_SMEM_BYTES));
    {
        float* pt = nullptr;
        CU(cudaMalloc(&pt, sizeof(float) * SP_NTS_DIM * SP_NTS_DIM * 4 * SP_TRI));
        k_sp_tables<<<(SP_NTS_DIM * SP_NTS_DIM + 63) / 64, 64>>>(pt);
        CU(cudaGetLastError());
        CU(cudaDeviceSynchronize());
        g_sp_p_tab = pt;
    }
    g_device = device;
    g_ready = true;
    return MJX_OK;
}

int mjx_obs_rows(int version) {
    switch (version) {
        case 1: return 938;
        case 2: return 942;
        case 3: return 934;
        case 4: return 1012;
        default: return MJX_ERR_ARG;
    }
}

}  // extern "C"

// allocate and initialise into a zeroed `env`; on failure the caller destroys the half-built env (nothing leaks)
static int env_create_impl(mjx_env* env, int n_tables, const uint64_t* nonces, const uint64_t* keys, int obs_version,
                           int shuffle_kind, int enable_quick_eval) {
    env->n_tables = n_tables;
    env->row_cap = n_tables * MJX_MAX_ROWS_PER_TABLE;
    env->obs_version = obs_version;
    env->shuffle_kind = shuffle_kind;
    env->quick_eval = enable_quick_eval ? 1 : 0;
    EnvView& V = env->V;
    memset(&V, 0, sizeof V);
    V.n_tables = n_tables;
    V.row_cap = env->row_cap;
    V.enable_quick_eval = env->quick_eval;
    const size_t cap = (size_t)env->row_cap;
    CU(cudaMalloc(&V.tables, sizeof(TableState) * (size_t)n_tables));
    CU(cudaMalloc(&V.n_rows, sizeof(i32)));
    CU(cudaMalloc(&V.row_table, sizeof(i32) * cap));
    CU(cudaMalloc(&V.row_seat, cap));
    CU(cudaMalloc(&V.row_step, sizeof(u32) * cap));
    CU(cudaMalloc(&V.masks, cap * ACTION_SPACE));
    CU(cudaMalloc(&V.scores, sizeof(i32) * 4 * (size_t)n_tables));
    CU(cudaMalloc(&V.ranks, 4 * (size_t)n_tables));
    CU(cudaMalloc(&V.done, sizeof(i32) * (size_t)n_tables));
    CU(cudaMalloc(&V.steps, sizeof(i32) * (size_t)n_tables));
    CU(cudaMalloc(&V.err, sizeof(i32) * (size_t)n_tables));
    CU(cudaMalloc(&V.counters, sizeof(unsigned long long) * 4));
    CU(cudaMalloc(&env->d_nonces, sizeof(u64) * (size_t)n_tables));
    CU(cudaMalloc(&env->d_keys, sizeof(u64) * (size_t)n_tables));
    CU(cudaMalloc(&env->d_dummy_actions, sizeof(i64) * cap));
    memset(&env->sp, 0, sizeof env->sp);
    {
        set_enc_args(env, obs_version);
        int max_compact = 0;  // the compact-form scratch fits every obs version (mjx_env_set_obs_version switches freely)
        for (int v = 1; v <= 4; v++) {
            const ObsLayout Lv = make_layout(v);
            max_compact = std::max(max_compact, Lv.bm_rows * 8 + Lv.n_sv * OBS_COLS * 4);
        }
        CU(cudaMalloc(&env->d_compact, cap * (size_t)max_compact));  // compact observations (mjx_obs.cuh)
        env->sp_enabled = obs_version == 4 ? 1 : 0;  // the single-player block exists in v4 only
        CU(cudaMalloc(&env->d_enc_work, sizeof(int)));
        CU(cudaMemset(env->d_enc_work, 0, sizeof(int)));
    }
    {
        // state table: the slot index is the state id; ~3K slots per table keeps the load under ~20 % in the heaviest steps seen
        long long want = (long long)n_tables * 3072;
        if (const char* e = getenv("MJX_SP_SLOTS_PER_TABLE")) want = (long long)n_tables * atoll(e);
        env->sp_want_slots = want;
        CU(cudaMalloc(&env->sp.rows, cap * sizeof(SpRow)));
        int rc = sp_alloc(env->sp, want);
        if (rc) return rc;
        int lanes = n_tables >= 1024 ? 2 : 1;  // small batches do not fill the SMs with one DP either, but launch-bound
        if (const char* e = getenv("MJX_SP_LANES")) lanes = std::max(1, std::min(MJX_SP_MAX_LANES, atoi(e)));
        env->sp_lanes = lanes;
        if (const char* e = getenv("MJX_SP_GRID_X")) env->sp_grid_x = std::max(1, atoi(e));
        if (const char* e = getenv("MJX_SP_GRID_E")) env->sp_grid_e = std::max(1, atoi(e));
        if (const char* e = getenv("MJX_SP_THR_X")) env->sp_thr_x = std::max(32, std::min(SP_THREADS, atoi(e) / 32 * 32));
        if (const char* e = getenv("MJX_SP_THR_E")) env->sp_thr_e = std::max(32, std::min(SP_THREADS, atoi(e) / 32 * 32));
    }
    CU(cudaMemset(env->d_dummy_actions, 0, sizeof(i64) * cap));
    CU(cudaMemset(V.masks, 0, cap * ACTION_SPACE));
    CU(cudaMemset(V.scores, 0, sizeof(i32) * 4 * (size_t)n_tables));
    CU(cudaMemset(V.ranks, 0, 4 * (size_t)n_tables));
    CU(cudaMemset(V.n_rows, 0, sizeof(i32)));
    CU(cudaMemset(V.counters, 0, sizeof(unsigned long long) * 4));
    CU(cudaMemcpy(env->d_nonces, nonces, sizeof(u64) * (size_t)n_tables, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(env->d_keys, keys, sizeof(u64) * (size_t)n_tables, cudaMemcpyHostToDevice));
    k_init_tables<<<(n_tables + 127) / 128, 128>>>(V.tables, n_tables, env->d_nonces, env->d_keys, shuffle_kind, V.done,
                                                   V.steps, V.err);
    CU(cudaGetLastError());
    CU(cudaDeviceSynchronize());
    return MJX_OK;
}

// a creator failed half way: free what the env owns, keep the error text of the failure
static int destroy_failed(mjx_env** out, mjx_env* env, int rc) {
    const std::string msg = g_err;
    mjx_env_destroy(env);
    cudaGetLastError();
    if (out) *out = nullptr;
    g_err = msg;
    return rc;
}

extern "C" {

int mjx_env_create(mjx_env** out, int n_tables, const uint64_t* nonces, const uint64_t* keys, int obs_version,
                   int shuffle_kind, int enable_quick_eval) {
    if (out) *out = nullptr;
    if (!g_ready) return fail(MJX_ERR_STATE, "mjx_env_create: call mjx_init first");
    if (!out || n_tables <= 0 || !nonces || !keys) return fail(MJX_ERR_ARG, "mjx_env_create: bad arguments");
    if (obs_version < 1 || obs_version > 4) return fail(MJX_ERR_ARG, "mjx_env_create: obs_version must be 1..4 (consts.rs:18)");
    if (shuffle_kind != 0 && shuffle_kind != 1) return fail(MJX_ERR_ARG, "mjx_env_create: shuffle_kind must be 0 or 1");
    CU(cudaSetDevice(g_device));  // the calling thread may not be the one that ran mjx_init
    mjx_env* env = new mjx_env();
    const int rc = env_create_impl(env, n_tables, nonces, keys, obs_version, shuffle_kind, enable_quick_eval);
    if (rc) return destroy_failed(out, env, rc);  // e.g. out of memory on the single-player state table
    *out = env;
    return MJX_OK;
}

void mjx_env_destroy(mjx_env* env) {
    if (!env) return;
    EnvView& V = env->V;
    cudaFree(V.tables); cudaFree(V.n_rows); cudaFree(V.row_table); cudaFree(V.row_seat); cudaFree(V.row_step);
    cudaFree(V.masks); cudaFree(V.scores); cudaFree(V.ranks); cudaFree(V.done); cudaFree(V.steps); cudaFree(V.err);
    cudaFree(V.counters); cudaFree(env->d_nonces); cudaFree(env->d_keys); cudaFree(env->d_dummy_actions); if (env->replay) {
        ReplayView& R = env->R;
        cudaFree((void*)R.hdr); cudaFree((void*)R.kyoku); cudaFree((void*)R.ev_off); cudaFree((void*)R.ev_cnt); cudaFree((void*)R.ky_off);
        cudaFree((void*)R.player); cudaFree(R.pos); cudaFree(R.ky_idx); cudaFree(R.ky_seen); cudaFree(R.row_label); cudaFree(R.row_meta);
    }
    for (int i = 0; i < 3; i++) if (env->ev_enc[i]) cudaEventDestroy(env->ev_enc[i]);
    cudaFree(env->d_guard); cudaFree(env->d_quick_eval); cudaFree(env->d_compact); cudaFree(env->d_enc_work); cudaFree(env->V.log); cudaFree(env->V.log_len); cudaFree(env->V.grp); cudaFree(env->V.grp_len);
    cudaFree(env->sp.rows);
    sp_free(env->sp);
    for (int g = 1; g < env->sp_lanes_alloc; g++) sp_free(env->sp_lane[g - 1]);
    for (int g = 0; g < MJX_SP_MAX_LANES; g++)
        if (env->sp_stream[g]) { cudaStreamDestroy(env->sp_stream[g]); cudaEventDestroy(env->ev_sp_join[g]); }
    if (env->ev_sp_fork) { cudaEventDestroy(env->ev_sp_fork); cudaEventDestroy(env->ev_sp_store); }
    cudaFree(env->d_state_words); cudaFree(env->d_state_pay); cudaFree(env->d_state_cans); cudaFree(env->d_state_misc);
    if (env->copy_stream) { cudaStreamDestroy(env->copy_stream); cudaEventDestroy(env->ev_rows); cudaEventDestroy(env->ev_sp); for (int g = 0; g < MJX_HOST_COPY_GROUPS; g++) cudaEventDestroy(env->ev_grp[g]); }
    delete env;
}

int mjx_env_set_quick_eval(mjx_env* env, const uint8_t* flags_host) {
    if (!env) return fail(MJX_ERR_ARG, "mjx_env_set_quick_eval: null env");
    if (!flags_host) { cudaFree(env->d_quick_eval); env->d_quick_eval = nullptr; return MJX_OK; }
    if (!env->d_quick_eval) CU(cudaMalloc(&env->d_quick_eval, (size_t)env->n_tables * 4));
    CU(cudaMemcpy(env->d_quick_eval, flags_host, (size_t)env->n_tables * 4, cudaMemcpyHostToDevice));
    return MJX_OK;
}

int mjx_env_set_agari_guard(mjx_env* env, const uint8_t* flags_host) {
    if (!env) return fail(MJX_ERR_ARG, "mjx_env_set_agari_guard: null env");
    if (!flags_host) { cudaFree(env->d_guard); env->d_guard = nullptr; return MJX_OK; }
    if (!env->d_guard) CU(cudaMalloc(&env->d_guard, (size_t)env->n_tables * 4));
    CU(cudaMemcpy(env->d_guard, flags_host, (size_t)env->n_tables * 4, cudaMemcpyHostToDevice));
    return MJX_OK;
}

int mjx_env_step(mjx_env* env, const int64_t* actions_dev, const float* q_values_dev, void* stream) {
    if (!env) return fail(MJX_ERR_ARG, "mjx_env_step: null env");
    if (!env->first && !actions_dev) return fail(MJX_ERR_ARG, "mjx_env_step: actions required after the first step");
    cudaStream_t st = (cudaStream_t)stream;
    EnvView V = env->V;
    V.actions = actions_dev ? (const i64*)actions_dev : env->d_dummy_actions;
    V.q_values = q_values_dev;
    V.agari_guard = env->d_guard;
    V.quick_eval_seat = env->d_quick_eval;
    k_begin_step<<<1, 1, 0, st>>>(V);
    k_step<<<(env->n_tables + STEP_WARPS - 1) / STEP_WARPS, STEP_WARPS * 32, 0, st>>>(V, g_T);
    CU(cudaGetLastError());
    env->launches += 2;
    env->first = false;
    return MJX_OK;
}

static int launch_encode_rows(mjx_env* env, float* obs_dev, cudaStream_t st) {
    if (env->time_encode) CU(cudaEventRecord(env->ev_enc[0], st));
    switch (env->obs_version) {
        case 1: launch_features<1>(env, st); break;
        case 2: launch_features<2>(env, st); break;
        case 3: launch_features<3>(env, st); break;
        default: launch_features<4>(env, st); break;
    }
    if (env->time_encode) CU(cudaEventRecord(env->ev_enc[1], st));
    k_encode_store<<<g_sm_count, ENCS_WARPS * 32, ENCS_SMEM_BYTES, st>>>(env->V, env->enc_args, env->d_compact, obs_dev, env->d_enc_work);
    if (env->time_encode) CU(cudaEventRecord(env->ev_enc[2], st));
    CU(cudaGetLastError());
    env->launches += 2;
    return MJX_OK;
}

// single-player block (rows 889..1011): init -> expand levels 0..7 -> score -> evaluate levels 7..0 -> finalize -> release
// rows [row_lo, row_hi) of the step form one DP (the whole step by default; mjx_env_encode_obs_host runs it in row groups)
// `before_finalize`: an event the stream waits for before the block writes into the observations (the rows must have been stored)
static int launch_sp_block(mjx_env* env, const SpGlobal& G, float* obs_dev, cudaStream_t st, int row_lo = 0, int row_hi = 0x7fffffff,
                           int part = 0, int parts = 1, cudaEvent_t before_finalize = nullptr) {
    if (!env->sp_enabled) return MJX_OK;
    const int grid_rows = g_sm_count * 8, grid = g_sm_count * env->sp_grid_x, grid_eval = g_sm_count * env->sp_grid_e;
    k_sp_begin<<<1, 32, 0, st>>>(G);
    k_sp_init<<<grid_rows, SP_WARPS * 32, 0, st>>>(G, g_T, env->V, row_lo, row_hi, part, parts);
    for (int level = 0; level < SP_SLOTS; level++) {
        if (level == SP_SLOTS - 1) {
            k_sp_mark<<<1, 1, 0, st>>>(G, 0);
            k_sp_expand<2><<<grid, env->sp_thr_x, 0, st>>>(G, g_T, level);
        } else if (sp_slot_is_w(level)) k_sp_expand<1><<<grid, env->sp_thr_x, 0, st>>>(G, g_T, level);
        else k_sp_expand<0><<<grid, env->sp_thr_x, 0, st>>>(G, g_T, level);
    }
    k_sp_mark<<<1, 1, 0, st>>>(G, 1);
    k_sp_densify<<<g_sm_count * 8, 256, 0, st>>>(G);
    k_sp_score<<<g_sm_count * 16, 128, 0, st>>>(G, g_T);
    for (int level = SP_SLOTS - 1; level >= 0; level--) {
        if (!sp_slot_is_w(level)) k_sp_eval<0><<<grid_eval, env->sp_thr_e, 0, st>>>(G, level);
        else if (level == SP_SLOTS - 1) k_sp_eval<2><<<grid_eval, env->sp_thr_e, 0, st>>>(G, level);
        else k_sp_eval<1><<<grid_eval, env->sp_thr_e, 0, st>>>(G, level);
    }
    if (before_finalize) CU(cudaStreamWaitEvent(st, before_finalize, 0));
    k_sp_finalize<<<grid_rows, SP_WARPS * 32, 0, st>>>(G, g_T, env->V, obs_dev, row_lo, row_hi, part, parts);
    k_sp_release<<<g_sm_count * 4, 256, 0, st>>>(G);
    CU(cudaGetLastError());
    env->launches += 7 + 2 * SP_SLOTS + 1;
    return MJX_OK;
}

int mjx_env_encode_obs(mjx_env* env, float* obs_dev, void* stream) {
    if (!env || !obs_dev) return fail(MJX_ERR_ARG, "mjx_env_encode_obs: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    const int lanes = env->sp_enabled ? env->sp_lanes : 0;
    int rc;
    if (lanes <= 1) {
        if ((rc = launch_encode_rows(env, obs_dev, st))) return rc;
        return lanes ? launch_sp_block(env, env->sp, obs_dev, st) : MJX_OK;
    }
    // The step's rows are solved as `lanes` independent DPs on concurrent side streams while this stream runs the two encoder
    // kernels: the latency-bound launches of one lane (small levels, init / finalize / release, the tail of every level) and the
    // bandwidth-bound store run under the other lanes' work. A lane only touches the observations in its last kernel, after the store.
    if ((rc = sp_ensure_lanes(env, lanes))) return rc;
    // (with mjx_env_set_encode_timing the lanes start after the store, so that the two encoder kernels are timed alone)
    if (!env->time_encode) CU(cudaEventRecord(env->ev_sp_fork, st));
    if ((rc = launch_encode_rows(env, obs_dev, st))) return rc;
    CU(cudaEventRecord(env->ev_sp_store, st));
    if (env->time_encode) CU(cudaEventRecord(env->ev_sp_fork, st));
    for (int g = 0; g < lanes; g++) {
        CU(cudaStreamWaitEvent(env->sp_stream[g], env->ev_sp_fork, 0));
        if ((rc = launch_sp_block(env, sp_of(env, g), obs_dev, env->sp_stream[g], 0, 0x7fffffff, g, lanes, env->ev_sp_store))) return rc;
        CU(cudaEventRecord(env->ev_sp_join[g], env->sp_stream[g]));
    }
    for (int g = 0; g < lanes; g++) CU(cudaStreamWaitEvent(st, env->ev_sp_join[g], 0));
    return MJX_OK;
}

int mjx_oracle_obs_rows(int version) { return (version >= 1 && version <= 4) ? oracle_obs_rows(version) : MJX_ERR_ARG; }

int mjx_env_encode_invisible(mjx_env* env, float* inv_dev, int version, void* stream) {
    if (!env || !inv_dev || version < 1 || version > 4) return fail(MJX_ERR_ARG, "mjx_env_encode_invisible: bad arguments");
    // a log replay follows dataset/invisible.rs (every tile left in the live wall), self-play follows board.rs:748-758
    k_encode_invisible<<<g_sm_count * 8, 128, 0, (cudaStream_t)stream>>>(env->V, version, inv_dev, env->replay ? 1 : 0);
    CU(cudaGetLastError());
    env->launches += 1;
    return MJX_OK;
}

int mjx_env_encode_obs_host(mjx_env* env, float* obs_dev, float* obs_host, uint8_t* masks_host, int* n_rows_out, void* stream) {
    int rc = mjx_env_encode_obs_host_begin(env, obs_dev, obs_host, masks_host, n_rows_out, stream);
    if (rc) return rc;
    return mjx_env_encode_obs_host_finish(env);
}

int mjx_env_encode_obs_host_finish(mjx_env* env) {
    if (!env) return fail(MJX_ERR_ARG, "mjx_env_encode_obs_host_finish: null env");
    if (env->copy_stream) CU(cudaStreamSynchronize(env->copy_stream));
    return MJX_OK;
}

int mjx_env_encode_obs_host_begin(mjx_env* env, float* obs_dev, float* obs_host, uint8_t* masks_host, int* n_rows_out, void* stream) {
    if (!env || !obs_dev || !obs_host || !masks_host || !n_rows_out)
        return fail(MJX_ERR_ARG, "mjx_env_encode_obs_host: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    if (!env->copy_stream) {
        CU(cudaStreamCreateWithFlags(&env->copy_stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&env->ev_rows, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&env->ev_sp, cudaEventDisableTiming));
        for (int g = 0; g < MJX_HOST_COPY_GROUPS; g++) CU(cudaEventCreateWithFlags(&env->ev_grp[g], cudaEventDisableTiming));
    }
    int n = 0;
    CU(cudaMemcpyAsync(&n, env->V.n_rows, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *n_rows_out = n;
    if (n == 0) return MJX_OK;
    const size_t pitch = (size_t)env->enc_args.rows * 34 * sizeof(float);  // bytes of one observation
    int rc = launch_encode_rows(env, obs_dev, st);
    if (rc) return rc;
    if (!env->sp_enabled) {
        CU(cudaEventRecord(env->ev_rows, st));
        CU(cudaStreamWaitEvent(env->copy_stream, env->ev_rows, 0));
        CU(cudaMemcpyAsync(obs_host, obs_dev, pitch * (size_t)n, cudaMemcpyDeviceToHost, env->copy_stream));
    } else {
        // The single-player block is computed in row groups, each its own DP, so that the finished observations of one
        // group (one CONTIGUOUS chunk) drain through the copy engine while the SMs work on the next group.
        constexpr int GROUPS = MJX_HOST_COPY_GROUPS;
        for (int g = 0; g < GROUPS; g++) {
            const int r0 = (int)((long long)n * g / GROUPS), r1 = (int)((long long)n * (g + 1) / GROUPS);
            if (r1 <= r0) continue;
            rc = launch_sp_block(env, env->sp, obs_dev, st, r0, r1);
            if (rc) return rc;
            CU(cudaEventRecord(env->ev_grp[g], st));
            CU(cudaStreamWaitEvent(env->copy_stream, env->ev_grp[g], 0));
            CU(cudaMemcpyAsync((char*)obs_host + pitch * (size_t)r0, (const char*)obs_dev + pitch * (size_t)r0, pitch * (size_t)(r1 - r0),
                               cudaMemcpyDeviceToHost, env->copy_stream));
        }
    }
    CU(cudaMemcpyAsync(masks_host, env->V.masks, (size_t)n * MJX_ACTION_SPACE, cudaMemcpyDeviceToHost, env->copy_stream));
    return MJX_OK;
}

int mjx_env_enable_log(mjx_env* env, int words_per_table) {
    if (!env || words_per_table <= 0) return fail(MJX_ERR_ARG, "mjx_env_enable_log: bad arguments");
    if (!env->first) return fail(MJX_ERR_STATE, "mjx_env_enable_log: must be called before the first mjx_env_step");
    if (env->V.log) return MJX_OK;
    CU(cudaMalloc(&env->V.log, (size_t)env->n_tables * (size_t)words_per_table * sizeof(u64)));
    CU(cudaMalloc(&env->V.log_len, (size_t)env->n_tables * sizeof(i32)));
    CU(cudaMemset(env->V.log_len, 0, (size_t)env->n_tables * sizeof(i32)));
    env->V.log_cap = words_per_table;
    return MJX_OK;
}

int mjx_env_enable_grp(mjx_env* env, int max_kyoku) {
    if (!env || max_kyoku <= 0) return fail(MJX_ERR_ARG, "mjx_env_enable_grp: bad arguments");
    if (!env->first) return fail(MJX_ERR_STATE, "mjx_env_enable_grp: must be called before the first mjx_env_step");
    if (env->V.grp) return MJX_OK;
    CU(cudaMalloc(&env->V.grp, (size_t)env->n_tables * (size_t)max_kyoku * 7 * sizeof(i32)));
    CU(cudaMalloc(&env->V.grp_len, (size_t)env->n_tables * sizeof(i32)));
    CU(cudaMemset(env->V.grp_len, 0, (size_t)env->n_tables * sizeof(i32)));
    env->V.grp_cap = max_kyoku;
    return MJX_OK;
}

int mjx_env_read_grp(mjx_env* env, void* stream, int32_t* feat_host, int32_t* n_kyoku_host) {
    if (!env || !feat_host || !n_kyoku_host) return fail(MJX_ERR_ARG, "mjx_env_read_grp: bad arguments");
    if (!env->V.grp) return fail(MJX_ERR_STATE, "mjx_env_read_grp: mjx_env_enable_grp was not called");
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    CU(cudaMemcpy(n_kyoku_host, env->V.grp_len, (size_t)env->n_tables * sizeof(i32), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(feat_host, env->V.grp, (size_t)env->n_tables * (size_t)env->V.grp_cap * 7 * sizeof(i32), cudaMemcpyDeviceToHost));
    return MJX_OK;
}

int32_t* mjx_env_log_len_dev(mjx_env* env) { return env ? env->V.log_len : nullptr; }

int mjx_env_read_log(mjx_env* env, void* stream, uint64_t* words_host, int32_t* len_host) {
    if (!env || !words_host || !len_host) return fail(MJX_ERR_ARG, "mjx_env_read_log: bad arguments");
    if (!env->V.log) return fail(MJX_ERR_STATE, "mjx_env_read_log: mjx_env_enable_log was not called");
    cudaStream_t st = (cudaStream_t)stream;
    CU(cudaStreamSynchronize(st));
    CU(cudaMemcpy(len_host, env->V.log_len, (size_t)env->n_tables * sizeof(i32), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(words_host, env->V.log, (size_t)env->n_tables * (size_t)env->V.log_cap * sizeof(u64), cudaMemcpyDeviceToHost));
    return MJX_OK;
}

int mjx_env_create_replay(mjx_env** out, int n_jobs, const uint64_t* hdr, const int32_t* ev_off, const int32_t* ev_cnt, long long n_hdr,
                          const uint64_t* kyoku, const int32_t* ky_off, long long n_kyoku_words, const uint8_t* players,
                          int obs_version, int always_include_kan_select) {
    if (!out || n_jobs <= 0 || !hdr || !ev_off || !ev_cnt || !ky_off || !players || n_hdr <= 0)
        return fail(MJX_ERR_ARG, "mjx_env_create_replay: bad arguments");
    std::vector<uint64_t> zeros((size_t)n_jobs, 0);
    int rc = mjx_env_create(out, n_jobs, zeros.data(), zeros.data(), obs_version, 0, 0);
    if (rc) return rc;
    mjx_env* env = *out;
    env->replay = true;
    rc = [&]() -> int {  // every buffer belongs to the env as soon as it exists, so a failure below frees it with the env
        ReplayView& R = env->R;
        const size_t cap = (size_t)env->row_cap;
        CU(cudaMalloc((void**)&R.hdr, sizeof(u64) * (size_t)n_hdr));
        CU(cudaMalloc((void**)&R.kyoku, sizeof(u64) * (size_t)(n_kyoku_words > 0 ? n_kyoku_words : 1)));
        CU(cudaMalloc((void**)&R.ev_off, sizeof(i32) * (size_t)n_jobs));
        CU(cudaMalloc((void**)&R.ev_cnt, sizeof(i32) * (size_t)n_jobs));
        CU(cudaMalloc((void**)&R.ky_off, sizeof(i32) * (size_t)n_jobs));
        CU(cudaMalloc((void**)&R.player, (size_t)n_jobs));
        CU(cudaMalloc(&R.pos, sizeof(i32) * (size_t)n_jobs));
        CU(cudaMalloc(&R.ky_idx, sizeof(i32) * (size_t)n_jobs));
        CU(cudaMalloc(&R.ky_seen, sizeof(i32) * (size_t)n_jobs));
        CU(cudaMalloc(&R.row_label, sizeof(i64) * cap));
        CU(cudaMalloc(&R.row_meta, cap * 4));
        CU(cudaMemcpy((void*)R.hdr, hdr, sizeof(u64) * (size_t)n_hdr, cudaMemcpyHostToDevice));
        if (n_kyoku_words > 0) CU(cudaMemcpy((void*)R.kyoku, kyoku, sizeof(u64) * (size_t)n_kyoku_words, cudaMemcpyHostToDevice));
        CU(cudaMemcpy((void*)R.ev_off, ev_off, sizeof(i32) * (size_t)n_jobs, cudaMemcpyHostToDevice));
        CU(cudaMemcpy((void*)R.ev_cnt, ev_cnt, sizeof(i32) * (size_t)n_jobs, cudaMemcpyHostToDevice));
        CU(cudaMemcpy((void*)R.ky_off, ky_off, sizeof(i32) * (size_t)n_jobs, cudaMemcpyHostToDevice));
        CU(cudaMemcpy((void*)R.player, players, (size_t)n_jobs, cudaMemcpyHostToDevice));
        CU(cudaMemset(R.pos, 0, sizeof(i32) * (size_t)n_jobs));
        CU(cudaMemset(R.ky_idx, 0, sizeof(i32) * (size_t)n_jobs));
        CU(cudaMemset(R.ky_seen, 0, sizeof(i32) * (size_t)n_jobs));
        R.always_include_kan_select = always_include_kan_select ? 1 : 0;
        return MJX_OK;
    }();
    if (rc) return destroy_failed(out, env, rc);
    return MJX_OK;
}

// ---- libriichi.state.PlayerState batch
int mjx_state_create(mjx_env** out, int n, const uint8_t* player_ids_host, int obs_version) {
    if (!out || n <= 0 || !player_ids_host) return fail(MJX_ERR_ARG, "mjx_state_create: bad arguments");
    for (int i = 0; i < n; i++) if (player_ids_host[i] > 3) return fail(MJX_ERR_ARG, "mjx_state_create: player_id must be within 0..3");
    std::vector<uint64_t> zeros((size_t)n, 0);
    int rc = mjx_env_create(out, n, zeros.data(), zeros.data(), obs_version, 0, 0);
    if (rc) return rc;
    mjx_env* env = *out;
    env->is_state = true;
    rc = [&]() -> int {
        CU(cudaMalloc(&env->d_state_words, sizeof(u64) * (size_t)n));
        u8* d_ids = reinterpret_cast<u8*>(env->d_state_words);  // n bytes of scratch until the first update
        CU(cudaMemcpy(d_ids, player_ids_host, (size_t)n, cudaMemcpyHostToDevice));
        k_state_init<<<(n + 127) / 128, 128>>>(env->V.tables, n, d_ids);
        CU(cudaGetLastError());
        CU(cudaDeviceSynchronize());
        CU(cudaMalloc(&env->d_state_pay, sizeof(u64) * (size_t)n * REPLAY_KYOKU_WORDS));
        CU(cudaMalloc(&env->d_state_cans, sizeof(u32) * (size_t)n));
        CU(cudaMalloc(&env->d_state_misc, 256));
        return MJX_OK;
    }();
    if (rc) return destroy_failed(out, env, rc);
    return MJX_OK;
}

int mjx_state_update(mjx_env* env, const uint64_t* words_host, const uint64_t* payload_host, uint32_t* cans_host) {
    if (!env || !env->is_state || !words_host || !cans_host) return fail(MJX_ERR_ARG, "mjx_state_update: bad arguments");
    const size_t n = (size_t)env->n_tables;
    CU(cudaMemcpy(env->d_state_words, words_host, sizeof(u64) * n, cudaMemcpyHostToDevice));
    if (payload_host) CU(cudaMemcpy(env->d_state_pay, payload_host, sizeof(u64) * n * REPLAY_KYOKU_WORDS, cudaMemcpyHostToDevice));
    k_state_update<<<(env->n_tables + STEP_WARPS - 1) / STEP_WARPS, STEP_WARPS * 32>>>(env->V, g_T, env->d_state_words,
                                                                                       payload_host ? env->d_state_pay : nullptr, env->d_state_cans);
    CU(cudaGetLastError());
    CU(cudaMemcpy(cans_host, env->d_state_cans, sizeof(u32) * n, cudaMemcpyDeviceToHost));
    env->launches += 1;
    return MJX_OK;
}

int mjx_state_view(mjx_env* env, int index, mjx_player_view* out_host) {
    if (!env || !env->is_state || !out_host || index < 0 || index >= env->n_tables) return fail(MJX_ERR_ARG, "mjx_state_view: bad arguments");
    static_assert(sizeof(mjx_player_view) <= 512, "view scratch");
    mjx_player_view* d = nullptr;
    CU(cudaMalloc(&d, sizeof(mjx_player_view)));
    CU(cudaMemset(d, 0, sizeof(mjx_player_view)));
    k_state_view<<<(env->n_tables + STEP_WARPS - 1) / STEP_WARPS, STEP_WARPS * 32>>>(env->V, g_T, index, d);
    cudaError_t e = cudaMemcpy(out_host, d, sizeof(mjx_player_view), cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(MJX_ERR_CUDA, std::string("mjx_state_view: ") + cudaGetErrorString(e));
    return MJX_OK;
}

int mjx_state_rows(mjx_env* env, const uint8_t* at_kan_select_host, void* stream) {
    if (!env || !env->is_state) return fail(MJX_ERR_ARG, "mjx_state_rows: not a state batch");
    cudaStream_t st = (cudaStream_t)stream;
    u8* d_kan = nullptr;
    if (at_kan_select_host) {
        d_kan = reinterpret_cast<u8*>(env->d_state_words);  // scratch: n bytes fit in the n words
        CU(cudaMemcpyAsync(d_kan, at_kan_select_host, (size_t)env->n_tables, cudaMemcpyHostToDevice, st));
    }
    k_state_rows<<<(env->n_tables + STEP_WARPS - 1) / STEP_WARPS, STEP_WARPS * 32, 0, st>>>(env->V, g_T, d_kan);
    CU(cudaGetLastError());
    env->launches += 1;
    return MJX_OK;
}

int mjx_state_query(mjx_env* env, int index, int what, const int32_t* args, int32_t* out) {
    if (!env || !env->is_state || !out || index < 0 || index >= env->n_tables || what < 0 || what > 4)
        return fail(MJX_ERR_ARG, "mjx_state_query: bad arguments");
    i32* d = reinterpret_cast<i32*>(env->d_state_misc);
    i32 host_args[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (args) for (int k = 0; k < 8; k++) host_args[k] = args[k];
    CU(cudaMemcpy(d, host_args, sizeof host_args, cudaMemcpyHostToDevice));
    CU(cudaMemset(d + 8, 0, 8 * sizeof(i32)));
    k_state_query<<<(env->n_tables + STEP_WARPS - 1) / STEP_WARPS, STEP_WARPS * 32>>>(env->V, g_T, index, what, d, d + 8);
    CU(cudaGetLastError());
    CU(cudaMemcpy(out, d + 8, 4 * sizeof(i32), cudaMemcpyDeviceToHost));
    return MJX_OK;
}

int mjx_state_copy(mjx_env* dst, int dst_index, mjx_env* src, int src_index) {
    if (!dst || !src || !dst->is_state || !src->is_state || dst_index < 0 || dst_index >= dst->n_tables || src_index < 0 ||
        src_index >= src->n_tables)
        return fail(MJX_ERR_ARG, "mjx_state_copy: bad arguments");
    CU(cudaMemcpy(dst->V.tables + dst_index, src->V.tables + src_index, sizeof(TableState), cudaMemcpyDeviceToDevice));
    return MJX_OK;
}

int mjx_env_replay_trust_seeds(mjx_env* env, const uint64_t* nonces_host, const uint64_t* keys_host, int shuffle_kind) {
    if (!env || !env->replay || !nonces_host || !keys_host) return fail(MJX_ERR_ARG, "mjx_env_replay_trust_seeds: bad arguments");
    if (!env->first) return fail(MJX_ERR_STATE, "mjx_env_replay_trust_seeds: must be called before the first mjx_env_replay_step");
    if (shuffle_kind != 0 && shuffle_kind != 1) return fail(MJX_ERR_ARG, "mjx_env_replay_trust_seeds: shuffle_kind must be 0 or 1");
    const size_t n = (size_t)env->n_tables;
    CU(cudaMemcpy(env->d_nonces, nonces_host, sizeof(u64) * n, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(env->d_keys, keys_host, sizeof(u64) * n, cudaMemcpyHostToDevice));
    k_set_seeds<<<(env->n_tables + 127) / 128, 128>>>(env->V.tables, env->n_tables, env->d_nonces, env->d_keys, shuffle_kind);
    CU(cudaGetLastError());
    CU(cudaDeviceSynchronize());
    env->R.trust_seed = 1;
    return MJX_OK;
}

int mjx_env_replay_step(mjx_env* env, void* stream) {
    if (!env || !env->replay) return fail(MJX_ERR_ARG, "mjx_env_replay_step: not a replay env");
    cudaStream_t st = (cudaStream_t)stream;
    k_begin_step<<<1, 1, 0, st>>>(env->V);
    k_replay_step<<<(env->n_tables + STEP_WARPS - 1) / STEP_WARPS, STEP_WARPS * 32, 0, st>>>(env->V, env->R, g_T);
    CU(cudaGetLastError());
    env->launches += 2;
    env->first = false;
    return MJX_OK;
}
int64_t* mjx_env_row_label(mjx_env* env) { return env && env->replay ? (int64_t*)env->R.row_label : nullptr; }
uint8_t* mjx_env_row_meta(mjx_env* env) { return env && env->replay ? env->R.row_meta : nullptr; }

int mjx_env_set_encode_timing(mjx_env* env, int enable) {
    if (!env) return fail(MJX_ERR_ARG, "mjx_env_set_encode_timing: null env");
    if (enable && !env->ev_enc[0]) for (int i = 0; i < 3; i++) CU(cudaEventCreate(&env->ev_enc[i]));
    env->time_encode = enable != 0;
    return MJX_OK;
}
int mjx_env_last_encode_ms(mjx_env* env, float* ms_features, float* ms_store) {
    if (!env || !ms_features || !ms_store || !env->ev_enc[0]) return fail(MJX_ERR_ARG, "mjx_env_last_encode_ms: timing not enabled");
    CU(cudaEventSynchronize(env->ev_enc[2]));
    CU(cudaEventElapsedTime(ms_features, env->ev_enc[0], env->ev_enc[1]));
    CU(cudaEventElapsedTime(ms_store, env->ev_enc[1], env->ev_enc[2]));
    return MJX_OK;
}

long long mjx_env_launch_count(mjx_env* env) { return env ? env->launches : -1; }

int mjx_env_set_obs_version(mjx_env* env, int version) {
    if (!env || version < 1 || version > 4) return fail(MJX_ERR_ARG, "mjx_env_set_obs_version: version must be 1..4 (consts.rs:18)");
    env->obs_version = version;
    set_enc_args(env, version);
    env->sp_enabled = (version == 4 && env->sp_wanted) ? 1 : 0;
    return MJX_OK;
}

int mjx_env_set_sp(mjx_env* env, int enable) {
    if (!env) return fail(MJX_ERR_ARG, "mjx_env_set_sp: null env");
    env->sp_wanted = enable ? 1 : 0;
    env->sp_enabled = (enable && env->obs_version == 4) ? 1 : 0;
    return MJX_OK;
}

int mjx_env_sp_overflows(mjx_env* env, void* stream, int* n) {
    if (!env || !n) return fail(MJX_ERR_ARG, "mjx_env_sp_overflows: bad arguments");
    int cnt[MJX_SP_MAX_LANES][4] = {};
    for (int g = 0; g < env->sp_lanes_alloc; g++)
        CU(cudaMemcpyAsync(cnt[g], sp_of(env, g).counters, sizeof cnt[g], cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    *n = 0;
    for (int g = 0; g < env->sp_lanes_alloc; g++) *n += cnt[g][3] + (cnt[g][2] ? 1 : 0);
    return MJX_OK;
}

int mjx_env_sp_stats(mjx_env* env, void* stream, int* out10) {
    if (!env || !out10) return fail(MJX_ERR_ARG, "mjx_env_sp_stats: bad arguments");
    int cnt[MJX_SP_MAX_LANES][8] = {}, wl[MJX_SP_MAX_LANES][SP_SLOTS] = {};
    for (int g = 0; g < env->sp_lanes_alloc; g++) {
        CU(cudaMemcpyAsync(cnt[g], sp_of(env, g).counters, sizeof cnt[g], cudaMemcpyDeviceToHost, (cudaStream_t)stream));
        CU(cudaMemcpyAsync(wl[g], sp_of(env, g).wl_count, sizeof wl[g], cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    }
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    for (int i = 0; i < 10; i++) out10[i] = 0;
    for (int g = 0; g < env->sp_lanes_alloc; g++) {
        for (int i = 0; i < SP_SLOTS; i++) { out10[2 + i] += wl[g][i]; out10[0] += wl[g][i]; }  // states = sum of the level work lists
        out10[1] += cnt[g][1];                                                                    // edges
    }
    return MJX_OK;
}

int mjx_env_num_rows(mjx_env* env, void* stream, int* n_rows) {
    if (!env || !n_rows) return fail(MJX_ERR_ARG, "mjx_env_num_rows: bad arguments");
    CU(cudaMemcpyAsync(n_rows, env->V.n_rows, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    return MJX_OK;
}

int mjx_env_poll(mjx_env* env, void* stream, int* out4) {
    if (!env || !out4) return fail(MJX_ERR_ARG, "mjx_env_poll: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long c[4] = {0, 0, 0, 0};
    int sp[MJX_SP_MAX_LANES][4] = {};
    CU(cudaMemcpyAsync(&out4[0], env->V.n_rows, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(c, env->V.counters, sizeof c, cudaMemcpyDeviceToHost, st));
    if (env->sp.counters)
        for (int g = 0; g < env->sp_lanes_alloc; g++) CU(cudaMemcpyAsync(sp[g], sp_of(env, g).counters, sizeof sp[g], cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    out4[1] = (int)c[0];
    out4[2] = (int)c[2];
    out4[3] = 0;
    for (int g = 0; g < env->sp_lanes_alloc; g++) out4[3] += sp[g][3] + (sp[g][2] ? 1 : 0);
    return MJX_OK;
}

int mjx_env_num_live(mjx_env* env, void* stream, int* n_live) {
    if (!env || !n_live) return fail(MJX_ERR_ARG, "mjx_env_num_live: bad arguments");
    unsigned long long v = 0;
    CU(cudaMemcpyAsync(&v, env->V.counters, sizeof v, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    *n_live = (int)v;
    return MJX_OK;
}

int mjx_env_total_steps(mjx_env* env, void* stream, int64_t* steps) {
    if (!env || !steps) return fail(MJX_ERR_ARG, "mjx_env_total_steps: bad arguments");
    unsigned long long v = 0;
    CU(cudaMemcpyAsync(&v, env->V.counters + 1, sizeof v, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    *steps = (int64_t)v;
    return MJX_OK;
}

int mjx_env_row_cap(mjx_env* env) { return env ? env->row_cap : MJX_ERR_ARG; }
uint8_t* mjx_env_masks(mjx_env* env) { return env ? env->V.masks : nullptr; }
int32_t* mjx_env_row_table(mjx_env* env) { return env ? env->V.row_table : nullptr; }
uint8_t* mjx_env_row_seat(mjx_env* env) { return env ? env->V.row_seat : nullptr; }
uint32_t* mjx_env_row_step(mjx_env* env) { return env ? env->V.row_step : nullptr; }
int32_t* mjx_env_num_rows_dev(mjx_env* env) { return env ? env->V.n_rows : nullptr; }

int mjx_env_results(mjx_env* env, void* stream, int32_t* scores, uint8_t* ranks, int32_t* steps, int32_t* err,
                    int32_t* done) {
    if (!env) return fail(MJX_ERR_ARG, "mjx_env_results: null env");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)env->n_tables;
    CU(cudaStreamSynchronize(st));
    if (scores) CU(cudaMemcpy(scores, env->V.scores, sizeof(i32) * 4 * n, cudaMemcpyDeviceToHost));
    if (ranks) CU(cudaMemcpy(ranks, env->V.ranks, 4 * n, cudaMemcpyDeviceToHost));
    if (steps) CU(cudaMemcpy(steps, env->V.steps, sizeof(i32) * n, cudaMemcpyDeviceToHost));
    if (err) CU(cudaMemcpy(err, env->V.err, sizeof(i32) * n, cudaMemcpyDeviceToHost));
    if (done) CU(cudaMemcpy(done, env->V.done, sizeof(i32) * n, cudaMemcpyDeviceToHost));
    return MJX_OK;
}

int mjx_env_policy_test(mjx_env* env, int kind, int64_t* actions_dev, int64_t* trace_dev, float* q_values_dev, void* stream) {
    if (!env || !actions_dev) return fail(MJX_ERR_ARG, "mjx_env_policy_test: bad arguments");
    k_policy_test<<<g_sm_count * 2, 128, 0, (cudaStream_t)stream>>>(env->V, kind, (i64*)actions_dev, (i64*)trace_dev, q_values_dev);
    CU(cudaGetLastError());
    env->launches += 1;
    return MJX_OK;
}

// ---- policy-net helpers (csrc/mjx_nn.cuh): bf16 NHWC activations [batch, length, channels], channels % 8 == 0
static int nn_grid(size_t n_items) {
    size_t g = (n_items + 255) / 256;
    const size_t cap = (size_t)g_sm_count * 16;
    return (int)(g < cap ? (g ? g : 1) : cap);
}
// a grid of 256-thread CTAs whose total thread count is a multiple of c8 (every thread then keeps one channel group for the whole
// grid-stride loop): gridDim is rounded up to a multiple of c8 / gcd(c8, 256)
static int nn_grid_for(size_t n_items, int c8) {
    int q = c8, p = 256;
    while (p) { const int t = q % p; q = p; p = t; }  // q = gcd(c8, 256)
    const int unit = c8 / q;
    const int g = nn_grid(n_items);
    return (g + unit - 1) / unit * unit;
}
int mjx_nn_affine_mish_bf16(const void* x, const float* scale, const float* bias, void* out, long long n_elems, int channels,
                            void* stream) {
    if (!x || !scale || !bias || !out || channels <= 0 || channels % 8 || n_elems % channels)
        return fail(MJX_ERR_ARG, "mjx_nn_affine_mish_bf16: bad arguments");
    if (!g_ready) return fail(MJX_ERR_STATE, "mjx_nn_*: call mjx_init first");
    const size_t n_vec = (size_t)n_elems / 8;
    mjx_nn::k_affine_mish<<<nn_grid_for(n_vec, channels / 8), 256, 0, (cudaStream_t)stream>>>((const mjx_nn::Vec8*)x, scale, bias, (mjx_nn::Vec8*)out,
                                                                            n_vec, channels / 8);
    CU(cudaGetLastError());
    return MJX_OK;
}
int mjx_nn_pool_bf16(const void* x, void* avg, void* mx, int batch, int length, int channels, void* stream) {
    if (!x || !avg || !mx || batch <= 0 || length <= 0 || channels <= 0 || channels % 8)
        return fail(MJX_ERR_ARG, "mjx_nn_pool_bf16: bad arguments");
    if (!g_ready) return fail(MJX_ERR_STATE, "mjx_nn_*: call mjx_init first");
    mjx_nn::k_pool<<<nn_grid((size_t)batch * (channels / 8)), 256, 0, (cudaStream_t)stream>>>(
        (const mjx_nn::Vec8*)x, (mjx_nn::Vec8*)avg, (mjx_nn::Vec8*)mx, batch, length, channels / 8);
    CU(cudaGetLastError());
    return MJX_OK;
}
int mjx_nn_obs_to_nhwc_bf16(const float* obs, void* out, int batch, int channels, int length, int channels_padded, void* stream) {
    if (!obs || !out || batch <= 0 || channels <= 0 || length <= 0 || length > 128 || channels_padded < channels ||
        channels_padded % mjx_nn::NHWC_TC)
        return fail(MJX_ERR_ARG, "mjx_nn_obs_to_nhwc_bf16: bad arguments (channels_padded a multiple of 64, length <= 128)");
    if (!g_ready) return fail(MJX_ERR_STATE, "mjx_nn_*: call mjx_init first");
    const size_t smem = (size_t)mjx_nn::NHWC_TC * (length + 1) * sizeof(float);
    const long long grid = (long long)batch * (channels_padded / mjx_nn::NHWC_TC);
    if (grid > 0x7fffffffLL) return fail(MJX_ERR_ARG, "mjx_nn_obs_to_nhwc_bf16: batch too large");
    mjx_nn::k_obs_to_nhwc<false><<<(int)grid, 256, smem, (cudaStream_t)stream>>>(obs, (__nv_bfloat16*)out, channels, length, channels_padded,
                                                                          nullptr, nullptr);
    CU(cudaGetLastError());
    return MJX_OK;
}
int mjx_nn_obs_rows_to_nhwc_bf16(const float* obs, const int* rows, const int* count, void* out, int batch, int channels, int length,
                                 int channels_padded, void* stream) {
    if (!obs || !rows || !count || !out || batch <= 0 || channels <= 0 || length <= 0 || length > 128 || channels_padded < channels ||
        channels_padded % mjx_nn::NHWC_TC)
        return fail(MJX_ERR_ARG, "mjx_nn_obs_rows_to_nhwc_bf16: bad arguments (channels_padded a multiple of 64, length <= 128)");
    if (!g_ready) return fail(MJX_ERR_STATE, "mjx_nn_*: call mjx_init first");
    const size_t smem = (size_t)mjx_nn::NHWC_TC * (length + 1) * sizeof(float);
    const long long grid = (long long)batch * (channels_padded / mjx_nn::NHWC_TC);
    if (grid > 0x7fffffffLL) return fail(MJX_ERR_ARG, "mjx_nn_obs_rows_to_nhwc_bf16: batch too large");
    mjx_nn::k_obs_to_nhwc<true><<<(int)grid, 256, smem, (cudaStream_t)stream>>>(obs, (__nv_bfloat16*)out, channels, length, channels_padded,
                                                                         rows, count);
    CU(cudaGetLastError());
    return MJX_OK;
}
int mjx_select_actions(const float* v, long long v_stride, const float* a, long long a_stride, const int* rows, const int* count,
                       int n_max, const void* masks, const int* row_table, const uint32_t* row_step, const uint8_t* row_seat,
                       unsigned long long seed, int table_offset, float epsilon, float temp, float top_p, int64_t* actions,
                       float* q_out, uint8_t* greedy, void* stream) {
    if (!v || !a || !count || !masks || !row_table || !row_step || !row_seat || !actions || !q_out || n_max < 0 || a_stride < 46 ||
        v_stride < 1 || epsilon < 0.f || epsilon > 1.f || (epsilon > 0.f && !(temp > 0.f)))
        return fail(MJX_ERR_ARG, "mjx_select_actions: bad arguments");
    if (n_max == 0) return MJX_OK;
    mjx_sel::SelectArgs A{v, v_stride, a, a_stride, rows, count, n_max, (const uint8_t*)masks, row_table, row_step, row_seat,
                          (uint32_t)seed, (uint32_t)(seed >> 32), table_offset, epsilon, epsilon > 0.f ? 1.f / temp : 1.f, top_p,
                          actions, q_out, greedy};
    const int warps_per_cta = 8;
    const int grid = std::max(1, std::min((n_max + warps_per_cta - 1) / warps_per_cta, g_sm_count * 16));
    mjx_sel::k_select_actions<<<grid, warps_per_cta * 32, 0, (cudaStream_t)stream>>>(A);
    CU(cudaGetLastError());
    return MJX_OK;
}
int mjx_split_rows(const int* row_table, const uint8_t* row_seat, const int* count, const uint8_t* agent_of, int* rows0, int* rows1,
                   int* counts, void* stream) {
    if (!row_table || !row_seat || !count || !agent_of || !rows0 || !rows1 || !counts)
        return fail(MJX_ERR_ARG, "mjx_split_rows: bad arguments");
    mjx_sel::k_split_rows<<<1, mjx_sel::SPLIT_THREADS, 0, (cudaStream_t)stream>>>(row_table, row_seat, count, agent_of, rows0, rows1,
                                                                                 counts);
    CU(cudaGetLastError());
    return MJX_OK;
}
int mjx_nn_block_tail_bf16(const void* y, const void* x, const float* w1, const float* b1, const float* w2t, const float* b2,
                           const float* scale, const float* bias, void* gate_scratch, void* x_out, void* a_out, int batch, int length,
                           int channels, int hidden, void* stream) {
    if (!y || !x || !w1 || !b1 || !w2t || !b2 || !scale || !bias || !gate_scratch || !x_out || !a_out || batch <= 0 || length <= 0 ||
        channels <= 0 || channels % 8 || channels > 256 || hidden <= 0 || hidden > 64)
        return fail(MJX_ERR_ARG, "mjx_nn_block_tail_bf16: bad arguments (channels % 8 == 0, <= 256; hidden <= 64)");
    if (!g_ready) return fail(MJX_ERR_STATE, "mjx_nn_*: call mjx_init first");
    cudaStream_t st = (cudaStream_t)stream;
    const int c8 = channels / 8;
    const int warps_per_cta = 8;
    const int grid = std::max(1, std::min((batch + warps_per_cta - 1) / warps_per_cta, g_sm_count * 8));
    mjx_nn::k_pool_gate<<<grid, warps_per_cta * 32, 0, st>>>((const mjx_nn::Vec8*)y, w1, b1, w2t, b2, (mjx_nn::Vec8*)gate_scratch, batch, length,
                                                               c8, hidden);
    CU(cudaGetLastError());
    const size_t n_vec = (size_t)batch * length * c8;
    mjx_nn::k_gate_residual_mish<<<nn_grid_for(n_vec, c8), 256, 0, st>>>(
        (const mjx_nn::Vec8*)y, (const mjx_nn::Vec8*)gate_scratch, (const mjx_nn::Vec8*)x, scale, bias, (mjx_nn::Vec8*)x_out,
        (mjx_nn::Vec8*)a_out, n_vec, length, c8);
    CU(cudaGetLastError());
    return MJX_OK;
}
int mjx_nn_gate_residual_bf16(const void* y, const void* gate, const void* x, void* out, int batch, int length, int channels,
                              void* stream) {
    if (!y || !gate || !x || !out || batch <= 0 || length <= 0 || channels <= 0 || channels % 8)
        return fail(MJX_ERR_ARG, "mjx_nn_gate_residual_bf16: bad arguments");
    if (!g_ready) return fail(MJX_ERR_STATE, "mjx_nn_*: call mjx_init first");
    const size_t n_vec = (size_t)batch * length * (channels / 8);
    mjx_nn::k_gate_residual<<<nn_grid(n_vec), 256, 0, (cudaStream_t)stream>>>((const mjx_nn::Vec8*)y, (const mjx_nn::Vec8*)gate,
                                                                              (const mjx_nn::Vec8*)x, (mjx_nn::Vec8*)out, n_vec,
                                                                              length, channels / 8);
    CU(cudaGetLastError());
    return MJX_OK;
}

int mjx_shanten(const uint8_t* tiles_dev, const uint8_t* len_dev, int8_t* out_dev, int n, void* stream) {
    if (!g_ready) return fail(MJX_ERR_STATE, "mjx_shanten: call mjx_init first");
    if (n <= 0) return MJX_OK;
    k_shanten<<<(n + SH_THREADS - 1) / SH_THREADS, SH_THREADS, 0, (cudaStream_t)stream>>>(g_T, tiles_dev, len_dev,
                                                                                         (i8*)out_dev, n);
    CU(cudaGetLastError());
    return MJX_OK;
}

int mjx_agari(const mjx_agari_in* in_dev, mjx_agari_out* out_dev, int n, int mode, void* stream) {
    if (!g_ready) return fail(MJX_ERR_STATE, "mjx_agari: call mjx_init first");
    if (mode < 0 || mode > 3) return fail(MJX_ERR_ARG, "mjx_agari: mode must be 0..3");
    if (n <= 0) return MJX_OK;
    k_agari<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(g_T, in_dev, out_dev, n, mode);
    CU(cudaGetLastError());
    return MJX_OK;
}

// grow-only device scratch of the *_host entry points (they are called repeatedly with similar sizes: no cudaMalloc per call)
namespace {
struct HostScratch {
    std::mutex mu;
    void* p[3] = {nullptr, nullptr, nullptr};
    size_t cap[3] = {0, 0, 0};
    int reserve(int i, size_t bytes, void** out) {
        if (cap[i] < bytes) {
            cudaFree(p[i]); p[i] = nullptr; cap[i] = 0;
            size_t want = 1 << 16;
            while (want < bytes) want <<= 1;
            cudaError_t e = cudaMalloc(&p[i], want);
            if (e != cudaSuccess) return fail(MJX_ERR_CUDA, cudaGetErrorString(e));
            cap[i] = want;
        }
        *out = p[i];
        return MJX_OK;
    }
};
HostScratch g_host_scratch;
}  // namespace

int mjx_shanten_host(const uint8_t* tiles, const uint8_t* len_div3, int8_t* out, int n) {
    if (!g_ready) return fail(MJX_ERR_STATE, "mjx_shanten_host: call mjx_init first");
    if (n <= 0) return MJX_OK;
    std::lock_guard<std::mutex> lk(g_host_scratch.mu);
    void *d_t = nullptr, *d_l = nullptr, *d_o = nullptr;
    int rc;
    if ((rc = g_host_scratch.reserve(0, (size_t)n * 34, &d_t)) || (rc = g_host_scratch.reserve(1, (size_t)n, &d_l)) ||
        (rc = g_host_scratch.reserve(2, (size_t)n, &d_o)))
        return rc;
    CU(cudaMemcpy(d_t, tiles, (size_t)n * 34, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_l, len_div3, (size_t)n, cudaMemcpyHostToDevice));
    rc = mjx_shanten((const uint8_t*)d_t, (const uint8_t*)d_l, (int8_t*)d_o, n, nullptr);
    if (rc == MJX_OK) {
        cudaError_t e = cudaMemcpy(out, d_o, (size_t)n, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) rc = fail(MJX_ERR_CUDA, cudaGetErrorString(e));
    }
    return rc;
}

int mjx_agari_host(const mjx_agari_in* in, mjx_agari_out* out, int n, int mode) {
    if (!g_ready) return fail(MJX_ERR_STATE, "mjx_agari_host: call mjx_init first");
    if (n <= 0) return MJX_OK;
    std::lock_guard<std::mutex> lk(g_host_scratch.mu);
    void *d_i = nullptr, *d_o = nullptr;
    int rc;
    if ((rc = g_host_scratch.reserve(0, sizeof(mjx_agari_in) * (size_t)n, &d_i)) || (rc = g_host_scratch.reserve(1, sizeof(mjx_agari_out) * (size_t)n, &d_o)))
        return rc;
    CU(cudaMemcpy(d_i, in, sizeof(mjx_agari_in) * (size_t)n, cudaMemcpyHostToDevice));
    rc = mjx_agari((const mjx_agari_in*)d_i, (mjx_agari_out*)d_o, n, mode, nullptr);
    if (rc == MJX_OK) {
        cudaError_t e = cudaMemcpy(out, d_o, sizeof(mjx_agari_out) * (size_t)n, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) rc = fail(MJX_ERR_CUDA, cudaGetErrorString(e));
    }
    return rc;
}

int mjx_make_wall_host(uint64_t nonce, uint64_t key, int kyoku, int honba, int shuffle_kind, uint8_t* wall136) {
    if (!g_ready) return fail(MJX_ERR_STATE, "mjx_make_wall_host: call mjx_init first");
    u8* d = nullptr;
    CU(cudaMalloc(&d, 136));
    k_make_wall<<<1, 32>>>(nonce, key, kyoku, honba, shuffle_kind, d);
    CU(cudaGetLastError());
    CU(cudaMemcpy(wall136, d, 136, cudaMemcpyDeviceToHost));
    cudaFree(d);
    return MJX_OK;
}

}  // extern "C"
