// bfgpu.cu — host side of the B200 proving backend: context, device-memory plumbing and the C ABI
// declared in include/bfgpu.h.  One translation unit: the kernels live in the .cuh files included
// below so that the Poseidon2 constant bank is a single __constant__ object.
//
// Mirrors, phase by phase, what the reference does on the CPU in `CpuProver::commit`
// (reference crates/stark/src/prover.rs:209-236) through Plonky3's `TwoAdicFriPcs::commit`
// (coset LDE + bit-reversed rows + MerkleTreeMmcs::commit).  There is no CPU fallback.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/bfgpu.h"
#include "kb31.cuh"
#include "poseidon2.cuh"
#include "rc_16_30.h"

#include "kernels_hash.cuh"
#include "kernels_ntt.cuh"
#include "kernels_ntt2.cuh"
#include "kernels_ntt3.cuh"
#include <array>
#include <functional>
#include <map>
#include <mutex>
#include <set>
#include <tuple>
#include <unordered_map>

// ------------------------------------------------------------------------------------------------
struct DMat {  // device matrix, Montgomery words; element (r, c) = d[r * rs + c * col_stride()]
    uint32_t* d = nullptr;
    uint64_t rows = 0;
    uint32_t cols = 0;
    uint32_t rs = 1;  // 1: column-major (the default everywhere); cols: row-major (FRI layer matrices)
    uint64_t col_stride() const { return rs == 1 ? rows : 1; }
};

struct bfgpu_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    int repr = BFGPU_REPR_CANONICAL;
    int input_space = BFGPU_MEM_HOST;
    std::string err;
    uint32_t* d_tw = nullptr;  // w^e, w of order 2^24, e < 2^23
    uint32_t log_blowup = 1, num_queries = 84, pow_bits = 16;
    uint64_t launches = 0;
    // optional per-phase device timing (bfgpu_profile_*): CUDA events recorded on ctx->stream
    bool profiling = false;
    struct Span { int phase; cudaEvent_t a, b; };
    std::vector<Span> spans;
    float phase_ms[BFGPU_NUM_PHASES] = {0};
    uint64_t phase_launches[BFGPU_NUM_PHASES] = {0};
    int cur_phase = -1;
    // cached radix-16 pass plans (twiddle tables) per (log_n, inverse)
    struct NttPass { unsigned p, g; ntt2::TWT* twA; ntt2::TWT* twB; };
    std::map<std::pair<unsigned, bool>, std::vector<NttPass>> plans;
    // cached coset scale vectors pw[h*n + k] = (shift_h)^k / n, keyed by (log_n, added_bits, shift)
    std::map<std::tuple<unsigned, unsigned, uint32_t>, uint32_t*> pw_cache;
    // size-exact caching allocator: every buffer is used on ctx->stream only, so a block freed by
    // dfree() can be handed out again immediately (stream order protects it).  Identical commits
    // reuse identical blocks; the CUDA async pool fragmented (a 4 GiB request carved out of the 8 GiB
    // block forced a fresh 8 GiB mapping every step).
    // host->device copies of a multi-matrix commit are issued up front on a second stream so that the copy of
    // matrix i+1 overlaps the LDE of matrix i (prestage_all / ingest)
    cudaStream_t copy_stream = nullptr;
    struct Prestaged { uint32_t* d; cudaEvent_t ready; };
    std::map<const uint32_t*, Prestaged> prestaged;
    std::multimap<size_t, void*> free_blocks;
    std::unordered_map<void*, size_t> live;
    size_t cached_bytes = 0;
    // pipelined host commit (commit_host_pipelined): columns per block, multiple of 8; 0 disables.
    // $BFGPU_PIPE_COLS overrides (experiments)
    // device-resident single-matrix commits: leaf sponge of block b concurrent with the NTT of block b+1 ($BFGPU_OVERLAP=1).
    // Measured at 2^22 x 256: 75.3 ms against 71.4 ms for the plain sequence (both kernels want the same two integer pipes;
    // the blocked LDE and the parked sponge states cost more than co-scheduling recovers) => off.
    // page-locked ring for small host->device parameter uploads (pointer tables, descriptors): the copy becomes truly asynchronous and
    // the host source may die right after the call (upload_small)
    uint8_t* ring = nullptr;
    size_t ring_size = 0, ring_pos = 0;
    uint32_t top_x1_max = 0;  // cluster tops: levels of at most this many nodes per CTA use the one-thread permutation ($BFGPU_TOP_X1_MAX); MEASURED: every setting > 0 is slower (hello 3.65 ms at 0, 3.74 at 1, 3.87 at 64): the four-lane chain is the shorter one
    bool top_cluster = true;  // tree tops of >= 256 digests on an 8-CTA cluster (hashk::k_compress_top_cluster); $BFGPU_TOP_CLUSTER=0: one CTA
    uint64_t x4_layer_max = 1u << 15;  // Merkle layers up to this many nodes use k_compress_layer_x4 ($BFGPU_X4_MAX)
    // opening points evaluated per pass over a matrix; one pass per point ($BFGPU_BARY_POINTS=1, 66 instead of 110 registers but the
    // matrix read twice) measured slower: open_eval 2.91 vs 2.51 ms at 2^22 rows
    uint32_t bary_points_per_pass = 2;
    bool fri_tail = true;  // small FRI rounds in one single-CTA launch (openk::k_fri_tail); $BFGPU_FRI_TAIL=0 disables
    bool overlap_device = false;
    int pipe_tail_splits = 1;  // $BFGPU_PIPE_SPLITS
    uint32_t pipe_cols = 64;  // 256-byte row segments per strided copy: 32 was 3 % slower end to end, 128 19 % (fewer stages)
    std::vector<std::pair<void*, uint64_t>> pinned_pool;  // page-locked cycle-record buffers parked between executions (tracegen.cuh)
    uint32_t* d_inv256 = nullptr;  // Montgomery inverses of 0..255 (tracegen.cuh, Jump chip)
    // peer receive buffers mapped through CUDA IPC (dist_commit.cuh), keyed by the 64-byte handle
    std::map<std::array<uint8_t, 64>, void*> ipc_open;
    // buffers whose IPC handle has been given to peers: their own pool (plain cudaMalloc, kept until the context dies, never
    // trimmed) so that a block a peer still has mapped is never returned to the driver behind its back
    std::multimap<size_t, void*> export_free;
    std::unordered_map<void*, size_t> export_live;
    // allocation scopes (AllocScope): blocks taken by an entry point that has not yet handed them to a returned object
    std::vector<std::vector<void*>*> scopes;
    // transcript options (bfgpu_set_transcript_option): the choices inside Plonky3 that cannot be confirmed offline (SURVEY.md P3 marks)
    uint32_t opt[BFGPU_NUM_OPTS] = {1, 0, 0};
    bool ntt_cfwd = false;  // contiguous forward pass through bulk copies (ntt3::k_cfwd, $BFGPU_NTT_CFWD=1).  MEASURED SLOWER than ntt2::k_pass
                            // at 2^22 x 256 (3.79 vs 3.61 ms: two CTA barriers per column and 512-thread CTAs cost more than the LDG.32
                            // address arithmetic saves), so it stays off; parity-tested behind the switch
    bool ntt_ingest = true;  // row-major input -> first inverse pass in one kernel (ntt3::k_ingest_pass); $BFGPU_NTT_INGEST=0: transpose, then pass
    bool ntt_tma = true;   // strided NTT passes through the TMA-fed 32-lane kernels (kernels_ntt3.cuh); $BFGPU_NTT_TMA=0: ntt2::k_pass
    std::set<int> ntt3_configured;  // (mode, G1) instantiations whose dynamic shared-memory limit has been raised on this device
    bool ntt_turn = true;  // last inverse pass fused with the first forward pass (k_pass TURN); $BFGPU_NTT_TURN=0 runs them as two launches
    bool ntt_dual = true;  // coset scaling on load in the first forward pass (k_pass DUAL) instead of the inverse-pass epilogue ($BFGPU_NTT_DUAL=0)
    bool dist_fused_scatter = true;  // sharded commitment: the last forward NTT pass stores straight into the peers' row shards
                                     // (ntt3::k_cfwd with CfwdArgs::scatter) instead of a k_scatter_rows pass over the finished block; $BFGPU_DIST_FUSED_SCATTER=0
    uint32_t dist_min_chunk = 32;  // dist_commit.cuh: smallest LDE / scatter block in columns ($BFGPU_DIST_MIN_CHUNK)
    unsigned dist_fri_gather_log = 20;  // dist_prove.cuh: global FRI length below which the sharded prover gathers ($BFGPU_DIST_FRI_GATHER_LOG)
    // test hook (bfgpu_debug_fail_alloc): the n-th dalloc from now fails with BFGPU_ERR_OOM
    int64_t fail_alloc_in = -1;
    // page-locked staging buffer of bfgpu_verify_batch (plan records and query words up, result bits down), grown on demand
    uint8_t* vstage = nullptr;
    size_t vstage_size = 0;
};

struct bfgpu_tree {
    bfgpu_ctx* ctx = nullptr;
    std::vector<DMat> mats;  // input order
    bool owns_mats = false;
    std::vector<uint32_t*> layers;  // layers[l]: layer_len[l] digests of 8 words
    std::vector<uint64_t> layer_len;
    unsigned log_max = 0;
};

struct bfgpu_pcs_data {
    bfgpu_ctx* ctx = nullptr;
    std::vector<DMat> ldes;  // bit-reversed rows
    bfgpu_tree* tree = nullptr;
};

static std::mutex g_ctx_mutex;
static std::set<bfgpu_ctx*> g_live_ctx;  // contexts that may still receive parked buffers

static int32_t fail(bfgpu_ctx* ctx, int32_t code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    return code;
}

#define CU(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess)                                                                            \
            return fail(ctx, e_ == cudaErrorMemoryAllocation ? BFGPU_ERR_OOM : BFGPU_ERR_CUDA, "%s: %s (%s:%d)", #call, \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                                      \
    } while (0)
#define TRY(call)                   \
    do {                            \
        int32_t rc_ = (call);       \
        if (rc_ != BFGPU_OK) return rc_; \
    } while (0)
#define LAUNCHED(ctx)                                                        \
    do {                                                                     \
        (ctx)->launches++;                                                   \
        if ((ctx)->cur_phase >= 0) (ctx)->phase_launches[(ctx)->cur_phase]++; \
    } while (0)

// RAII phase marker: when profiling is on, brackets the enclosed launches with two events
struct Phase {
    bfgpu_ctx* ctx;
    int prev;
    size_t idx = (size_t)-1;
    Phase(bfgpu_ctx* c, int phase) : ctx(c), prev(c->cur_phase) {
        c->cur_phase = phase;
        if (c->profiling) {
            bfgpu_ctx::Span sp{phase, nullptr, nullptr};
            cudaEventCreate(&sp.a);
            cudaEventCreate(&sp.b);
            cudaEventRecord(sp.a, c->stream);
            idx = c->spans.size();
            c->spans.push_back(sp);
        }
    }
    ~Phase() {
        if (idx != (size_t)-1) cudaEventRecord(ctx->spans[idx].b, ctx->stream);
        ctx->cur_phase = prev;
    }
};

static inline bool is_pow2(uint64_t x) { return x && !(x & (x - 1)); }
static inline unsigned ilog2(uint64_t x) {
    unsigned l = 0;
    while ((1ull << l) < x) l++;
    return l;
}

static void trim_cache(bfgpu_ctx* ctx) {
    if (ctx->free_blocks.empty()) return;
    cudaStreamSynchronize(ctx->stream);
    for (auto& kv : ctx->free_blocks) cudaFree(kv.second);
    ctx->free_blocks.clear();
    ctx->cached_bytes = 0;
}
static int32_t dalloc(bfgpu_ctx* ctx, void** p, size_t bytes) {
    *p = nullptr;
    // every compute entry point allocates before it launches: make the context's device current here, so that a process
    // holding contexts on several devices (or calling from a fresh thread) launches on the right one
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess || cur != ctx->device) CU(cudaSetDevice(ctx->device));
    bytes = (std::max<size_t>(bytes, 4) + 255) & ~(size_t)255;
    if (ctx->fail_alloc_in >= 0 && ctx->fail_alloc_in-- == 0) return fail(ctx, BFGPU_ERR_OOM, "injected allocation failure (%zu bytes)", bytes);
    auto it = ctx->free_blocks.find(bytes);
    if (it != ctx->free_blocks.end()) {
        *p = it->second;
        ctx->free_blocks.erase(it);
        ctx->cached_bytes -= bytes;
    } else {
        cudaError_t e = cudaMalloc(p, bytes);
        if (e == cudaErrorMemoryAllocation) {  // give cached blocks back to the driver and retry once
            cudaGetLastError();
            trim_cache(ctx);
            e = cudaMalloc(p, bytes);
        }
        if (e != cudaSuccess) {
            cudaGetLastError();
            *p = nullptr;
            return fail(ctx, e == cudaErrorMemoryAllocation ? BFGPU_ERR_OOM : BFGPU_ERR_CUDA, "cudaMalloc(%zu bytes): %s", bytes, cudaGetErrorString(e));
        }
    }
    ctx->live[*p] = bytes;
    if (!ctx->scopes.empty()) ctx->scopes.back()->push_back(*p);
    return BFGPU_OK;
}
static void dfree(bfgpu_ctx* ctx, void* p) {
    if (!p) return;
    auto it = ctx->live.find(p);
    if (it == ctx->live.end()) return;
    size_t bytes = it->second;
    ctx->live.erase(it);
    ctx->free_blocks.emplace(bytes, p);
    ctx->cached_bytes += bytes;
}

// Small host->device upload through the context's page-locked ring.  cudaMemcpyAsync from pageable memory blocks the host
// until the driver has staged the bytes (~8 us each, dozens per proof); from the ring it is a plain enqueue.
static int32_t upload_small(bfgpu_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (bytes == 0) return BFGPU_OK;
    if (!ctx->ring) {
        ctx->ring_size = 8u << 20;
        if (cudaHostAlloc((void**)&ctx->ring, ctx->ring_size, cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            ctx->ring = nullptr;
            ctx->ring_size = 0;
        }
    }
    const size_t need = (bytes + 63) & ~(size_t)63;
    if (!ctx->ring || need > ctx->ring_size / 4) {
        CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
        return BFGPU_OK;
    }
    if (ctx->ring_pos + need > ctx->ring_size) {
        CU(cudaStreamSynchronize(ctx->stream));  // every copy out of the ring so far has completed: start over
        ctx->ring_pos = 0;
    }
    memcpy(ctx->ring + ctx->ring_pos, src, bytes);
    CU(cudaMemcpyAsync(dst, ctx->ring + ctx->ring_pos, bytes, cudaMemcpyHostToDevice, ctx->stream));
    ctx->ring_pos += need;
    return BFGPU_OK;
}

// Scratch device buffers of one entry point: returned to the block cache on every exit path.
struct Scratch {
    bfgpu_ctx* ctx;
    std::vector<void*> bufs;
    explicit Scratch(bfgpu_ctx* c) : ctx(c) {}
    int32_t alloc(void** p, size_t bytes) {
        int32_t rc = dalloc(ctx, p, bytes);
        if (rc == BFGPU_OK) bufs.push_back(*p);
        return rc;
    }
    ~Scratch() {
        for (void* p : bufs) dfree(ctx, p);
    }
};

static void prestage_clear(bfgpu_ctx* ctx);
// Every compute entry point opens one: CU()/TRY() return early from anywhere, and whatever the call had taken from dalloc() by
// then and not yet released goes back to the block cache when the scope closes without ok() — the objects an entry point returns
// are only handed out after ok().  Nested scopes (bfgpu_pcs_open inside bfgpu_machine_open) pass their blocks up on success.
struct AllocScope {
    bfgpu_ctx* ctx;
    std::vector<void*> taken;
    bool success = false;
    explicit AllocScope(bfgpu_ctx* c) : ctx(c) {
        if (ctx) ctx->scopes.push_back(&taken);
    }
    int32_t ok(int32_t rc = BFGPU_OK) {
        success = rc == BFGPU_OK;
        return rc;
    }
    ~AllocScope() {
        if (!ctx) return;
        ctx->scopes.pop_back();
        if (success) {
            if (!ctx->scopes.empty()) {
                auto* up = ctx->scopes.back();
                for (void* p : taken)
                    if (ctx->live.count(p)) up->push_back(p);
            }
            return;
        }
        // kernels of the failed call may still be running on either stream: drain before the blocks can be handed out again
        if (ctx->stream) cudaStreamSynchronize(ctx->stream);
        if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
        cudaGetLastError();
        prestage_clear(ctx);
        for (void* p : taken) dfree(ctx, p);  // dfree ignores blocks that were already released
    }
};

// ---- context ----------------------------------------------------------------------------------
extern "C" int32_t bfgpu_ctx_create(int device, bfgpu_ctx** out) {
    if (!out) return BFGPU_ERR_INVALID;
    *out = nullptr;
    bfgpu_ctx* ctx = new bfgpu_ctx();
    ctx->device = device;
    *out = ctx;  // returned even on failure so the caller can read the message
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(ctx, BFGPU_ERR_CUDA, "no CUDA device available (%s); this backend has no CPU fallback", cudaGetErrorString(e));
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    if (const char* e = getenv("BFGPU_PIPE_COLS")) ctx->pipe_cols = (uint32_t)atoi(e) / 8 * 8;
    if (const char* e = getenv("BFGPU_OVERLAP")) ctx->overlap_device = atoi(e) != 0;
    if (const char* e = getenv("BFGPU_FRI_TAIL")) ctx->fri_tail = atoi(e) != 0;
    if (const char* e = getenv("BFGPU_BARY_POINTS")) ctx->bary_points_per_pass = atoi(e) == 1 ? 1 : 2;
    if (const char* e = getenv("BFGPU_X4_MAX")) ctx->x4_layer_max = strtoull(e, nullptr, 10);
    if (const char* e = getenv("BFGPU_PIPE_SPLITS")) ctx->pipe_tail_splits = atoi(e);
    if (const char* e = getenv("BFGPU_NTT_DUAL")) ctx->ntt_dual = atoi(e) != 0;
    if (const char* e = getenv("BFGPU_NTT_TURN")) ctx->ntt_turn = atoi(e) != 0;
    if (const char* e = getenv("BFGPU_NTT_TMA")) ctx->ntt_tma = atoi(e) != 0;
    if (const char* e = getenv("BFGPU_NTT_INGEST")) ctx->ntt_ingest = atoi(e) != 0;
    if (const char* e = getenv("BFGPU_NTT_CFWD")) ctx->ntt_cfwd = atoi(e) != 0;
    if (const char* e = getenv("BFGPU_TOP_CLUSTER")) ctx->top_cluster = atoi(e) != 0;
    if (const char* e = getenv("BFGPU_TOP_X1_MAX")) ctx->top_x1_max = (uint32_t)atoi(e);
    if (const char* e = getenv("BFGPU_DIST_FUSED_SCATTER")) ctx->dist_fused_scatter = atoi(e) != 0;
    if (const char* e = getenv("BFGPU_DIST_MIN_CHUNK")) ctx->dist_min_chunk = (uint32_t)std::max(8, atoi(e)) / 8 * 8;
    if (const char* e = getenv("BFGPU_DIST_FRI_GATHER_LOG")) ctx->dist_fri_gather_log = (unsigned)std::min(24, std::max(4, atoi(e)));
    if (const char* q = getenv("FRI_QUERIES")) ctx->num_queries = (uint32_t)atoi(q);  // kb31_poseidon2.rs:59-62

    // Poseidon2 constant bank (kb31_poseidon2.rs:35-50): internal constants = column 0 of table rows
    // 4..16; external initial = rows 0..3; external terminal = rows 17..20 (rows 4..7 after the drain).
    p2::Consts h;
    memset(&h, 0, sizeof h);
    for (int r = 0; r < 4; r++)
        for (int i = 0; i < 16; i++) {
            h.ext[r][i] = kb::to_mont(BFGPU_RC_16_30[r][i]);
            h.ext[4 + r][i] = kb::to_mont(BFGPU_RC_16_30[17 + r][i]);
        }
    for (int r = 0; r < 13; r++) h.internal[r] = kb::to_mont(BFGPU_RC_16_30[4 + r][0]);
    for (int r = 0; r < 8; r++)
        for (int i = 0; i < 16; i++) h.ext_s[r][i] = h.ext[r][i] - kb::P;
    for (int r = 0; r < 13; r++) h.internal_s[r] = h.internal[r] - kb::P;
    {  // V = [-2, 1, 2, 1/2, 3, 4, -1/2, -3, -4, 1/2^8, 1/8, 1/2^24, -1/2^8, -1/8, -1/16, -1/2^24]
        auto frac = [](int sign, unsigned k) {
            uint32_t v = kb::ONE;
            for (unsigned i = 0; i < k; i++) v = kb::halve(v);
            return sign < 0 ? kb::neg(v) : v;
        };
        auto small = [](int v) { return v >= 0 ? kb::to_mont((uint32_t)v) : kb::neg(kb::to_mont((uint32_t)(-v))); };
        uint32_t d[16] = {small(-2), small(1), small(2), frac(1, 1), small(3), small(4), frac(-1, 1), small(-3),
                          small(-4), frac(1, 8), frac(1, 3), frac(1, 24), frac(-1, 8), frac(-1, 3), frac(-1, 4), frac(-1, 24)};
        memcpy(h.diag, d, sizeof d);
        for (int i = 0; i < 16; i++) {
            h.diag_w[i] = kb::from_mont(d[i]);
            h.diag_wp[i] = (uint32_t)(((uint64_t)h.diag_w[i] << 32) / kb::P);
        }
    }
    CU(cudaMemcpyToSymbolAsync(p2::c_p2, &h, sizeof h, 0, cudaMemcpyHostToDevice, ctx->stream));

    // twiddle table
    CU(cudaMalloc(&ctx->d_tw, sizeof(uint32_t) << (nttk::TW_LOG - 1)));
    nttk::k_build_twiddles<<<(1u << (nttk::TW_LOG - 1)) / 256, 256, 0, ctx->stream>>>(ctx->d_tw, kb::two_adic_generator(nttk::TW_LOG));
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    {  // 16th roots of unity (canonical) with Shoup quotients, forward and inverse
        ntt2::Tw h16[2][8];
        uint32_t w16 = kb::two_adic_generator(4), w16i = kb::inv(w16);
        for (int j = 0; j < 8; j++) {
            uint32_t f = kb::from_mont(kb::pow(w16, j)), b = kb::from_mont(kb::pow(w16i, j));
            h16[0][j] = {f, (uint32_t)(((uint64_t)f << 32) / kb::P)};
            h16[1][j] = {b, (uint32_t)(((uint64_t)b << 32) / kb::P)};
        }
        CU(cudaMemcpyToSymbolAsync(ntt2::c_w16, h16, sizeof h16, 0, cudaMemcpyHostToDevice, ctx->stream));
    }
    CU(cudaFuncSetAttribute(nttk::k_ntt_pass<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 << (nttk::GMAX + nttk::LANES_LOG)));
    CU(cudaFuncSetAttribute(nttk::k_ntt_pass<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 << (nttk::GMAX + nttk::LANES_LOG)));
    CU(cudaStreamSynchronize(ctx->stream));
    {
        std::lock_guard<std::mutex> g(g_ctx_mutex);
        g_live_ctx.insert(ctx);
    }
    return BFGPU_OK;
}

extern "C" void bfgpu_ctx_destroy(bfgpu_ctx* ctx) {
    if (!ctx) return;
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->d_tw) cudaFree(ctx->d_tw);
    if (ctx->d_inv256) cudaFree(ctx->d_inv256);
    if (ctx->ring) cudaFreeHost(ctx->ring);
    if (ctx->vstage) cudaFreeHost(ctx->vstage);
    {
        std::lock_guard<std::mutex> g(g_ctx_mutex);
        g_live_ctx.erase(ctx);
        for (auto& b : ctx->pinned_pool) cudaFreeHost(b.first);
        ctx->pinned_pool.clear();
    }
    for (auto& kv : ctx->ipc_open) cudaIpcCloseMemHandle(kv.second);
    for (auto& kv : ctx->export_free) cudaFree(kv.second);
    for (auto& kv : ctx->export_live) cudaFree(kv.first);
    trim_cache(ctx);
    for (auto& kv : ctx->live) cudaFree(kv.first);
    for (auto& kv : ctx->pw_cache) cudaFree(kv.second);
    for (auto& kv : ctx->plans)
        for (auto& ps : kv.second) {
            if (ps.twA) cudaFree(ps.twA);
            if (ps.twB) cudaFree(ps.twB);
        }
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    delete ctx;
}
extern "C" const char* bfgpu_last_error(const bfgpu_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
extern "C" int32_t bfgpu_set_repr(bfgpu_ctx* ctx, int repr) {
    if (!ctx || (repr != BFGPU_REPR_CANONICAL && repr != BFGPU_REPR_MONTY)) return fail(ctx, BFGPU_ERR_INVALID, "bad repr");
    ctx->repr = repr;
    return BFGPU_OK;
}
extern "C" int32_t bfgpu_set_input_space(bfgpu_ctx* ctx, int s) {
    if (!ctx || (s != BFGPU_MEM_HOST && s != BFGPU_MEM_DEVICE)) return fail(ctx, BFGPU_ERR_INVALID, "bad memory space");
    ctx->input_space = s;
    return BFGPU_OK;
}
extern "C" int32_t bfgpu_set_stream(bfgpu_ctx* ctx, void* s) {
    if (!ctx) return BFGPU_ERR_INVALID;
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (s) {
        ctx->stream = (cudaStream_t)s;
        ctx->own_stream = false;
    } else {
        CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->own_stream = true;
    }
    return BFGPU_OK;
}
extern "C" int32_t bfgpu_synchronize(bfgpu_ctx* ctx) {
    if (!ctx) return BFGPU_ERR_INVALID;
    CU(cudaStreamSynchronize(ctx->stream));
    return BFGPU_OK;
}
extern "C" int32_t bfgpu_set_fri_params(bfgpu_ctx* ctx, uint32_t log_blowup, uint32_t num_queries, uint32_t pow_bits) {
    if (!ctx || log_blowup == 0 || log_blowup > 4) return fail(ctx, BFGPU_ERR_INVALID, "bad FRI parameters");
    ctx->log_blowup = log_blowup;
    ctx->num_queries = num_queries;
    ctx->pow_bits = pow_bits;
    return BFGPU_OK;
}
extern "C" int32_t bfgpu_set_transcript_option(bfgpu_ctx* ctx, int32_t option, uint32_t value) {
    if (!ctx || option < 0 || option >= BFGPU_NUM_OPTS || value > 1) return fail(ctx, BFGPU_ERR_INVALID, "bad transcript option %d = %u", option, value);
    ctx->opt[option] = value;
    return BFGPU_OK;
}
extern "C" uint64_t bfgpu_launch_count(const bfgpu_ctx* ctx) { return ctx ? ctx->launches : 0; }
extern "C" uint64_t bfgpu_debug_live_blocks(const bfgpu_ctx* ctx) { return ctx ? ctx->live.size() : 0; }
extern "C" int32_t bfgpu_debug_fail_alloc(bfgpu_ctx* ctx, int64_t nth) {
    if (!ctx) return BFGPU_ERR_INVALID;
    ctx->fail_alloc_in = nth;
    return BFGPU_OK;
}

// exported (IPC-shared) blocks: see bfgpu_ctx::export_free
static int32_t dalloc_export(bfgpu_ctx* ctx, void** p, size_t bytes) {
    *p = nullptr;
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess || cur != ctx->device) CU(cudaSetDevice(ctx->device));
    bytes = (std::max<size_t>(bytes, 4) + 255) & ~(size_t)255;
    auto it = ctx->export_free.find(bytes);
    if (it != ctx->export_free.end()) {
        *p = it->second;
        ctx->export_free.erase(it);
    } else {
        cudaError_t e = cudaMalloc(p, bytes);
        if (e == cudaErrorMemoryAllocation) {
            cudaGetLastError();
            trim_cache(ctx);
            e = cudaMalloc(p, bytes);
        }
        if (e != cudaSuccess) {
            cudaGetLastError();
            *p = nullptr;
            return fail(ctx, e == cudaErrorMemoryAllocation ? BFGPU_ERR_OOM : BFGPU_ERR_CUDA, "cudaMalloc(%zu bytes, exported): %s", bytes, cudaGetErrorString(e));
        }
    }
    ctx->export_live[*p] = bytes;
    return BFGPU_OK;
}
static void dfree_export(bfgpu_ctx* ctx, void* p) {
    auto it = ctx->export_live.find(p);
    if (it == ctx->export_live.end()) return;
    ctx->export_free.emplace(it->second, p);
    ctx->export_live.erase(it);
}

extern "C" int32_t bfgpu_host_alloc(bfgpu_ctx* ctx, uint64_t bytes, void** out) {
    if (!ctx || !out) return BFGPU_ERR_INVALID;
    CU(cudaHostAlloc(out, bytes ? bytes : 4, cudaHostAllocDefault));
    return BFGPU_OK;
}
extern "C" void bfgpu_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

// ---- measurement hooks -------------------------------------------------------------------------------
extern "C" int32_t bfgpu_profile_enable(bfgpu_ctx* ctx, int on) {
    if (!ctx) return BFGPU_ERR_INVALID;
    CU(cudaStreamSynchronize(ctx->stream));
    for (auto& sp : ctx->spans) {
        cudaEventDestroy(sp.a);
        cudaEventDestroy(sp.b);
    }
    ctx->spans.clear();
    ctx->profiling = on != 0;
    if (on)
        for (int i = 0; i < BFGPU_NUM_PHASES; i++) {
            ctx->phase_ms[i] = 0;
            ctx->phase_launches[i] = 0;
        }
    return BFGPU_OK;
}
extern "C" int32_t bfgpu_profile_read(bfgpu_ctx* ctx, float ms[BFGPU_NUM_PHASES], uint64_t launches[BFGPU_NUM_PHASES]) {
    if (!ctx || !ms) return BFGPU_ERR_INVALID;
    CU(cudaStreamSynchronize(ctx->stream));
    for (auto& sp : ctx->spans) {
        float t = 0;
        if (cudaEventElapsedTime(&t, sp.a, sp.b) == cudaSuccess) ctx->phase_ms[sp.phase] += t;
        cudaEventDestroy(sp.a);
        cudaEventDestroy(sp.b);
    }
    ctx->spans.clear();
    for (int i = 0; i < BFGPU_NUM_PHASES; i++) {
        ms[i] = ctx->phase_ms[i];
        if (launches) launches[i] = ctx->phase_launches[i];
    }
    return BFGPU_OK;
}

// Integer-pipe probe: 8 independent chains per thread, each iteration 1 IMAD + 1 IADD3 + 1 LOP3 per
// chain (the mix a Montgomery butterfly / Poseidon2 round issues), no memory traffic.
__global__ void __launch_bounds__(256) k_int32_probe(uint32_t* out, uint32_t iters, uint32_t seed) {
    uint32_t a[8];
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = seed + threadIdx.x * 8 + k;
    uint32_t m = seed | 1u, c = seed ^ 0x9e3779b9u;
    for (uint32_t i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            a[k] = a[k] * m + c;        // IMAD
            a[k] = a[k] + (a[k] >> 7);  // SHF + IADD
            a[k] ^= c;                  // LOP3
        }
    }
    uint32_t r = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) r ^= a[k];
    if (r == 0x12345678u) out[0] = r;  // practically never; keeps the chains alive
}
static int32_t int32_peak_probe_impl(bfgpu_ctx* ctx, double* giops);
extern "C" int32_t bfgpu_int32_peak_probe(bfgpu_ctx* ctx, double* giops) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(int32_peak_probe_impl(ctx, giops));
}
static int32_t int32_peak_probe_impl(bfgpu_ctx* ctx, double* giops) {
    if (!ctx || !giops) return BFGPU_ERR_INVALID;
    uint32_t* d = nullptr;
    TRY(dalloc(ctx, (void**)&d, 4));
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    const uint32_t iters = 4096, blocks = 148 * 8;
    k_int32_probe<<<blocks, 256, 0, ctx->stream>>>(d, 64, 12345u);  // warm-up
    CU(cudaEventRecord(a, ctx->stream));
    k_int32_probe<<<blocks, 256, 0, ctx->stream>>>(d, iters, 12345u);
    CU(cudaEventRecord(b, ctx->stream));
    ctx->launches += 2;
    CU(cudaEventSynchronize(b));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    dfree(ctx, d);
    // 4 integer instructions per chain-iteration (IMAD, SHF, IADD, LOP3)
    *giops = (double)blocks * 256 * iters * 8 * 4 / (ms * 1e-3) / 1e9;
    return BFGPU_OK;
}

// ---- staging helpers ----------------------------------------------------------------------------
// Bring a caller matrix (row-major, host or device, caller representation) into a fresh
// column-major Montgomery device matrix, optionally gathering rows in bit-reversed order.
// Issue the host->device copies of all caller matrices on the copy stream (ordered after everything already
// enqueued on the compute stream, because the staging blocks come from the single-stream block cache).
static int32_t prestage_all(bfgpu_ctx* ctx, const bfgpu_mat* mats, int32_t n) {
    if (ctx->input_space != BFGPU_MEM_HOST || n <= 1) return BFGPU_OK;
    Phase ph(ctx, BFGPU_PHASE_H2D);
    cudaEvent_t fence;
    CU(cudaEventCreateWithFlags(&fence, cudaEventDisableTiming));
    CU(cudaEventRecord(fence, ctx->stream));
    CU(cudaStreamWaitEvent(ctx->copy_stream, fence, 0));
    cudaEventDestroy(fence);
    for (int32_t i = 0; i < n; i++) {
        size_t bytes = (size_t)mats[i].rows * mats[i].cols * 4;
        if (!bytes || !mats[i].data || ctx->prestaged.count(mats[i].data)) continue;
        bfgpu_ctx::Prestaged ps{nullptr, nullptr};
        TRY(dalloc(ctx, (void**)&ps.d, bytes));
        CU(cudaMemcpyAsync(ps.d, mats[i].data, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
        CU(cudaEventCreateWithFlags(&ps.ready, cudaEventDisableTiming));
        CU(cudaEventRecord(ps.ready, ctx->copy_stream));
        ctx->prestaged[mats[i].data] = ps;
    }
    return BFGPU_OK;
}

// drop copies that were issued but never consumed (error paths)
static void prestage_clear(bfgpu_ctx* ctx) {
    if (ctx->prestaged.empty()) return;
    cudaStreamSynchronize(ctx->copy_stream);
    for (auto& kv : ctx->prestaged) {
        cudaEventDestroy(kv.second.ready);
        dfree(ctx, kv.second.d);
    }
    ctx->prestaged.clear();
}

// Transpose fused with the first inverse NTT pass (defined with the NTT orchestration below); *done = false: not applicable, nothing launched
static int32_t ingest_first_pass(bfgpu_ctx* ctx, const uint32_t* src, uint64_t rows, uint32_t cols, uint32_t* dst, uint64_t pitch, bool* done);

// row-major device words in the caller's representation -> column-major Montgomery words at dst
// first_pass_done != null (bit-reversed ingest feeding an inverse transform): the first inverse pass may be executed on the way
// (*first_pass_done = true), in which case the caller runs the transform with skip_first.
static int32_t ingest_device(bfgpu_ctx* ctx, const uint32_t* src, uint64_t rows, uint32_t cols, bool bitrev, uint32_t* dst, uint64_t src_pitch = 0,
                             bool* first_pass_done = nullptr) {
    Phase ph(ctx, BFGPU_PHASE_INGEST);
    const uint64_t pitch = src_pitch ? src_pitch : cols;
    if (first_pass_done) {
        *first_pass_done = false;
        if (bitrev) TRY(ingest_first_pass(ctx, src, rows, cols, dst, pitch, first_pass_done));
        if (*first_pass_done) return BFGPU_OK;
    }
    if (rows >= 128 && rows % 128 == 0 && cols % 4 == 0 && pitch % 4 == 0 && ((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 15) == 0) {
        dim3 grid((unsigned)(rows / 128), (unsigned)((cols + 31) / 32));
        nttk::k_ingest_wide<<<grid, 256, 0, ctx->stream>>>(src, dst, rows, cols, ilog2(rows), bitrev ? 1 : 0, ctx->repr == BFGPU_REPR_CANONICAL, pitch);
    } else {
        dim3 grid((unsigned)((rows + 31) / 32), (unsigned)((cols + 31) / 32)), block(32, 8);
        nttk::k_ingest<<<grid, block, 0, ctx->stream>>>(src, dst, rows, cols, ilog2(rows), bitrev ? 1 : 0, ctx->repr == BFGPU_REPR_CANONICAL, pitch);
    }
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    return BFGPU_OK;
}

static int32_t ingest(bfgpu_ctx* ctx, const bfgpu_mat& m, bool bitrev, DMat* out, bool* first_pass_done = nullptr) {
    if (first_pass_done) *first_pass_done = false;
    out->rows = m.rows;
    out->cols = (uint32_t)m.cols;
    size_t bytes = (size_t)m.rows * m.cols * 4;
    TRY(dalloc(ctx, (void**)&out->d, bytes));
    if (bytes == 0) return BFGPU_OK;
    const uint32_t* src = m.data;
    uint32_t* staged = nullptr;
    if (ctx->input_space == BFGPU_MEM_HOST) {
        auto it = ctx->prestaged.find(m.data);
        if (it != ctx->prestaged.end()) {
            staged = it->second.d;
            CU(cudaStreamWaitEvent(ctx->stream, it->second.ready, 0));
            cudaEventDestroy(it->second.ready);
            ctx->prestaged.erase(it);
        } else {
            Phase ph(ctx, BFGPU_PHASE_H2D);
            TRY(dalloc(ctx, (void**)&staged, bytes));
            CU(cudaMemcpyAsync(staged, m.data, bytes, cudaMemcpyHostToDevice, ctx->stream));
        }
        src = staged;
    }
    int32_t rc = ingest_device(ctx, src, m.rows, (uint32_t)m.cols, bitrev, out->d, 0, first_pass_done);
    dfree(ctx, staged);
    return rc;
}

// column-major Montgomery device matrix -> caller's row-major host buffer
static int32_t egress(bfgpu_ctx* ctx, const DMat& m, bool bitrev, uint32_t* host_out) {
    size_t bytes = (size_t)m.rows * m.cols * 4;
    if (bytes == 0) return BFGPU_OK;
    uint32_t* tmp = nullptr;
    TRY(dalloc(ctx, (void**)&tmp, bytes));
    dim3 grid((unsigned)((m.rows + 31) / 32), (unsigned)((m.cols + 31) / 32)), block(32, 8);
    nttk::k_egress<<<grid, block, 0, ctx->stream>>>(m.d, tmp, m.rows, m.cols, ilog2(m.rows), bitrev ? 1 : 0, ctx->repr == BFGPU_REPR_CANONICAL);
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(host_out, tmp, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    dfree(ctx, tmp);
    return BFGPU_OK;
}

static int32_t check_mat(bfgpu_ctx* ctx, const bfgpu_mat* m, bool need_pow2) {
    if (!m) return fail(ctx, BFGPU_ERR_INVALID, "null matrix");
    if (m->rows == 0 || m->cols == 0) return fail(ctx, BFGPU_ERR_INVALID, "empty matrix (%llu x %llu)", (unsigned long long)m->rows, (unsigned long long)m->cols);
    if (!m->data) return fail(ctx, BFGPU_ERR_INVALID, "null matrix data");
    if (need_pow2 && !is_pow2(m->rows)) return fail(ctx, BFGPU_ERR_INVALID, "matrix height %llu is not a power of two", (unsigned long long)m->rows);
    if (m->rows > (1ull << 31) || m->cols > (1ull << 24)) return fail(ctx, BFGPU_ERR_INVALID, "matrix too large");
    return BFGPU_OK;
}

// ---- NTT orchestration ----------------------------------------------------------------------------
// Fallback for short columns (< 2^12): shared-memory radix-2 passes (kernels_ntt.cuh).
template <bool INVERSE>
static int32_t run_ntt_small(bfgpu_ctx* ctx, uint32_t* data, uint64_t col_stride, unsigned log_n, uint32_t ncols) {
    unsigned npass = (log_n + nttk::GMAX - 1) / nttk::GMAX;
    unsigned base = log_n / npass, extra = log_n % npass;
    unsigned g[8], p[8];
    unsigned acc = 0;
    for (unsigned i = 0; i < npass; i++) {  // low passes take the larger share, so every p > 0 is >= LANES_LOG
        g[i] = base + (i < extra ? 1 : 0);
        p[i] = acc;
        acc += g[i];
    }
    for (unsigned s = 0; s < npass; s++) {
        unsigned i = INVERSE ? s : npass - 1 - s;  // inverse DIT: low bits first; forward DIF: high bits first
        unsigned lanes_log = p[i] == 0 ? std::min<unsigned>(nttk::LANES_LOG, log_n - g[i]) : nttk::LANES_LOG;
        if (p[i] != 0 && p[i] < nttk::LANES_LOG) return fail(ctx, BFGPU_ERR_STATE, "internal: bad NTT pass plan");
        dim3 grid(1u << (log_n - g[i] - lanes_log), ncols);
        size_t smem = (size_t)4 << (g[i] + lanes_log);
        nttk::k_ntt_pass<INVERSE><<<grid, nttk::NTT_THREADS, smem, ctx->stream>>>(data, col_stride, log_n, p[i], g[i], lanes_log, ctx->d_tw);
        LAUNCHED(ctx);
        CU(cudaGetLastError());
    }
    return BFGPU_OK;
}

// Pass plan + twiddle tables of the radix-16 kernels for columns of 2^log_n points (cached).
static int32_t get_plan(bfgpu_ctx* ctx, unsigned log_n, bool inverse, const std::vector<bfgpu_ctx::NttPass>** out) {
    auto key = std::make_pair(log_n, inverse);
    auto it = ctx->plans.find(key);
    if (it == ctx->plans.end()) {
        std::vector<bfgpu_ctx::NttPass> passes;
        unsigned npass = (log_n + 7) / 8, base = log_n / npass, extra = log_n % npass, acc = 0;
        uint32_t wmax = kb::two_adic_generator(kb::TWO_ADICITY);
        for (unsigned i = 0; i < npass; i++) {
            bfgpu_ctx::NttPass ps{acc, base + (i < extra ? 1 : 0), nullptr, nullptr};
            acc += ps.g;
            unsigned G1 = ps.g - 4;
            if (G1 > 0) {
                uint32_t nq = (1u << G1) - 1, M = 1u << (ps.p + 4);
                CU(cudaMalloc(&ps.twA, (size_t)nq * M * sizeof(ntt2::TWT)));
                uint64_t total = (uint64_t)nq * M;
                ntt2::k_build_tw<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(ps.twA, nq, M, ps.p + ps.g, inverse, wmax);
                LAUNCHED(ctx);
            }
            if (ps.p > 0) {
                uint32_t nq = 15, M = 1u << ps.p;
                CU(cudaMalloc(&ps.twB, (size_t)nq * M * sizeof(ntt2::TWT)));
                uint64_t total = (uint64_t)nq * M;
                ntt2::k_build_tw<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(ps.twB, nq, M, ps.p + 4, inverse, wmax);
                LAUNCHED(ctx);
            }
            CU(cudaGetLastError());
            passes.push_back(ps);
        }
        it = ctx->plans.emplace(key, std::move(passes)).first;
    }
    *out = &it->second;
    return BFGPU_OK;
}


// ---- TMA-fed strided passes (kernels_ntt3.cuh) -------------------------------------------------------------------------------
// cuTensorMapEncodeTiled comes from the driver through the runtime (no link-time dependency on libcuda).
typedef CUresult (*tmap_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                   const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static tmap_encode_fn tmap_encoder() {
    static tmap_encode_fn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) f = nullptr;
        return (tmap_encode_fn)f;
    }();
    return fn;
}
static bool ntt3_usable(bfgpu_ctx* ctx, const bfgpu_ctx::NttPass& ps) { return ctx->ntt_tma && ps.p >= 5 && ps.g >= 5 && ps.g <= 8 && tmap_encoder() != nullptr; }

template <int MODE, int G1>
static int32_t launch3(bfgpu_ctx* ctx, const CUtensorMap& tm_in, const CUtensorMap& tm_out, const ntt3::PassArgs& a, dim3 grid) {
    const int key = MODE * 8 + G1;
    if (!ctx->ntt3_configured.count(key)) {
        CU(cudaFuncSetAttribute(ntt3::k_pass3<MODE, G1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ntt3::smem_bytes(MODE, G1)));
        ctx->ntt3_configured.insert(key);
    }
    ntt3::k_pass3<MODE, G1><<<grid, 1u << (G1 + 5), ntt3::smem_bytes(MODE, G1), ctx->stream>>>(tm_in, tm_out, a);
    return BFGPU_OK;
}
template <int MODE>
static int32_t launch3_g(bfgpu_ctx* ctx, unsigned g, const CUtensorMap& tm_in, const CUtensorMap& tm_out, const ntt3::PassArgs& a, dim3 grid) {
    switch (g - 4) {
        case 1: return launch3<MODE, 1>(ctx, tm_in, tm_out, a, grid);
        case 2: return launch3<MODE, 2>(ctx, tm_in, tm_out, a, grid);
        case 3: return launch3<MODE, 3>(ctx, tm_in, tm_out, a, grid);
        case 4: return launch3<MODE, 4>(ctx, tm_in, tm_out, a, grid);
    }
    return fail(ctx, BFGPU_ERR_STATE, "internal: bad pass size %u", g);
}
// 4-d view [column][hi][digit][lo] of `ncols` column vectors of 2^log_n words for the pass (p, g); box = 32 lanes x box_digits digits
static int32_t pass_tensor_map(bfgpu_ctx* ctx, CUtensorMap* tm, const uint32_t* base, uint64_t col_stride, uint32_t ncols, unsigned log_n, unsigned p, unsigned g,
                               uint32_t box_digits) {
    const cuuint64_t gdim[4] = {1ull << p, 1ull << g, 1ull << (log_n - p - g), ncols};
    const cuuint64_t gstride[3] = {4ull << p, 4ull << (p + g), col_stride * 4};
    const cuuint32_t box[4] = {32, box_digits, 1, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = tmap_encoder()(tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 4, const_cast<uint32_t*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, BFGPU_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for a 2^%u x %u pass p=%u g=%u", (int)r, log_n, ncols, p, g);
    return BFGPU_OK;
}
// One strided pass (p, g) of size-2^log_n transforms over `ncols` column vectors at src (stride src_stride words).
// FWD / INV: in place.  TURN: reads the columns of src, writes the 2*ncols half-columns of `out` (a.pw, a.twA2, a.twB2 set by the caller).
static int32_t run_pass3(bfgpu_ctx* ctx, int mode, const uint32_t* src, uint64_t src_stride, uint32_t ncols, unsigned log_n, const bfgpu_ctx::NttPass& ps,
                         ntt3::PassArgs a, uint32_t* out = nullptr) {
    const unsigned p = ps.p, g = ps.g;
    CUtensorMap tm_in, tm_out;
    TRY(pass_tensor_map(ctx, &tm_in, src, src_stride, ncols, log_n, p, g, 1u << g));
    if (mode == ntt3::FWD) TRY(pass_tensor_map(ctx, &tm_out, src, src_stride, ncols, log_n, p, g, 16));
    else if (mode == ntt3::INV) tm_out = tm_in;
    else TRY(pass_tensor_map(ctx, &tm_out, out, 1ull << log_n, 2 * ncols, log_n, p, g, 16));
    const uint32_t tiles = 1u << (log_n - g - 5);
    // CTAs hold 2^(g+1) threads: fill the machine several times over, but keep >= 8 columns per CTA (twiddle loads, ring start-up)
    const uint32_t want_groups = std::max<uint32_t>(1, (148u * 8 + tiles - 1) / tiles);
    uint32_t cpc = std::max<uint32_t>(std::min<uint32_t>(8, ncols), (ncols + want_groups - 1) / want_groups);
    cpc = std::min<uint32_t>(cpc, mode == ntt3::TURN ? 32 : 64);
    a.ncols = ncols;
    a.cols_per_cta = cpc;
    a.p = p;
    a.log_n = log_n;
    dim3 grid(tiles, (ncols + cpc - 1) / cpc);
    switch (mode) {
        case ntt3::FWD: TRY((launch3_g<ntt3::FWD>(ctx, g, tm_in, tm_out, a, grid))); break;
        case ntt3::INV: TRY((launch3_g<ntt3::INV>(ctx, g, tm_in, tm_out, a, grid))); break;
        default: TRY((launch3_g<ntt3::TURN>(ctx, g, tm_in, tm_out, a, grid))); break;
    }
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    return BFGPU_OK;
}



// Contiguous forward pass (p = 0) through the bulk-copy kernel ntt3::k_cfwd
template <int G1>
static int32_t launch_cfwd(bfgpu_ctx* ctx, const ntt3::CfwdArgs& a, dim3 grid, cudaStream_t st) {
    const int key = 128 + G1;
    if (!ctx->ntt3_configured.count(key)) {
        CU(cudaFuncSetAttribute(ntt3::k_cfwd<G1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ntt3::cfwd_smem_bytes(G1)));
        ctx->ntt3_configured.insert(key);
    }
    ntt3::k_cfwd<G1><<<grid, 1u << (G1 + 5), ntt3::cfwd_smem_bytes(G1), st>>>(a);
    return BFGPU_OK;
}
static bool cfwd_possible(bfgpu_ctx* ctx, const bfgpu_ctx::NttPass& ps, unsigned log_n, const uint32_t* data, uint64_t col_stride) {
    return ctx->ntt_tma && ps.p == 0 && ps.g >= 5 && ps.g <= 8 && log_n >= ps.g + 5 && ((uintptr_t)data & 15) == 0 && col_stride % 4 == 0;
}
static bool cfwd_usable(bfgpu_ctx* ctx, const bfgpu_ctx::NttPass& ps, unsigned log_n, const uint32_t* data, uint64_t col_stride) {
    return ctx->ntt_cfwd && cfwd_possible(ctx, ps, log_n, data, col_stride);
}
// where the last forward pass of a sharded LDE block sends its rows (ntt3::CfwdArgs::scatter)
struct ScatterTarget {
    uint32_t log_rpg = 0, dcol0 = 0, world = 0;
    uint32_t* dst[16] = {};
};
static int32_t run_cfwd(bfgpu_ctx* ctx, uint32_t* data, uint64_t col_stride, uint32_t ncols, unsigned log_n, const bfgpu_ctx::NttPass& ps,
                        const ScatterTarget* sc = nullptr, cudaStream_t stream = nullptr) {
    const uint32_t tiles = 1u << (log_n - ps.g - 5);
    const uint32_t want_groups = std::max<uint32_t>(1, (148u * 16 + tiles - 1) / tiles);
    uint32_t cpc = std::max<uint32_t>(std::min<uint32_t>(8, ncols), (ncols + want_groups - 1) / want_groups);
    cpc = std::min<uint32_t>(cpc, 64);
    ntt3::CfwdArgs a;
    memset(&a, 0, sizeof a);
    a.data = data;
    a.col_stride = col_stride;
    a.ncols = ncols;
    a.cols_per_cta = cpc;
    a.twA = ps.twA;
    a.log_n = log_n;
    if (sc) {
        a.scatter = 1;
        a.log_rpg = sc->log_rpg;
        a.dcol0 = sc->dcol0;
        for (uint32_t r = 0; r < sc->world && r < 16; r++) a.dst[r] = sc->dst[r];
    }
    dim3 grid(tiles, (ncols + cpc - 1) / cpc);
    cudaStream_t st = stream ? stream : ctx->stream;
    switch (ps.g - 4) {
        case 1: TRY(launch_cfwd<1>(ctx, a, grid, st)); break;
        case 2: TRY(launch_cfwd<2>(ctx, a, grid, st)); break;
        case 3: TRY(launch_cfwd<3>(ctx, a, grid, st)); break;
        default: TRY(launch_cfwd<4>(ctx, a, grid, st)); break;
    }
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    return BFGPU_OK;
}

template <int G1>
static int32_t launch_ingest_pass(bfgpu_ctx* ctx, const CUtensorMap& tm, const ntt3::IngestArgs& a, dim3 grid) {
    const bool canon = ctx->repr == BFGPU_REPR_CANONICAL;
    const int key = 64 + G1 * 2 + (canon ? 1 : 0);
    const size_t smem = ntt3::ingest_smem_bytes(G1);
    if (!ctx->ntt3_configured.count(key)) {
        if (canon) CU(cudaFuncSetAttribute(ntt3::k_ingest_pass<G1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        else CU(cudaFuncSetAttribute(ntt3::k_ingest_pass<G1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ctx->ntt3_configured.insert(key);
    }
    if (canon) ntt3::k_ingest_pass<G1, true><<<grid, 1u << (G1 + 5), smem, ctx->stream>>>(tm, a);
    else ntt3::k_ingest_pass<G1, false><<<grid, 1u << (G1 + 5), smem, ctx->stream>>>(tm, a);
    return BFGPU_OK;
}
static int32_t ingest_first_pass(bfgpu_ctx* ctx, const uint32_t* src, uint64_t rows, uint32_t cols, uint32_t* dst, uint64_t pitch, bool* done) {
    *done = false;
    if (!ctx->ntt_tma || !ctx->ntt_ingest || !is_pow2(rows) || tmap_encoder() == nullptr) return BFGPU_OK;
    const unsigned log_n = ilog2(rows);
    if (log_n < 12 || log_n > (unsigned)kb::TWO_ADICITY || pitch % 4 != 0 || ((uintptr_t)src & 15) != 0 || ((uintptr_t)dst & 15) != 0) return BFGPU_OK;
    const std::vector<bfgpu_ctx::NttPass>* plan = nullptr;
    TRY(get_plan(ctx, log_n, true, &plan));
    const auto& ps = plan->front();
    if (ps.p != 0 || ps.g < 6 || ps.g > 8) return BFGPU_OK;
    const unsigned g = ps.g;
    // 3-d view [k = high g row bits][low row bits][column] of the row-major source; box = 32 columns x 1 x 2^g
    CUtensorMap tm;
    const cuuint64_t gdim[3] = {cols, 1ull << (log_n - g), 1ull << g};
    const cuuint64_t gstride[2] = {pitch * 4, (pitch * 4) << (log_n - g)};
    const cuuint32_t box[3] = {32, 1, 1u << g};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = tmap_encoder()(&tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<uint32_t*>(src), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return BFGPU_OK;  // shapes the encoder refuses go through the two-kernel path
    const uint32_t tiles = 1u << (log_n - g), nblk = (cols + 31) / 32;
    // ~16 CTAs per SM over the launch, at most 64 tiles per CTA (twiddle loads and the ring start-up are paid once per CTA)
    const uint32_t tpc = (uint32_t)std::min<uint64_t>(64, std::max<uint64_t>(1, ((uint64_t)tiles * nblk) / (148u * 16)));
    ntt3::IngestArgs a{dst, cols, tpc, log_n, ps.twA};
    dim3 grid(nblk, (tiles + tpc - 1) / tpc);
    switch (g - 4) {
        case 2: TRY(launch_ingest_pass<2>(ctx, tm, a, grid)); break;
        case 3: TRY(launch_ingest_pass<3>(ctx, tm, a, grid)); break;
        default: TRY(launch_ingest_pass<4>(ctx, tm, a, grid)); break;
    }
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    *done = true;
    return BFGPU_OK;
}

template <bool INVERSE, int G1>
static void launch_pass(bfgpu_ctx* ctx, const ntt2::PassArgs& a, dim3 grid) {
    if (INVERSE && a.pw != nullptr) {  // last inverse pass with the fused coset epilogue (always a strided pass: log_n >= 12)
        ntt2::k_pass<INVERSE, G1, false, INVERSE><<<grid, 1u << (G1 + 4), 0, ctx->stream>>>(a);
    } else if (a.p == 0) {
        ntt2::k_pass<INVERSE, G1, true><<<grid, 1u << (G1 + 4), 0, ctx->stream>>>(a);
    } else {
        ntt2::k_pass<INVERSE, G1, false><<<grid, 1u << (G1 + 4), 0, ctx->stream>>>(a);
    }
}

template <int G1>
static void launch_pass_dual(bfgpu_ctx* ctx, const ntt2::PassArgs& a, dim3 grid) {
    if (a.twA2) ntt2::k_pass<true, G1, false, false, false, true><<<grid, 1u << (G1 + 4), 0, ctx->stream>>>(a);  // TURN
    else ntt2::k_pass<false, G1, false, false, true><<<grid, 1u << (G1 + 4), 0, ctx->stream>>>(a);
}

// Run all stages of a size-2^log_n transform on `ncols` column vectors (stride col_stride words).
// Fused coset epilogue (inverse only, log_n >= NTT2_MIN_LOG): see ntt2::PassArgs::pw.
struct CosetEpilogue {
    const uint32_t* pw = nullptr;
    uint32_t* out = nullptr;
    uint32_t ncosets = 0;
};
constexpr unsigned NTT2_MIN_LOG = 12;

template <bool INVERSE>
static int32_t run_ntt(bfgpu_ctx* ctx, uint32_t* data, uint64_t col_stride, unsigned log_n, uint32_t ncols, CosetEpilogue epi = CosetEpilogue(),
                       bool skip_last = false, bool skip_first = false) {
    if (log_n == 0 || ncols == 0) return BFGPU_OK;
    Phase ph(ctx, INVERSE ? BFGPU_PHASE_INTT : BFGPU_PHASE_NTT);
    if (log_n < NTT2_MIN_LOG) return run_ntt_small<INVERSE>(ctx, data, col_stride, log_n, ncols);
    const std::vector<bfgpu_ctx::NttPass>* plan = nullptr;
    TRY(get_plan(ctx, log_n, INVERSE, &plan));
    size_t np = plan->size() - (skip_last ? 1 : 0);  // skip_last: the top pass runs inside the TURN kernel of run_ntt_forward_dual
    for (size_t s = skip_first ? 1 : 0; s < np; s++) {  // skip_first (inverse): ntt3::k_ingest_pass has run the first pass already
        const auto& ps = (*plan)[INVERSE ? s : np - 1 - s];  // inverse DIT: low bits first; forward DIF: high bits first
        if (!INVERSE && cfwd_usable(ctx, ps, log_n, data, col_stride)) {
            TRY(run_cfwd(ctx, data, col_stride, ncols, log_n, ps));
            continue;
        }
        if (ntt3_usable(ctx, ps) && !(INVERSE && s + 1 == np && epi.pw)) {
            ntt3::PassArgs a3{0, 0, 0, 0, ps.twA, ps.twB, nullptr, nullptr, nullptr};
            TRY(run_pass3(ctx, INVERSE ? ntt3::INV : ntt3::FWD, data, col_stride, ncols, log_n, ps, a3));
            continue;
        }
        uint32_t tiles = 1u << (log_n - ps.g - 4);
        // enough CTAs to fill the machine several times, but >= 8 columns per CTA to amortise the twiddle loads
        uint32_t want_groups = std::max<uint32_t>(1, (148u * 16 + tiles - 1) / tiles);
        uint32_t cpc = std::max<uint32_t>(std::min<uint32_t>(8, ncols), (ncols + want_groups - 1) / want_groups);
        cpc = std::min<uint32_t>(cpc, 64);
        ntt2::PassArgs a{data, col_stride, ncols, cpc, ps.p, ps.twA, ps.twB, nullptr, nullptr, 0, log_n, nullptr, nullptr};
        if (INVERSE && s + 1 == np && epi.pw) {
            a.pw = epi.pw;
            a.out = epi.out;
            a.ncosets = epi.ncosets;
        }
        dim3 grid(tiles, (ncols + cpc - 1) / cpc);
        switch (ps.g - 4) {
            case 0: launch_pass<INVERSE, 0>(ctx, a, grid); break;
            case 1: launch_pass<INVERSE, 1>(ctx, a, grid); break;
            case 2: launch_pass<INVERSE, 2>(ctx, a, grid); break;
            case 3: launch_pass<INVERSE, 3>(ctx, a, grid); break;
            case 4: launch_pass<INVERSE, 4>(ctx, a, grid); break;
            default: return fail(ctx, BFGPU_ERR_STATE, "internal: bad pass size %u", ps.g);
        }
        LAUNCHED(ctx);
        CU(cudaGetLastError());
    }
    return BFGPU_OK;
}

// Forward half of a blow-up-2 coset LDE from the (unscaled) coefficients: the top pass reads coef once, scales by the two coset
// vectors on load and writes both half-columns of `out` (ntt2::k_pass<..., DUAL>); the remaining passes run in place on the 2W
// half-columns.  BFGPU_NTT_DUAL=0 falls back to the epilogue-in-the-inverse-pass path of round 1.
// turn: `coef` still lacks the top inverse pass, which the first launch executes too (ntt2::k_pass<..., TURN>).
// skip_last: stop before the contiguous last pass (the caller runs it itself: sharded commitment, ntt3::k_cfwd with the row scatter)
static int32_t run_ntt_forward_dual(bfgpu_ctx* ctx, const uint32_t* coef, uint32_t* out, const uint32_t* pw, unsigned log_n, uint32_t ncols, bool turn,
                                    bool skip_last = false) {
    Phase ph(ctx, BFGPU_PHASE_NTT);
    const std::vector<bfgpu_ctx::NttPass>* plan = nullptr;
    const std::vector<bfgpu_ctx::NttPass>* iplan = nullptr;
    TRY(get_plan(ctx, log_n, false, &plan));
    if (turn) TRY(get_plan(ctx, log_n, true, &iplan));
    const size_t np = plan->size();
    const uint64_t n = 1ull << log_n;
    for (size_t s = 0; s + (skip_last ? 1 : 0) < np; s++) {
        const auto& ps = (*plan)[np - 1 - s];  // forward DIF: high bits first
        const bool dual = s == 0;
        const uint32_t cols = dual ? ncols : 2 * ncols;
        if (!dual && cfwd_usable(ctx, ps, log_n, out, n)) {
            TRY(run_cfwd(ctx, out, n, cols, log_n, ps));
            continue;
        }
        if (ntt3_usable(ctx, ps) && (!dual || turn)) {  // (the DUAL pass without the inverse half exists only in ntt2::k_pass)
            ntt3::PassArgs a3{0, 0, 0, 0, ps.twA, ps.twB, nullptr, nullptr, nullptr};
            if (dual) {
                const auto& ips = iplan->back();
                if (ips.p != ps.p || ips.g != ps.g) return fail(ctx, BFGPU_ERR_STATE, "internal: inverse and forward top passes differ");
                a3.twA = ips.twA;
                a3.twB = ips.twB;
                a3.twA2 = ps.twA;
                a3.twB2 = ps.twB;
                a3.pw = pw;
                TRY(run_pass3(ctx, ntt3::TURN, coef, n, cols, log_n, ps, a3, out));
            } else {
                TRY(run_pass3(ctx, ntt3::FWD, out, n, cols, log_n, ps, a3));
            }
            continue;
        }
        uint32_t tiles = 1u << (log_n - ps.g - 4);
        uint32_t want_groups = std::max<uint32_t>(1, (148u * 16 + tiles - 1) / tiles);
        uint32_t cpc = std::max<uint32_t>(std::min<uint32_t>(8, cols), (cols + want_groups - 1) / want_groups);
        cpc = std::min<uint32_t>(cpc, dual ? 32 : 64);
        ntt2::PassArgs a{dual ? const_cast<uint32_t*>(coef) : out, n, cols, cpc, ps.p, ps.twA, ps.twB, nullptr, nullptr, 0, log_n, nullptr, nullptr};
        dim3 grid(tiles, (cols + cpc - 1) / cpc);
        if (dual) {
            a.pw = pw;
            a.out = out;
            a.ncosets = 2;
            if (turn) {  // inverse tables drive the first half of the kernel, the forward ones of the same (p, g) the second
                const auto& ips = iplan->back();
                if (ips.p != ps.p || ips.g != ps.g) return fail(ctx, BFGPU_ERR_STATE, "internal: inverse and forward top passes differ");
                a.twA = ips.twA;
                a.twB = ips.twB;
                a.twA2 = ps.twA;
                a.twB2 = ps.twB;
            }
            if (ps.p == 0 || ps.g < 5) return fail(ctx, BFGPU_ERR_STATE, "internal: dual pass needs a strided two-phase top pass");
            switch (ps.g - 4) {
                case 1: launch_pass_dual<1>(ctx, a, grid); break;
                case 2: launch_pass_dual<2>(ctx, a, grid); break;
                case 3: launch_pass_dual<3>(ctx, a, grid); break;
                case 4: launch_pass_dual<4>(ctx, a, grid); break;
                default: return fail(ctx, BFGPU_ERR_STATE, "internal: bad pass size %u", ps.g);
            }
        } else {
            switch (ps.g - 4) {
                case 0: launch_pass<false, 0>(ctx, a, grid); break;
                case 1: launch_pass<false, 1>(ctx, a, grid); break;
                case 2: launch_pass<false, 2>(ctx, a, grid); break;
                case 3: launch_pass<false, 3>(ctx, a, grid); break;
                case 4: launch_pass<false, 4>(ctx, a, grid); break;
                default: return fail(ctx, BFGPU_ERR_STATE, "internal: bad pass size %u", ps.g);
            }
        }
        LAUNCHED(ctx);
        CU(cudaGetLastError());
    }
    return BFGPU_OK;
}

// per-coset scale vectors: pw[h*n + k] = (shift * w_N^{bitrev(h)})^k / n  (cached: a proof reuses a handful)
static int32_t coset_powers(bfgpu_ctx* ctx, unsigned log_n, unsigned added_bits, uint32_t shift_mont, uint32_t** out) {
    auto key = std::make_tuple(log_n, added_bits, shift_mont);
    auto it = ctx->pw_cache.find(key);
    if (it != ctx->pw_cache.end()) {
        *out = it->second;
        return BFGPU_OK;
    }
    Phase ph(ctx, BFGPU_PHASE_SCALE);
    const uint64_t n = 1ull << log_n, N = n << added_bits;
    const uint32_t ncosets = 1u << added_bits;
    uint32_t* pw = nullptr;
    CU(cudaMalloc(&pw, N * 4));
    uint32_t ninv = kb::inv(kb::to_mont((uint32_t)(n % kb::P)));
    uint32_t wN = kb::two_adic_generator(log_n + added_bits);
    for (uint32_t h = 0; h < ncosets; h++) {
        uint32_t sh = kb::mul(shift_mont, kb::pow(wN, kb::bitrev(h, added_bits)));
        nttk::k_powers<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(pw + h * n, sh, ninv, n);
        LAUNCHED(ctx);
    }
    CU(cudaGetLastError());
    ctx->pw_cache[key] = pw;
    *out = pw;
    return BFGPU_OK;
}

// coset LDE of a column-major device matrix whose rows are already in bit-reversed order (consumed) ->
// column-major device matrix with bit-reversed rows.  shift_mont: Montgomery form of the coset shift.
// first_pass_done: the first inverse pass has been executed by the fused ingest (ntt3::k_ingest_pass)
// defer_last_pass != null (sharded commitment): if the shape allows, everything but the contiguous last forward pass is enqueued,
// *defer_last_pass = true and the caller finishes with lde_last_pass_scatter(); otherwise it stays false and the LDE is complete.
static int32_t lde_from_bitrev(bfgpu_ctx* ctx, DMat coef, unsigned added_bits, uint32_t shift_mont, DMat* out, bool consume = true,
                               uint32_t* out_buf = nullptr, bool first_pass_done = false, bool* defer_last_pass = nullptr) {
    unsigned log_n = ilog2(coef.rows);
    if (log_n + added_bits > kb::TWO_ADICITY) return fail(ctx, BFGPU_ERR_INVALID, "LDE height 2^%u exceeds the field's two-adicity", log_n + added_bits);
    uint64_t n = coef.rows, N = n << added_bits;
    uint32_t ncosets = 1u << added_bits;
    uint32_t* pw = nullptr;
    TRY(coset_powers(ctx, log_n, added_bits, shift_mont, &pw));
    out->rows = N;
    out->cols = coef.cols;
    if (out_buf) out->d = out_buf;  // caller-provided destination (a column block of a larger matrix)
    else TRY(dalloc(ctx, (void**)&out->d, N * coef.cols * 4));
    if (log_n >= NTT2_MIN_LOG && ncosets == 2 && ctx->ntt_dual) {
        // plain inverse transform; the coset scaling and the 2-fold expansion happen on load in the first forward pass
        bool defer = false;
        if (defer_last_pass) {
            const std::vector<bfgpu_ctx::NttPass>* fplan = nullptr;
            TRY(get_plan(ctx, log_n, false, &fplan));
            defer = ctx->dist_fused_scatter && fplan->size() >= 2 && cfwd_possible(ctx, fplan->front(), log_n, out->d, n);
            *defer_last_pass = defer;
        }
        TRY(run_ntt<true>(ctx, coef.d, n, log_n, coef.cols, CosetEpilogue(), ctx->ntt_turn, first_pass_done));
        TRY(run_ntt_forward_dual(ctx, coef.d, out->d, pw, log_n, coef.cols, ctx->ntt_turn, defer));
        if (consume) dfree(ctx, coef.d);  // stream order keeps it alive for the pass above
        return BFGPU_OK;
    }
    if (log_n >= NTT2_MIN_LOG && ncosets == 2) {
        // scaling and 2-fold expansion fused into the last inverse pass
        CosetEpilogue epi;
        epi.pw = pw;
        epi.out = out->d;
        epi.ncosets = ncosets;
        TRY(run_ntt<true>(ctx, coef.d, n, log_n, coef.cols, epi, false, first_pass_done));
    } else {
        TRY(run_ntt<true>(ctx, coef.d, n, log_n, coef.cols, CosetEpilogue(), false, first_pass_done));
        Phase ph(ctx, BFGPU_PHASE_SCALE);
        dim3 grid((unsigned)((n + 255) / 256), coef.cols);
        nttk::k_scale_cosets<<<grid, 256, 0, ctx->stream>>>(coef.d, out->d, pw, n, ncosets, coef.cols);
        LAUNCHED(ctx);
        CU(cudaGetLastError());
    }
    if (consume) dfree(ctx, coef.d);
    TRY(run_ntt<false>(ctx, out->d, n, log_n, coef.cols * ncosets));
    return BFGPU_OK;
}

// Last (contiguous) forward pass of a blow-up-2 LDE block whose earlier passes were enqueued by lde_from_bitrev(defer_last_pass):
// reads the 2W half-columns of `lde`, sends every run of rows to the rank that owns it (ScatterTarget), on `stream`.
static int32_t lde_last_pass_scatter(bfgpu_ctx* ctx, const DMat& lde, const ScatterTarget& sc, cudaStream_t stream) {
    const unsigned log_n = ilog2(lde.rows) - 1;
    const std::vector<bfgpu_ctx::NttPass>* fplan = nullptr;
    TRY(get_plan(ctx, log_n, false, &fplan));
    const auto& ps = fplan->front();
    if (sc.log_rpg < ps.g) return fail(ctx, BFGPU_ERR_STATE, "internal: a row shard is shorter than a run of the last pass");
    Phase ph(ctx, BFGPU_PHASE_EXCHANGE);
    return run_cfwd(ctx, lde.d, 1ull << log_n, 2 * lde.cols, log_n, ps, &sc, stream);
}

// Coset LDEs of several coefficient matrices (column-major, bit-reversed rows, consumed): columns of at most
// 2^SMALL_LDE_MAX_LOG points of ALL matrices go through one nttk::k_lde_small launch, the rest through lde_from_bitrev.
static int32_t lde_many(bfgpu_ctx* ctx, std::vector<DMat>& coefs, unsigned added_bits, const std::vector<uint32_t>& shift_mont, std::vector<DMat>* out) {
    out->assign(coefs.size(), DMat());
    nttk::SmallLdeArgs sa;
    memset(&sa, 0, sizeof sa);
    sa.ncosets = 1u << added_bits;
    sa.tw = ctx->d_tw;
    std::vector<size_t> small;
    auto flush = [&]() -> int32_t {
        if (!sa.nmats) return BFGPU_OK;
        Phase ph(ctx, BFGPU_PHASE_NTT);
        nttk::k_lde_small<<<sa.first_cta[sa.nmats], 256, 0, ctx->stream>>>(sa);
        LAUNCHED(ctx);
        CU(cudaGetLastError());
        for (size_t i : small) {
            dfree(ctx, coefs[i].d);
            coefs[i].d = nullptr;
        }
        small.clear();
        sa.nmats = 0;
        return BFGPU_OK;
    };
    for (size_t i = 0; i < coefs.size(); i++) {
        const unsigned log_n = ilog2(coefs[i].rows);
        if (log_n + added_bits > (unsigned)kb::TWO_ADICITY) return fail(ctx, BFGPU_ERR_INVALID, "LDE height 2^%u exceeds the field's two-adicity", log_n + added_bits);
        if (log_n > (unsigned)nttk::SMALL_LDE_MAX_LOG || coefs[i].cols == 0) {
            TRY(lde_from_bitrev(ctx, coefs[i], added_bits, shift_mont[i], &(*out)[i]));
            coefs[i].d = nullptr;
            continue;
        }
        if (sa.nmats == (uint32_t)nttk::SMALL_LDE_MAX_MATS) TRY(flush());
        DMat& o = (*out)[i];
        o.rows = coefs[i].rows << added_bits;
        o.cols = coefs[i].cols;
        TRY(dalloc(ctx, (void**)&o.d, o.rows * o.cols * 4));
        uint32_t* pw = nullptr;
        TRY(coset_powers(ctx, log_n, added_bits, shift_mont[i], &pw));
        const uint32_t k = sa.nmats++;
        sa.coef[k] = coefs[i].d;
        sa.out[k] = o.d;
        sa.pw[k] = pw;
        sa.log_n[k] = log_n;
        sa.first_cta[k + 1] = sa.first_cta[k] + coefs[i].cols;
        small.push_back(i);
    }
    return flush();
}

// coset LDE of a caller matrix.  keep != null: also return a copy of the ingested trace (column-major,
// bit-reversed rows), which the LogUp kernel reads later.
static int32_t lde_device(bfgpu_ctx* ctx, const bfgpu_mat& m, unsigned added_bits, uint32_t shift_mont, DMat* out, DMat* keep = nullptr) {
    if (ilog2(m.rows) + added_bits > kb::TWO_ADICITY)
        return fail(ctx, BFGPU_ERR_INVALID, "LDE height 2^%u exceeds the field's two-adicity (2^%d)", ilog2(m.rows) + added_bits, kb::TWO_ADICITY);
    DMat coef;
    bool first_pass_done = false;
    TRY(ingest(ctx, m, /*bitrev=*/true, &coef, keep ? nullptr : &first_pass_done));  // a kept copy must be the plain transposed trace
    if (keep) {
        *keep = coef;
        size_t bytes = (size_t)coef.rows * coef.cols * 4;
        TRY(dalloc(ctx, (void**)&keep->d, bytes));
        CU(cudaMemcpyAsync(keep->d, coef.d, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    return lde_from_bitrev(ctx, coef, added_bits, shift_mont, out, true, nullptr, first_pass_done);
}

static int32_t coset_lde_batch_impl(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t added_bits, uint32_t shift, int bit_reversed_rows,
                                         uint32_t* out);
extern "C" int32_t bfgpu_coset_lde_batch(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t added_bits, uint32_t shift, int bit_reversed_rows,
                                         uint32_t* out) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(coset_lde_batch_impl(ctx, mat, added_bits, shift, bit_reversed_rows, out));
}
static int32_t coset_lde_batch_impl(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t added_bits, uint32_t shift, int bit_reversed_rows,
                                         uint32_t* out) {
    if (!ctx || !out) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    TRY(check_mat(ctx, mat, true));
    uint32_t sm = ctx->repr == BFGPU_REPR_CANONICAL ? kb::to_mont(shift % kb::P) : shift;
    DMat lde;
    TRY(lde_device(ctx, *mat, added_bits, sm, &lde));
    int32_t rc = egress(ctx, lde, !bit_reversed_rows, out);  // stored bit-reversed: un-reverse for natural order
    dfree(ctx, lde.d);
    return rc;
}

static int32_t dft_batch_impl(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t* out);
extern "C" int32_t bfgpu_dft_batch(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t* out) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(dft_batch_impl(ctx, mat, out));
}
static int32_t dft_batch_impl(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t* out) {
    if (!ctx || !out) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    TRY(check_mat(ctx, mat, true));
    DMat d;
    TRY(ingest(ctx, *mat, false, &d));
    TRY(run_ntt<false>(ctx, d.d, d.rows, ilog2(d.rows), d.cols));
    int32_t rc = egress(ctx, d, true, out);
    dfree(ctx, d.d);
    return rc;
}

static int32_t idft_batch_impl(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t* out);
extern "C" int32_t bfgpu_idft_batch(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t* out) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(idft_batch_impl(ctx, mat, out));
}
static int32_t idft_batch_impl(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t* out) {
    if (!ctx || !out) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    TRY(check_mat(ctx, mat, true));
    DMat d;
    TRY(ingest(ctx, *mat, true, &d));
    TRY(run_ntt<true>(ctx, d.d, d.rows, ilog2(d.rows), d.cols));
    uint64_t total = d.rows * d.cols;
    nttk::k_scale<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(d.d, total, kb::inv(kb::to_mont((uint32_t)(d.rows % kb::P))));
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    int32_t rc = egress(ctx, d, false, out);
    dfree(ctx, d.d);
    return rc;
}

// ---- Poseidon2 primitives --------------------------------------------------------------------------
static int32_t convert_inplace(bfgpu_ctx* ctx, uint32_t* d, uint64_t n, bool to_mont) {
    if (ctx->repr != BFGPU_REPR_CANONICAL || n == 0) return BFGPU_OK;
    hashk::k_convert<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(d, n, to_mont ? 1 : 0);
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    return BFGPU_OK;
}

static int32_t poseidon2_permute_impl(bfgpu_ctx* ctx, uint32_t* states, uint64_t n);
extern "C" int32_t bfgpu_poseidon2_permute(bfgpu_ctx* ctx, uint32_t* states, uint64_t n) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(poseidon2_permute_impl(ctx, states, n));
}
static int32_t poseidon2_permute_impl(bfgpu_ctx* ctx, uint32_t* states, uint64_t n) {
    if (!ctx || (!states && n)) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    if (n == 0) return BFGPU_OK;
    uint32_t* d = nullptr;
    size_t bytes = n * 64;
    if (ctx->input_space == BFGPU_MEM_HOST) {
        TRY(dalloc(ctx, (void**)&d, bytes));
        CU(cudaMemcpyAsync(d, states, bytes, cudaMemcpyHostToDevice, ctx->stream));
    } else {
        d = states;
    }
    TRY(convert_inplace(ctx, d, n * 16, true));
    hashk::k_permute_many<<<(unsigned)((n + hashk::HASH_THREADS - 1) / hashk::HASH_THREADS), hashk::HASH_THREADS, 0, ctx->stream>>>(d, n);
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    TRY(convert_inplace(ctx, d, n * 16, false));
    if (ctx->input_space == BFGPU_MEM_HOST) {
        CU(cudaMemcpyAsync(states, d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        dfree(ctx, d);
    }
    return BFGPU_OK;
}

// device array of column base pointers for a list of matrices (in the given order)
static int32_t make_colptr(bfgpu_ctx* ctx, const std::vector<const DMat*>& mats, const uint32_t*** d_out, uint32_t* ncols_out) {
    std::vector<const uint32_t*> h;
    for (const DMat* m : mats)
        for (uint32_t c = 0; c < m->cols; c++) h.push_back(m->d + (uint64_t)c * m->col_stride());
    *ncols_out = (uint32_t)h.size();
    TRY(dalloc(ctx, (void**)d_out, h.size() * sizeof(void*)));
    TRY(upload_small(ctx, (void*)*d_out, h.data(), h.size() * sizeof(void*)));
    return BFGPU_OK;
}

static int32_t sponge_hash_rows_impl(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t* digests);
extern "C" int32_t bfgpu_sponge_hash_rows(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t* digests) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(sponge_hash_rows_impl(ctx, mat, digests));
}
static int32_t sponge_hash_rows_impl(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t* digests) {
    if (!ctx || !digests) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    TRY(check_mat(ctx, mat, false));
    DMat d;
    TRY(ingest(ctx, *mat, false, &d));
    const uint32_t** colptr = nullptr;
    uint32_t ncols = 0;
    TRY(make_colptr(ctx, {&d}, &colptr, &ncols));
    uint32_t* out = nullptr;
    TRY(dalloc(ctx, (void**)&out, d.rows * 32));
    hashk::k_leaf_hash<<<(unsigned)((d.rows + hashk::HASH_THREADS - 1) / hashk::HASH_THREADS), hashk::HASH_THREADS, 0, ctx->stream>>>(colptr, ncols, d.rows, out, 1);
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    TRY(convert_inplace(ctx, out, d.rows * 8, false));
    CU(cudaMemcpyAsync(digests, out, d.rows * 32, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    dfree(ctx, out);
    dfree(ctx, (void*)colptr);
    dfree(ctx, d.d);
    return BFGPU_OK;
}

static int32_t compress_impl(bfgpu_ctx* ctx, const uint32_t* left, const uint32_t* right, uint64_t n, uint32_t* out);
extern "C" int32_t bfgpu_compress(bfgpu_ctx* ctx, const uint32_t* left, const uint32_t* right, uint64_t n, uint32_t* out) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(compress_impl(ctx, left, right, n, out));
}
static int32_t compress_impl(bfgpu_ctx* ctx, const uint32_t* left, const uint32_t* right, uint64_t n, uint32_t* out) {
    if (!ctx || !left || !right || !out) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    if (n == 0) return BFGPU_OK;
    uint32_t *l = nullptr, *r = nullptr, *o = nullptr;
    TRY(dalloc(ctx, (void**)&l, n * 32));
    TRY(dalloc(ctx, (void**)&r, n * 32));
    TRY(dalloc(ctx, (void**)&o, n * 32));
    CU(cudaMemcpyAsync(l, left, n * 32, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(r, right, n * 32, cudaMemcpyHostToDevice, ctx->stream));
    TRY(convert_inplace(ctx, l, n * 8, true));
    TRY(convert_inplace(ctx, r, n * 8, true));
    hashk::k_compress_pairs<<<(unsigned)((n + hashk::HASH_THREADS - 1) / hashk::HASH_THREADS), hashk::HASH_THREADS, 0, ctx->stream>>>(l, r, o, n);
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    TRY(convert_inplace(ctx, o, n * 8, false));
    CU(cudaMemcpyAsync(out, o, n * 32, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    dfree(ctx, l);
    dfree(ctx, r);
    dfree(ctx, o);
    return BFGPU_OK;
}

// ---- MerkleTreeMmcs ----------------------------------------------------------------------------------
static void tree_release(bfgpu_tree* t) {
    if (!t) return;
    for (uint32_t* l : t->layers) dfree(t->ctx, l);
    if (t->owns_mats)
        for (DMat& m : t->mats) dfree(t->ctx, m.d);
    delete t;
}

// Build the tree over device matrices (input order preserved in t->mats).
// first_layer != null: the leaf digests of the tallest group were already produced (pipelined commit) and are adopted.
static int32_t build_tree(bfgpu_ctx* ctx, std::vector<DMat> mats, bool owns, bfgpu_tree** out, uint32_t* first_layer = nullptr) {
    bfgpu_tree* t = new bfgpu_tree();
    t->ctx = ctx;
    t->mats = std::move(mats);
    t->owns_mats = owns;
    *out = t;
    size_t n = t->mats.size();
    std::vector<size_t> order(n);
    for (size_t i = 0; i < n; i++) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return t->mats[a].rows > t->mats[b].rows; });
    uint64_t max_h = t->mats[order[0]].rows;
    t->log_max = ilog2(max_h);
    size_t pos = 0;
    auto take_group = [&](uint64_t h) {
        std::vector<const DMat*> g;
        while (pos < n && t->mats[order[pos]].rows == h) g.push_back(&t->mats[order[pos++]]);
        return g;
    };
    if (first_layer) {
        take_group(max_h);
        t->layers.push_back(first_layer);
        t->layer_len.push_back(max_h);
    } else {
        Phase ph(ctx, BFGPU_PHASE_LEAF);
        auto g = take_group(max_h);
        const uint32_t** colptr = nullptr;
        uint32_t ncols = 0;
        TRY(make_colptr(ctx, g, &colptr, &ncols));
        uint32_t* layer = nullptr;
        TRY(dalloc(ctx, (void**)&layer, max_h * 32));
        t->layers.push_back(layer);
        t->layer_len.push_back(max_h);
        hashk::k_leaf_hash<<<(unsigned)((max_h + hashk::HASH_THREADS - 1) / hashk::HASH_THREADS), hashk::HASH_THREADS, 0, ctx->stream>>>(colptr, ncols, max_h, layer, g[0]->rs);
        LAUNCHED(ctx);
        CU(cudaGetLastError());
        dfree(ctx, (void*)colptr);
    }
    Phase ph(ctx, BFGPU_PHASE_COMPRESS);
    std::vector<void*> colptrs_to_free;
    hashk::TopArgs top;
    memset(&top, 0, sizeof top);
    for (unsigned l = 1; l <= t->log_max; l++) {
        uint64_t len = max_h >> l;
        auto g = take_group(len);
        const uint32_t** colptr = nullptr;
        uint32_t ncols = 0;
        if (!g.empty()) TRY(make_colptr(ctx, g, &colptr, &ncols));
        uint32_t* layer = nullptr;
        TRY(dalloc(ctx, (void**)&layer, len * 32));
        t->layers.push_back(layer);
        t->layer_len.push_back(len);
        uint32_t rs = g.empty() ? 1u : g[0]->rs;
        if (2 * len <= hashk::TOP_MAX) {
            // the rest of the tree is computed by one single-CTA launch
            if (top.nlevels == 0) {
                top.in = t->layers[l - 1];
                top.len0 = (uint32_t)(2 * len);
            }
            top.out[top.nlevels] = layer;
            top.colptr[top.nlevels] = colptr;
            top.ncols[top.nlevels] = ncols;
            top.row_stride[top.nlevels] = rs;
            top.nlevels++;
            colptrs_to_free.push_back((void*)colptr);
            continue;
        }
        if (len <= ctx->x4_layer_max)  // narrow layer: latency-bound, four lanes per node
            hashk::k_compress_layer_x4<<<(unsigned)((4 * len + hashk::HASH_THREADS - 1) / hashk::HASH_THREADS), hashk::HASH_THREADS, 0, ctx->stream>>>(
                t->layers[l - 1], layer, len, colptr, ncols, rs);
        else
            hashk::k_compress_layer<<<(unsigned)((len + hashk::HASH_THREADS - 1) / hashk::HASH_THREADS), hashk::HASH_THREADS, 0, ctx->stream>>>(
                t->layers[l - 1], layer, len, colptr, ncols, rs);
        LAUNCHED(ctx);
        CU(cudaGetLastError());
        dfree(ctx, (void*)colptr);
    }
    if (top.nlevels) {
        top.x1_max = ctx->top_x1_max;
        // wide tops run on a cluster of 8 CTAs (their first levels are bound by one SM's issue rate), narrow ones on one CTA
        if (ctx->top_cluster && top.len0 >= (uint32_t)hashk::TOPC_MIN_LEN0 && top.nlevels == ilog2(top.len0))
            hashk::k_compress_top_cluster<<<hashk::TOPC_CLUSTER, hashk::TOPC_THREADS, 0, ctx->stream>>>(top);
        else
            hashk::k_compress_top<<<1, hashk::TOP_THREADS, 0, ctx->stream>>>(top);
        LAUNCHED(ctx);
        CU(cudaGetLastError());
        for (void* p : colptrs_to_free) dfree(ctx, p);
    }
    if (pos != n) return fail(ctx, BFGPU_ERR_INVALID, "matrix heights are not powers of two below the tallest");
    return BFGPU_OK;
}

static int32_t read_digest(bfgpu_ctx* ctx, const uint32_t* d, uint32_t out[8]) {
    CU(cudaMemcpyAsync(out, d, 32, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->repr == BFGPU_REPR_CANONICAL)
        for (int i = 0; i < 8; i++) out[i] = kb::from_mont(out[i]);
    return BFGPU_OK;
}

static int32_t mmcs_commit_impl(bfgpu_ctx* ctx, const bfgpu_mat* mats, int32_t n, uint32_t root[8], bfgpu_tree** out);
extern "C" int32_t bfgpu_mmcs_commit(bfgpu_ctx* ctx, const bfgpu_mat* mats, int32_t n, uint32_t root[8], bfgpu_tree** out) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(mmcs_commit_impl(ctx, mats, n, root, out));
}
static int32_t mmcs_commit_impl(bfgpu_ctx* ctx, const bfgpu_mat* mats, int32_t n, uint32_t root[8], bfgpu_tree** out) {
    if (!ctx || !mats || n <= 0 || !root || !out) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    *out = nullptr;
    for (int i = 0; i < n; i++) TRY(check_mat(ctx, &mats[i], true));
    std::vector<DMat> d(n);
    for (int i = 0; i < n; i++) TRY(ingest(ctx, mats[i], false, &d[i]));
    bfgpu_tree* t = nullptr;
    int32_t rc = build_tree(ctx, std::move(d), true, &t);
    if (rc == BFGPU_OK) rc = read_digest(ctx, t->layers.back(), root);
    if (rc != BFGPU_OK) {
        tree_release(t);
        return rc;
    }
    *out = t;
    return BFGPU_OK;
}

static int32_t mmcs_open_batch_impl(bfgpu_tree* t, uint64_t index, uint32_t* opened_rows, uint32_t* siblings);
extern "C" int32_t bfgpu_mmcs_open_batch(bfgpu_tree* t, uint64_t index, uint32_t* opened_rows, uint32_t* siblings) {
    AllocScope scope(t ? t->ctx : nullptr);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(mmcs_open_batch_impl(t, index, opened_rows, siblings));
}
static int32_t mmcs_open_batch_impl(bfgpu_tree* t, uint64_t index, uint32_t* opened_rows, uint32_t* siblings) {
    if (!t) return BFGPU_ERR_INVALID;
    bfgpu_ctx* ctx = t->ctx;
    if (!opened_rows || (!siblings && t->log_max)) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    if (index >= (1ull << t->log_max)) return fail(ctx, BFGPU_ERR_INVALID, "index %llu out of range", (unsigned long long)index);
    std::vector<const uint32_t*> cp;
    std::vector<uint64_t> ri;
    for (const DMat& m : t->mats) {
        uint64_t r = index >> (t->log_max - ilog2(m.rows));
        for (uint32_t c = 0; c < m.cols; c++) {
            cp.push_back(m.d + (uint64_t)c * m.col_stride());
            ri.push_back(r * m.rs);
        }
    }
    uint32_t nc = (uint32_t)cp.size();
    const uint32_t** d_cp = nullptr;
    uint64_t* d_ri = nullptr;
    uint32_t* d_out = nullptr;
    TRY(dalloc(ctx, (void**)&d_cp, nc * sizeof(void*)));
    TRY(dalloc(ctx, (void**)&d_ri, nc * 8));
    TRY(dalloc(ctx, (void**)&d_out, nc * 4));
    TRY(upload_small(ctx, (void*)d_cp, cp.data(), nc * sizeof(void*)));
    TRY(upload_small(ctx, d_ri, ri.data(), nc * 8));
    hashk::k_gather_row<<<(nc + 127) / 128, 128, 0, ctx->stream>>>(d_cp, d_ri, nc, d_out, ctx->repr == BFGPU_REPR_CANONICAL);
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(opened_rows, d_out, nc * 4, cudaMemcpyDeviceToHost, ctx->stream));
    for (unsigned l = 0; l < t->log_max; l++)
        CU(cudaMemcpyAsync(siblings + 8 * l, t->layers[l] + 8 * ((index >> l) ^ 1), 32, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->repr == BFGPU_REPR_CANONICAL)
        for (unsigned i = 0; i < 8 * t->log_max; i++) siblings[i] = kb::from_mont(siblings[i]);
    dfree(ctx, (void*)d_cp);
    dfree(ctx, d_ri);
    dfree(ctx, d_out);
    return BFGPU_OK;
}

extern "C" int32_t bfgpu_tree_num_layers(const bfgpu_tree* t) { return t ? (int32_t)t->layers.size() : 0; }
extern "C" uint64_t bfgpu_tree_layer_len(const bfgpu_tree* t, int32_t l) {
    return (t && l >= 0 && (size_t)l < t->layers.size()) ? t->layer_len[l] : 0;
}
static int32_t tree_get_layer_impl(bfgpu_tree* t, int32_t l, uint32_t* digests);
extern "C" int32_t bfgpu_tree_get_layer(bfgpu_tree* t, int32_t l, uint32_t* digests) {
    AllocScope scope(t ? t->ctx : nullptr);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(tree_get_layer_impl(t, l, digests));
}
static int32_t tree_get_layer_impl(bfgpu_tree* t, int32_t l, uint32_t* digests) {
    if (!t) return BFGPU_ERR_INVALID;
    bfgpu_ctx* ctx = t->ctx;
    if (l < 0 || (size_t)l >= t->layers.size() || !digests) return fail(ctx, BFGPU_ERR_INVALID, "bad layer");
    uint64_t words = t->layer_len[l] * 8;
    CU(cudaMemcpyAsync(digests, t->layers[l], words * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->repr == BFGPU_REPR_CANONICAL)
        for (uint64_t i = 0; i < words; i++) digests[i] = kb::from_mont(digests[i]);
    return BFGPU_OK;
}
extern "C" void bfgpu_tree_free(bfgpu_tree* t) { tree_release(t); }

// ---- TwoAdicFriPcs::commit ------------------------------------------------------------------------------
// Commit of ONE tall host matrix as a three-stage pipeline over blocks of `pipe_cols` columns:
//   copy stream   : strided host->device copy of block b+1 (cudaMemcpy2DAsync out of the row-major host matrix)
//   compute stream: ingest + coset LDE of block b into its slice of the column-major LDE, then the leaf sponge
//                   absorbs the block's columns (k_leaf_absorb; 16-word states parked in HBM between blocks).
// PCIe (~55 GB/s) and the GPU work (~LDE + hash) take about the same time at 2^22 x 256, so the commit from host
// memory costs about max(copy, compute) instead of their sum.  Same LDE, same digests as the one-shot path.
// Experiment switch (ctx->overlap_device, off): device-resident input through the same block structure with the leaf
// sponge of block b on the second stream, concurrent with the NTT of block b+1.  It lost 5 % (see bfgpu_ctx).
static int32_t commit_host_pipelined(bfgpu_ctx* ctx, const bfgpu_mat& m, unsigned added_bits, uint32_t shift_mont, DMat* lde, uint32_t** first_layer) {
    const bool from_device = ctx->input_space == BFGPU_MEM_DEVICE;
    const uint64_t R = m.rows, N = R << added_bits;
    const uint32_t W = (uint32_t)m.cols, CB = ctx->pipe_cols;
    // block boundaries (multiples of 8 columns).  The copy is the longer stage, so the commit ends one block of compute
    // after the last byte arrives: the final block is split in two to shorten that tail (narrower strided copies are
    // slower per byte, so only the tail is split).
    std::vector<uint32_t> start;
    uint32_t max_block = CB;
    if (const char* e = getenv("BFGPU_PIPE_SCHEDULE")) {  // experiment: explicit block widths "w0,w1,..." (multiples of 8 summing to W)
        uint32_t c = 0;
        bool ok = true;
        for (const char* q = e; *q && ok;) {
            char* end = nullptr;
            const unsigned long w = strtoul(q, &end, 10);
            if (end == q || w == 0 || w % 8 != 0 || c + w > W) ok = false;
            else {
                start.push_back(c);
                c += (uint32_t)w;
                max_block = std::max<uint32_t>(max_block, (uint32_t)w);
                q = *end == ',' ? end + 1 : end;
            }
        }
        if (!ok || c != W) start.clear();
    }
    if (start.empty()) {
        for (uint32_t c = 0; c < W; c += CB) start.push_back(c);
        for (int split = 0; split < ctx->pipe_tail_splits; split++) {  // halve the final block (down to 16 columns)
            uint32_t last = start.back(), len = W - last, half = (len / 2 + 7) / 8 * 8;
            if (len < 32 || half >= len) break;
            start.push_back(last + half);
        }
    }
    start.push_back(W);
    const uint32_t nb = (uint32_t)start.size() - 1;
    if (ilog2(R) + added_bits > kb::TWO_ADICITY)
        return fail(ctx, BFGPU_ERR_INVALID, "LDE height 2^%u exceeds the field's two-adicity (2^%d)", ilog2(R) + added_bits, kb::TWO_ADICITY);
    lde->rows = N;
    lde->cols = W;
    lde->rs = 1;
    uint32_t *staged[2] = {nullptr, nullptr}, *state = nullptr, *layer = nullptr;
    TRY(dalloc(ctx, (void**)&lde->d, N * W * 4));
    if (!from_device) {
        TRY(dalloc(ctx, (void**)&staged[0], R * max_block * 4));
        TRY(dalloc(ctx, (void**)&staged[1], R * max_block * 4));
    }
    TRY(dalloc(ctx, (void**)&state, N * 16 * 4));
    TRY(dalloc(ctx, (void**)&layer, N * 32));
    cudaEvent_t ready[2] = {nullptr, nullptr}, consumed[2] = {nullptr, nullptr}, fence;
    struct EventGuard {  // CU() below may return from inside the block loop
        cudaEvent_t *a, *b;
        ~EventGuard() {
            for (int k = 0; k < 2; k++) {
                if (a[k]) cudaEventDestroy(a[k]);
                if (b[k]) cudaEventDestroy(b[k]);
            }
        }
    } event_guard{ready, consumed};
    for (int k = 0; k < 2; k++) {
        CU(cudaEventCreateWithFlags(&ready[k], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&consumed[k], cudaEventDisableTiming));
    }
    CU(cudaEventCreateWithFlags(&fence, cudaEventDisableTiming));
    CU(cudaEventRecord(fence, ctx->stream));  // the staging blocks come from the single-stream block cache
    CU(cudaStreamWaitEvent(ctx->copy_stream, fence, 0));
    cudaEventDestroy(fence);
    int32_t rc = BFGPU_OK;
    auto copy_block = [&](uint32_t b) -> int32_t {
        const int slot = b & 1;
        const uint32_t cb = start[b + 1] - start[b];
        if (b >= 2) CU(cudaStreamWaitEvent(ctx->copy_stream, consumed[slot], 0));
        CU(cudaMemcpy2DAsync(staged[slot], (size_t)cb * 4, m.data + start[b], (size_t)W * 4, (size_t)cb * 4, R, cudaMemcpyHostToDevice, ctx->copy_stream));
        CU(cudaEventRecord(ready[slot], ctx->copy_stream));
        return BFGPU_OK;
    };
    if (!from_device) rc = copy_block(0);
    for (uint32_t b = 0; b < nb && rc == BFGPU_OK; b++) {
        const int slot = b & 1;
        const uint32_t cb = start[b + 1] - start[b];
        DMat coef, blk;
        coef.rows = R;
        coef.cols = cb;
        bool first_pass_done = false;
        if ((rc = dalloc(ctx, (void**)&coef.d, R * cb * 4)) != BFGPU_OK) break;
        if (from_device) {
            if ((rc = ingest_device(ctx, m.data + start[b], R, cb, /*bitrev=*/true, coef.d, W, &first_pass_done)) != BFGPU_OK) break;
        } else {
            CU(cudaStreamWaitEvent(ctx->stream, ready[slot], 0));
            if ((rc = ingest_device(ctx, staged[slot], R, cb, /*bitrev=*/true, coef.d, 0, &first_pass_done)) != BFGPU_OK) break;
            CU(cudaEventRecord(consumed[slot], ctx->stream));
            // enqueue the copy after next only now: its wait on consumed[slot] must see this record
            if (b + 1 < nb && b == 0) rc = copy_block(1);
            if (rc == BFGPU_OK && b + 2 < nb) rc = copy_block(b + 2);
            if (rc != BFGPU_OK) break;
        }
        if ((rc = lde_from_bitrev(ctx, coef, added_bits, shift_mont, &blk, /*consume=*/true, lde->d + (uint64_t)start[b] * N, first_pass_done)) != BFGPU_OK) break;
        Phase ph(ctx, BFGPU_PHASE_LEAF);
        cudaStream_t hs = ctx->stream;
        if (from_device) {  // sponge on the second stream, behind this block's LDE
            CU(cudaEventRecord(ready[slot], ctx->stream));
            CU(cudaStreamWaitEvent(ctx->copy_stream, ready[slot], 0));
            hs = ctx->copy_stream;
        }
        hashk::k_leaf_absorb<<<(unsigned)((N + hashk::HASH_THREADS - 1) / hashk::HASH_THREADS), hashk::HASH_THREADS, 0, hs>>>(
            blk.d, N, cb, N, state, b == 0, b + 1 == nb, layer);
        LAUNCHED(ctx);
        CU(cudaGetLastError());
    }
    if (from_device && rc == BFGPU_OK) {  // the tree is built on the compute stream: join
        CU(cudaEventRecord(consumed[0], ctx->copy_stream));
        CU(cudaStreamWaitEvent(ctx->stream, consumed[0], 0));
    }
    if (rc != BFGPU_OK) cudaStreamSynchronize(ctx->copy_stream);
    dfree(ctx, staged[0]);
    dfree(ctx, staged[1]);
    dfree(ctx, state);
    if (rc != BFGPU_OK) {
        dfree(ctx, layer);
        dfree(ctx, lde->d);
        lde->d = nullptr;
        return rc;
    }
    *first_layer = layer;
    return BFGPU_OK;
}

static int32_t pcs_commit_impl(bfgpu_ctx* ctx, const bfgpu_mat* evals, const uint32_t* domain_shifts, int32_t n, uint32_t root[8],
                                    bfgpu_pcs_data** out);
extern "C" int32_t bfgpu_pcs_commit(bfgpu_ctx* ctx, const bfgpu_mat* evals, const uint32_t* domain_shifts, int32_t n, uint32_t root[8],
                                    bfgpu_pcs_data** out) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(pcs_commit_impl(ctx, evals, domain_shifts, n, root, out));
}
static int32_t pcs_commit_impl(bfgpu_ctx* ctx, const bfgpu_mat* evals, const uint32_t* domain_shifts, int32_t n, uint32_t root[8],
                                    bfgpu_pcs_data** out) {
    if (!ctx || !evals || n <= 0 || !root || !out) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    *out = nullptr;
    for (int i = 0; i < n; i++) TRY(check_mat(ctx, &evals[i], true));
    bfgpu_pcs_data* pd = new bfgpu_pcs_data();
    pd->ctx = ctx;
    pd->ldes.resize(n);
    int32_t rc = prestage_all(ctx, evals, n);
    uint32_t gen = kb::to_mont(kb::GEN);
    uint32_t* first_layer = nullptr;
    const bool pipelined = (ctx->input_space == BFGPU_MEM_HOST || ctx->overlap_device) && n == 1 && ctx->pipe_cols >= 8 &&
                           evals[0].cols >= 2 * (uint64_t)ctx->pipe_cols && evals[0].rows * evals[0].cols >= (1ull << 20);
    for (int i = 0; i < n && rc == BFGPU_OK; i++) {
        // shift = GENERATOR / domain.shift  (TwoAdicFriPcs::commit)
        uint32_t shift = gen;
        if (domain_shifts) {
            uint32_t ds = ctx->repr == BFGPU_REPR_CANONICAL ? kb::to_mont(domain_shifts[i] % kb::P) : domain_shifts[i];
            if (ds == 0) rc = fail(ctx, BFGPU_ERR_INVALID, "zero domain shift");
            else shift = kb::mul(gen, kb::inv(ds));
        }
        if (rc == BFGPU_OK && pipelined) rc = commit_host_pipelined(ctx, evals[i], ctx->log_blowup, shift, &pd->ldes[i], &first_layer);
        else if (rc == BFGPU_OK) rc = lde_device(ctx, evals[i], ctx->log_blowup, shift, &pd->ldes[i]);
    }
    prestage_clear(ctx);
    if (rc == BFGPU_OK) rc = build_tree(ctx, pd->ldes, false, &pd->tree, first_layer);
    if (rc == BFGPU_OK) rc = read_digest(ctx, pd->tree->layers.back(), root);
    if (rc != BFGPU_OK) {
        bfgpu_pcs_data_free(pd);
        return rc;
    }
    *out = pd;
    return BFGPU_OK;
}

extern "C" int32_t bfgpu_pcs_num_matrices(const bfgpu_pcs_data* d) { return d ? (int32_t)d->ldes.size() : 0; }
extern "C" int32_t bfgpu_pcs_lde_dims(const bfgpu_pcs_data* d, int32_t idx, uint64_t* rows, uint64_t* cols) {
    if (!d || idx < 0 || (size_t)idx >= d->ldes.size()) return BFGPU_ERR_INVALID;
    if (rows) *rows = d->ldes[idx].rows;
    if (cols) *cols = d->ldes[idx].cols;
    return BFGPU_OK;
}
static int32_t pcs_get_evaluations_impl(bfgpu_pcs_data* d, int32_t idx, int bit_reversed_rows, uint32_t* out);
extern "C" int32_t bfgpu_pcs_get_evaluations(bfgpu_pcs_data* d, int32_t idx, int bit_reversed_rows, uint32_t* out) {
    AllocScope scope(d ? d->ctx : nullptr);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(pcs_get_evaluations_impl(d, idx, bit_reversed_rows, out));
}
static int32_t pcs_get_evaluations_impl(bfgpu_pcs_data* d, int32_t idx, int bit_reversed_rows, uint32_t* out) {
    if (!d) return BFGPU_ERR_INVALID;
    bfgpu_ctx* ctx = d->ctx;
    if (idx < 0 || (size_t)idx >= d->ldes.size() || !out) return fail(ctx, BFGPU_ERR_INVALID, "bad matrix index");
    return egress(ctx, d->ldes[idx], !bit_reversed_rows, out);
}
extern "C" bfgpu_tree* bfgpu_pcs_tree(bfgpu_pcs_data* d) { return d ? d->tree : nullptr; }
extern "C" void bfgpu_pcs_data_free(bfgpu_pcs_data* d) {
    if (!d) return;
    tree_release(d->tree);
    for (DMat& m : d->ldes) dfree(d->ctx, m.d);
    delete d;
}

// =====================================================================================================
// Challenger + Pcs::open
// =====================================================================================================
#include "challenger.h"
#include "kernels_open.cuh"

#include <array>

// the challenger handle remembers the context only for the caller-representation conversions
struct bfgpu_challenger_box {
    bfgpu_challenger ch;
    bfgpu_ctx* ctx;
};
static inline bfgpu_challenger_box* box(bfgpu_challenger* c) { return reinterpret_cast<bfgpu_challenger_box*>(c); }
static inline const bfgpu_challenger_box* box(const bfgpu_challenger* c) { return reinterpret_cast<const bfgpu_challenger_box*>(c); }
static inline uint32_t in_word(const bfgpu_ctx* ctx, uint32_t v) { return ctx->repr == BFGPU_REPR_CANONICAL ? kb::to_mont(v % kb::P) : v; }
static inline uint32_t out_word(const bfgpu_ctx* ctx, uint32_t v) { return ctx->repr == BFGPU_REPR_CANONICAL ? kb::from_mont(v) : v; }

extern "C" int32_t bfgpu_challenger_create(bfgpu_ctx* ctx, bfgpu_challenger** out) {
    if (!ctx || !out) return BFGPU_ERR_INVALID;
    auto* b = new bfgpu_challenger_box();
    b->ctx = ctx;
    *out = reinterpret_cast<bfgpu_challenger*>(b);
    return BFGPU_OK;
}
extern "C" int32_t bfgpu_challenger_clone(const bfgpu_challenger* ch, bfgpu_challenger** out) {
    if (!ch || !out) return BFGPU_ERR_INVALID;
    *out = reinterpret_cast<bfgpu_challenger*>(new bfgpu_challenger_box(*box(ch)));
    return BFGPU_OK;
}
extern "C" void bfgpu_challenger_free(bfgpu_challenger* ch) { delete box(ch); }
extern "C" int32_t bfgpu_challenger_observe(bfgpu_challenger* ch, const uint32_t* values, uint64_t n) {
    if (!ch || (!values && n)) return BFGPU_ERR_INVALID;
    for (uint64_t i = 0; i < n; i++) box(ch)->ch.observe(in_word(box(ch)->ctx, values[i]));
    return BFGPU_OK;
}
extern "C" int32_t bfgpu_challenger_sample(bfgpu_challenger* ch, uint32_t* out, uint64_t n) {
    if (!ch || !out) return BFGPU_ERR_INVALID;
    for (uint64_t i = 0; i < n; i++) out[i] = out_word(box(ch)->ctx, box(ch)->ch.sample());
    return BFGPU_OK;
}
extern "C" int32_t bfgpu_challenger_sample_bits(bfgpu_challenger* ch, uint32_t bits, uint32_t* out) {
    if (!ch || !out || bits > 31) return BFGPU_ERR_INVALID;
    *out = box(ch)->ch.sample_bits(bits);
    return BFGPU_OK;
}
extern "C" int32_t bfgpu_challenger_export(const bfgpu_challenger* ch, uint32_t state[16], uint32_t input[8], uint32_t* n_input,
                                           uint32_t output[8], uint32_t* n_output) {
    if (!ch || !state || !input || !n_input || !output || !n_output) return BFGPU_ERR_INVALID;
    const auto* b = box(ch);
    for (int i = 0; i < 16; i++) state[i] = out_word(b->ctx, b->ch.state[i]);
    *n_input = (uint32_t)b->ch.input.size();
    for (size_t i = 0; i < b->ch.input.size(); i++) input[i] = out_word(b->ctx, b->ch.input[i]);
    *n_output = (uint32_t)b->ch.output.size();
    for (size_t i = 0; i < b->ch.output.size(); i++) output[i] = out_word(b->ctx, b->ch.output[i]);
    return BFGPU_OK;
}
extern "C" int32_t bfgpu_challenger_import(bfgpu_challenger* ch, const uint32_t state[16], const uint32_t* input, uint32_t n_input,
                                           const uint32_t* output, uint32_t n_output) {
    if (!ch || !state || n_input > 8 || n_output > 8) return BFGPU_ERR_INVALID;
    auto* b = box(ch);
    for (int i = 0; i < 16; i++) b->ch.state[i] = in_word(b->ctx, state[i]);
    b->ch.input.clear();
    b->ch.output.clear();
    for (uint32_t i = 0; i < n_input; i++) b->ch.input.push_back(in_word(b->ctx, input[i]));
    for (uint32_t i = 0; i < n_output; i++) b->ch.output.push_back(in_word(b->ctx, output[i]));
    return BFGPU_OK;
}

struct bfgpu_opening {
    std::vector<uint32_t> flat;
};
extern "C" uint64_t bfgpu_opening_size(const bfgpu_opening* o) { return o ? o->flat.size() : 0; }
extern "C" int32_t bfgpu_opening_read(const bfgpu_opening* o, uint32_t* out) {
    if (!o || !out) return BFGPU_ERR_INVALID;
    memcpy(out, o->flat.data(), o->flat.size() * 4);
    return BFGPU_OK;
}
extern "C" void bfgpu_opening_free(bfgpu_opening* o) { delete o; }

static kb::Ext ext_pow(kb::Ext a, uint64_t e) {
    kb::Ext r = kb::ext_one();
    while (e) {
        if (e & 1) r = kb::ext_mul(r, a);
        a = kb::ext_sqr(a);
        e >>= 1;
    }
    return r;
}
struct ExtKey {
    unsigned log_h;
    std::array<uint32_t, 4> z;
    bool operator<(const ExtKey& o) const { return log_h != o.log_h ? log_h < o.log_h : z < o.z; }
};

// Proof of work of the FRI argument (`challenger.grind(bits)`): the witness (canonical) that makes the next sample_bits zero; the
// transcript `ch` observes it.  fixed >= 0 reuses a known witness (pinning against a reference run).
static int32_t pow_grind(bfgpu_ctx* ctx, bfgpu_challenger& ch, int64_t fixed_pow_witness, uint32_t* witness_out) {
    Phase ph(ctx, BFGPU_PHASE_POW);
    if (fixed_pow_witness >= 0) {
        *witness_out = (uint32_t)fixed_pow_witness;
    } else {
        uint32_t st[16];
        memcpy(st, ch.state, sizeof st);
        for (size_t i = 0; i < ch.input.size(); i++) st[i] = ch.input[i];
        uint32_t pos = (uint32_t)ch.input.size();
        uint32_t* d_st = nullptr;
        unsigned int* d_best = nullptr;
        TRY(dalloc(ctx, (void**)&d_st, 64));
        TRY(dalloc(ctx, (void**)&d_best, 4));
        TRY(upload_small(ctx, d_st, st, 64));
        // batches in increasing order keep "the smallest witness"; the first one covers 4x the expected search length
        // (2^bits candidates on average), the following ones are bigger
        const uint32_t mask = (1u << ctx->pow_bits) - 1;
        uint64_t batch = std::min<uint64_t>(std::max<uint64_t>(4ull << ctx->pow_bits, 1u << 14), 1u << 22);
        // BFGPU_OPT_POW_ORDER: 0 = the smallest witness (ascending batches), 1 = the largest one below p (descending batches).
        // The reference's rayon `find_any` returns an arbitrary valid witness; both ends are deterministic.
        const bool desc = ctx->opt[BFGPU_OPT_POW_ORDER] == 1;
        const unsigned int none = desc ? 0u : 0xffffffffu;
        unsigned int best = none;
        for (uint64_t done = 0; done < kb::P && best == none; done += batch, batch = std::min<uint64_t>(batch * 4, 1u << 24)) {
            TRY(upload_small(ctx, d_best, &best, 4));
            uint32_t count = (uint32_t)std::min<uint64_t>(batch, kb::P - done);
            uint32_t start = desc ? (uint32_t)(kb::P - done - count) : (uint32_t)done;
            openk::k_pow_grind<<<(count + 127) / 128, 128, 0, ctx->stream>>>(d_st, pos, mask, start, count, d_best, desc ? 1 : 0);
            LAUNCHED(ctx);
            CU(cudaGetLastError());
            CU(cudaMemcpyAsync(&best, d_best, 4, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaStreamSynchronize(ctx->stream));
        }
        if (desc && best != none) best -= 1;  // the kernel stores w + 1
        else if (desc) best = 0xffffffffu;
        dfree(ctx, d_st);
        dfree(ctx, d_best);
        if (best == 0xffffffffu) { return fail(ctx, BFGPU_ERR_STATE, "proof-of-work search failed"); }
        *witness_out = best;
    }
    if (!ch.check_witness(ctx->pow_bits, kb::to_mont(*witness_out))) { return fail(ctx, BFGPU_ERR_STATE, "invalid proof-of-work witness %u", *witness_out); }
    return BFGPU_OK;
}

// One committed FRI layer: the folded vector it commits to (pairs of extension elements = rows of 8 words) and its Merkle tree.
struct FriLayer {
    uint32_t* vec;  // folded input of this layer: len ext elements = len/2 rows of 8 words
    uint64_t len;
    bfgpu_tree* tree;
};
// FRI commit phase on ONE device from the folded vector `folded` (len extension elements, consumed) down to the final constant:
// commit, observe the root, sample beta, fold, roll in the reduced openings of `reduced` (log height -> ext vector, tallest first,
// entries consumed and set to null) whose length matches.  Appends to layers / commits; the caller releases them.
// (The single-GPU Pcs::open runs all of it here; the sharded prover enters with the vector it gathered below its threshold.)
static int32_t fri_commit_phase(bfgpu_ctx* ctx, bfgpu_challenger& ch, uint32_t* folded, uint64_t len,
                                std::map<unsigned, uint32_t*, std::greater<unsigned>>& reduced, std::vector<FriLayer>& layers,
                                std::vector<std::array<uint32_t, 8>>& commits, uint32_t final_poly[4]) {
    const unsigned log_blowup = ctx->log_blowup;
    using Layer = FriLayer;
    (void)sizeof(Layer);
    Phase ph(ctx, BFGPU_PHASE_FRI);
    auto it = reduced.begin();
    while (it != reduced.end() && (it->second == nullptr || (1ull << it->first) >= len)) ++it;
    // The challenger rides along on the device for the whole commit phase (openk::k_challenger_round, k_fri_tail): rounds
    // are enqueued back to back with no host round trip; all roots come back in ONE copy and the host challenger replays them.
    Scratch fs(ctx);
    uint32_t *d_ch = nullptr, *d_roots = nullptr, *d_betas = nullptr;
    const uint32_t total_rounds = ilog2(len) - log_blowup;
    TRY(fs.alloc((void**)&d_ch, 32 * 4));
    TRY(fs.alloc((void**)&d_roots, (size_t)std::max(total_rounds, 1u) * 32));
    TRY(fs.alloc((void**)&d_betas, (size_t)std::max(total_rounds, 1u) * 16));
    {
        uint32_t h[32] = {0};
        memcpy(h, ch.state, 64);
        for (size_t k = 0; k < ch.input.size(); k++) h[16 + k] = ch.input[k];
        h[24] = (uint32_t)ch.input.size();
        TRY(upload_small(ctx, d_ch, h, sizeof h));
    }
    uint32_t round = 0;
    while (len > (1ull << log_blowup)) {
        if (ctx->fri_tail && len <= (1ull << openk::TAIL_MAX_LOG) && ilog2(len) - log_blowup <= (unsigned)openk::TAIL_MAX_ROUNDS) {
            // ---- all remaining rounds in one single-CTA launch (openk::k_fri_tail) ----
            openk::FriTailArgs ta;
            memset(&ta, 0, sizeof ta);
            ta.log_len = ilog2(len);
            ta.nrounds = ta.log_len - log_blowup;
            ta.tw = ctx->d_tw;
            ta.rollin = (int)ctx->opt[BFGPU_OPT_FRI_ROLLIN];
            ta.ch = d_ch;
            ta.roots = d_roots + 8 * (size_t)round;
            ta.vec[0] = folded;
            int32_t rc = BFGPU_OK;
            for (uint32_t r = 0; r < ta.nrounds && rc == BFGPU_OK; r++) {
                const uint64_t nleaves = len >> (r + 1);
                bfgpu_tree* t = new bfgpu_tree();
                t->ctx = ctx;
                DMat leaves;
                leaves.d = ta.vec[r];
                leaves.rows = nleaves;
                leaves.cols = 8;
                leaves.rs = 8;
                t->mats.push_back(leaves);
                t->log_max = ilog2(nleaves);
                layers.push_back({ta.vec[r], len >> r, t});
                for (unsigned l = 0; l <= t->log_max && rc == BFGPU_OK; l++) {
                    uint32_t* lay = nullptr;
                    rc = dalloc(ctx, (void**)&lay, (nleaves >> l) * 32);
                    t->layers.push_back(lay);
                    t->layer_len.push_back(nleaves >> l);
                    ta.layer[r][l] = lay;
                }
                if (rc == BFGPU_OK) rc = dalloc(ctx, (void**)&ta.vec[r + 1], nleaves * 16);
                if (it != reduced.end() && (1ull << it->first) == nleaves) {
                    ta.add[r] = it->second;
                    ++it;
                }
            }
            if (rc != BFGPU_OK) { return rc; }
            openk::k_fri_tail<<<1, openk::TAIL_THREADS, 0, ctx->stream>>>(ta);
            LAUNCHED(ctx);
            CU(cudaGetLastError());
            for (uint32_t r = 0; r < ta.nrounds; r++)  // the reduced openings consumed by the tail (stream order keeps them alive)
                if (ta.add[r])
                    for (auto& kv : reduced)
                        if (kv.second == ta.add[r]) {
                            dfree(ctx, kv.second);
                            kv.second = nullptr;
                        }
            round += ta.nrounds;
            folded = ta.vec[ta.nrounds];
            len = 1ull << log_blowup;
            break;
        }
        DMat leaves;
        leaves.d = folded;
        leaves.rows = len / 2;
        leaves.cols = 8;
        leaves.rs = 8;
        bfgpu_tree* t = nullptr;
        int32_t rc = build_tree(ctx, {leaves}, false, &t);
        layers.push_back({folded, len, t});
        if (rc != BFGPU_OK) { return rc; }
        openk::k_challenger_round<<<1, 32, 0, ctx->stream>>>(d_ch, t->layers.back(), d_betas + 4 * (size_t)round, d_roots + 8 * (size_t)round);
        LAUNCHED(ctx);
        uint64_t nlen = len / 2;
        unsigned log_nlen = ilog2(nlen);
        uint32_t* next = nullptr;
        TRY(dalloc(ctx, (void**)&next, nlen * 16));
        const uint32_t* add = nullptr;
        if (it != reduced.end() && (1ull << it->first) == nlen) add = it->second;
        openk::k_fri_fold_dev<<<(unsigned)((nlen + 127) / 128), 128, 0, ctx->stream>>>(folded, next, add, log_nlen, d_betas + 4 * (size_t)round, ctx->d_tw,
                                                                                     (int)ctx->opt[BFGPU_OPT_FRI_ROLLIN], 0, (uint32_t)nlen);
        LAUNCHED(ctx);
        CU(cudaGetLastError());
        if (add) {
            dfree(ctx, it->second);
            it->second = nullptr;
            ++it;
        }
        folded = next;
        len = nlen;
        round++;
    }
    std::vector<uint32_t> fin(len * 4);
    {   // one copy for every root of the phase (and the final vector); the host transcript catches up
        std::vector<uint32_t> roots((size_t)round * 8);
        if (round) CU(cudaMemcpyAsync(roots.data(), d_roots, roots.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaMemcpyAsync(fin.data(), folded, len * 16, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        for (uint32_t r = 0; r < round; r++) {
            std::array<uint32_t, 8> root;
            memcpy(root.data(), &roots[8 * r], 32);
            ch.observe_slice(root.data(), 8);
            commits.push_back(root);
            (void)ch.sample_ext();
        }
    }
    if (it != reduced.end()) { return fail(ctx, BFGPU_ERR_STATE, "FRI inputs left over after the commit phase"); }
    dfree(ctx, folded);
    for (uint64_t i = 1; i < len; i++)
        if (memcmp(&fin[0], &fin[4 * i], 16)) { return fail(ctx, BFGPU_ERR_STATE, "FRI final layer is not constant: a committed matrix is not low-degree"); }
    memcpy(final_poly, fin.data(), 16);
    ch.observe_slice(final_poly, 4);
    return BFGPU_OK;
}

static int32_t pcs_open_impl(bfgpu_ctx* ctx, const bfgpu_open_round* rounds, int32_t n_rounds, bfgpu_challenger* chh,
                                  int64_t fixed_pow_witness, bfgpu_opening** out);
extern "C" int32_t bfgpu_pcs_open(bfgpu_ctx* ctx, const bfgpu_open_round* rounds, int32_t n_rounds, bfgpu_challenger* chh,
                                  int64_t fixed_pow_witness, bfgpu_opening** out) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(pcs_open_impl(ctx, rounds, n_rounds, chh, fixed_pow_witness, out));
}
static int32_t pcs_open_impl(bfgpu_ctx* ctx, const bfgpu_open_round* rounds, int32_t n_rounds, bfgpu_challenger* chh,
                                  int64_t fixed_pow_witness, bfgpu_opening** out) {
    if (!ctx || !rounds || n_rounds <= 0 || !chh || !out) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    *out = nullptr;
    bfgpu_challenger& ch = box(chh)->ch;
    const uint32_t gen = kb::to_mont(kb::GEN);
    const unsigned log_blowup = ctx->log_blowup;
    auto res = new bfgpu_opening();
    std::vector<uint32_t>& flat = res->flat;
    struct Guard {
        bfgpu_opening* r;
        bool keep = false;
        ~Guard() { if (!keep) delete r; }
    } guard{res};

    // ---- (i) opened values: barycentric evaluation over the low coset of every matrix -----------------
    struct MatPts {
        const DMat* m;
        std::vector<kb::Ext> pts;
        std::vector<std::vector<kb::Ext>> ys;  // [point][col]
    };
    std::vector<std::vector<MatPts>> R(n_rounds);
    unsigned log_global_max = 0;
    for (int r = 0; r < n_rounds; r++) {
        if (!rounds[r].data || !rounds[r].num_points) return fail(ctx, BFGPU_ERR_INVALID, "null round");
        const uint32_t* pp = rounds[r].points;
        for (size_t i = 0; i < rounds[r].data->ldes.size(); i++) {
            MatPts mp;
            mp.m = &rounds[r].data->ldes[i];
            for (uint32_t t = 0; t < rounds[r].num_points[i]; t++, pp += 4)
                mp.pts.push_back(kb::Ext{{in_word(ctx, pp[0]), in_word(ctx, pp[1]), in_word(ctx, pp[2]), in_word(ctx, pp[3])}});
            log_global_max = std::max(log_global_max, ilog2(mp.m->rows));
            R[r].push_back(std::move(mp));
        }
    }
    {
        Phase ph(ctx, BFGPU_PHASE_OPEN_EVAL);
        std::map<ExtKey, uint32_t*> wcache;
        auto weights = [&](unsigned log_h, const kb::Ext& z, uint32_t** w) -> int32_t {
            ExtKey key{log_h, {z.c[0], z.c[1], z.c[2], z.c[3]}};
            auto it = wcache.find(key);
            if (it == wcache.end()) {
                uint32_t* d = nullptr;
                TRY(dalloc(ctx, (void**)&d, (size_t)16 << log_h));
                uint32_t h = 1u << log_h;
                openk::k_bary_weights<<<(h + 255) / 256, 256, 0, ctx->stream>>>(d, log_h, gen, z, ctx->d_tw, 0, h);
                LAUNCHED(ctx);
                CU(cudaGetLastError());
                it = wcache.emplace(key, d).first;
            }
            *w = it->second;
            return BFGPU_OK;
        };
        // launch every dot product first (results land in one buffer), then a single copy + synchronisation
        struct Job {
            MatPts* mp;
            size_t t0;
            uint32_t np;
            size_t off;  // word offset of this job's sums (cols x np x 4) in sums_all
        };
        std::vector<Job> jobs;
        size_t total_words = 0;
        for (auto& rv : R)
            for (auto& mp : rv)
                for (size_t t0 = 0; t0 < mp.pts.size(); t0 += ctx->bary_points_per_pass) {
                    uint32_t np = (uint32_t)std::min<size_t>(ctx->bary_points_per_pass, mp.pts.size() - t0);
                    jobs.push_back({&mp, t0, np, total_words});
                    total_words += (size_t)mp.m->cols * np * 4;
                }
        uint32_t* sums_all = nullptr;
        TRY(dalloc(ctx, (void**)&sums_all, total_words * 4));
        std::vector<openk::BaryJob> batch[2];  // single-chunk jobs with 1 / 2 opening points
        uint32_t batch_groups[2] = {0, 0};
        for (Job& jb : jobs) {
            const DMat& m = *jb.mp->m;
            uint32_t h = (uint32_t)(m.rows >> log_blowup);
            unsigned log_h = ilog2(h);
            uint32_t nchunks = (h + openk::BARY_ROWS - 1) / openk::BARY_ROWS;
            uint32_t *w0 = nullptr, *w1 = nullptr;
            TRY(weights(log_h, jb.mp->pts[jb.t0], &w0));
            if (jb.np == 2) TRY(weights(log_h, jb.mp->pts[jb.t0 + 1], &w1));
            if (nchunks == 1) {
                batch[jb.np - 1].push_back({m.d, m.rows, w0, w1, sums_all + jb.off, m.cols, h});
                batch_groups[jb.np - 1] = std::max(batch_groups[jb.np - 1], (m.cols + openk::BARY_COLS - 1) / openk::BARY_COLS);
                continue;
            }
            uint32_t* partial = nullptr;
            size_t nsum = (size_t)m.cols * jb.np * 4;
            TRY(dalloc(ctx, (void**)&partial, nsum * nchunks * 4));
            dim3 grid((m.cols + openk::BARY_COLS - 1) / openk::BARY_COLS, nchunks);
            if (jb.np == 1) openk::k_bary_dot<1><<<grid, openk::BARY_THREADS, 0, ctx->stream>>>(m.d, m.rows, m.cols, h, w0, w1, partial, nchunks);
            else openk::k_bary_dot<2><<<grid, openk::BARY_THREADS, 0, ctx->stream>>>(m.d, m.rows, m.cols, h, w0, w1, partial, nchunks);
            LAUNCHED(ctx);
            openk::k_bary_finish<<<(unsigned)((nsum + 127) / 128), 128, 0, ctx->stream>>>(partial, sums_all + jb.off, m.cols, nchunks, jb.np);
            LAUNCHED(ctx);
            CU(cudaGetLastError());
            dfree(ctx, partial);
        }
        for (int k = 0; k < 2; k++) {
            if (batch[k].empty()) continue;
            openk::BaryJob* d_jobs = nullptr;
            TRY(dalloc(ctx, (void**)&d_jobs, batch[k].size() * sizeof(openk::BaryJob)));
            TRY(upload_small(ctx, d_jobs, batch[k].data(), batch[k].size() * sizeof(openk::BaryJob)));
            dim3 grid(batch_groups[k], (unsigned)batch[k].size());
            if (k == 0) openk::k_bary_dot_batch<1><<<grid, openk::BARY_THREADS, 0, ctx->stream>>>(d_jobs);
            else openk::k_bary_dot_batch<2><<<grid, openk::BARY_THREADS, 0, ctx->stream>>>(d_jobs);
            LAUNCHED(ctx);
            CU(cudaGetLastError());
            dfree(ctx, d_jobs);
        }
        std::vector<uint32_t> hs(total_words);
        CU(cudaMemcpyAsync(hs.data(), sums_all, total_words * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        dfree(ctx, sums_all);
        for (Job& jb : jobs) {
            const DMat& m = *jb.mp->m;
            uint32_t h = (uint32_t)(m.rows >> log_blowup);
            jb.mp->ys.resize(jb.mp->pts.size());
            for (uint32_t t = 0; t < jb.np; t++) {
                // p(z) = (z^h - s^h) / (h s^(h-1)) * sum
                const kb::Ext& z = jb.mp->pts[jb.t0 + t];
                kb::Ext zer = ext_pow(z, h);
                zer.c[0] = kb::sub(zer.c[0], kb::pow(gen, h));
                uint32_t den = kb::mul(kb::pow(gen, h - 1), kb::to_mont(h % kb::P));
                kb::Ext scale = kb::ext_scale(zer, kb::inv(den));
                auto& ys = jb.mp->ys[jb.t0 + t];
                ys.resize(m.cols);
                for (uint32_t c = 0; c < m.cols; c++) {
                    const uint32_t* sp = &hs[jb.off + ((size_t)c * jb.np + t) * 4];
                    ys[c] = kb::ext_mul(scale, kb::Ext{{sp[0], sp[1], sp[2], sp[3]}});
                }
            }
        }
        for (auto& kv : wcache) dfree(ctx, kv.second);
    }
    // opened values go to the proof and (Plonky3 "write evaluations to challenger") into the transcript
    for (auto& rv : R)
        for (auto& mp : rv)
            for (auto& ys : mp.ys)
                for (auto& y : ys) {
                    for (int k = 0; k < 4; k++) flat.push_back(out_word(ctx, y.c[k]));
                    if (ctx->opt[BFGPU_OPT_OBSERVE_OPENED_VALUES]) ch.observe_ext(y);
                }
    const kb::Ext alpha = ch.sample_ext();

    // ---- (ii) reduced openings per LDE height ------------------------------------------------------------
    std::map<unsigned, uint32_t*, std::greater<unsigned>> reduced;  // log height -> ext vector, tallest first
    {
        Phase ph(ctx, BFGPU_PHASE_OPEN_REDUCE);
        uint32_t maxw = 1;
        for (auto& rv : R)
            for (auto& mp : rv) maxw = std::max(maxw, mp.m->cols);
        std::vector<kb::Ext> apow(maxw);
        apow[0] = kb::ext_one();
        for (uint32_t k = 1; k < maxw; k++) apow[k] = kb::ext_mul(apow[k - 1], alpha);
        uint32_t* d_apow = nullptr;
        TRY(dalloc(ctx, (void**)&d_apow, (size_t)maxw * 16));
        TRY(upload_small(ctx, d_apow, apow.data(), (size_t)maxw * 16));
        struct Group {
            std::vector<openk::RoMat> mats;
            std::vector<kb::Ext> pts;
            uint64_t num_reduced = 0;
        };
        std::map<unsigned, Group> groups;
        for (auto& rv : R)
            for (auto& mp : rv) {
                unsigned lh = ilog2(mp.m->rows);
                Group& g = groups[lh];
                openk::RoMat rm;
                memset(&rm, 0, sizeof rm);
                rm.d = mp.m->d;
                rm.stride = mp.m->rows;
                rm.width = mp.m->cols;
                if (mp.pts.size() > 2) return fail(ctx, BFGPU_ERR_INVALID, "more than two opening points per matrix are not supported");
                rm.npoints = (uint32_t)mp.pts.size();
                for (size_t t = 0; t < mp.pts.size(); t++) {
                    size_t pi = 0;
                    for (; pi < g.pts.size(); pi++)
                        if (!memcmp(g.pts[pi].c, mp.pts[t].c, 16)) break;
                    if (pi == g.pts.size()) g.pts.push_back(mp.pts[t]);
                    if (g.pts.size() > 4) return fail(ctx, BFGPU_ERR_INVALID, "more than four distinct opening points per height are not supported");
                    rm.pt[t] = (uint32_t)pi;
                    kb::Ext yr = kb::ext_zero();
                    for (uint32_t k = 0; k < mp.m->cols; k++) yr = kb::ext_add(yr, kb::ext_mul(apow[k], mp.ys[t][k]));
                    kb::Ext ao = ext_pow(alpha, g.num_reduced);
                    memcpy(rm.yred[t], yr.c, 16);
                    memcpy(rm.aoff[t], ao.c, 16);
                    g.num_reduced += mp.m->cols;
                }
                g.mats.push_back(rm);
            }
        for (auto& kv : groups) {
            unsigned lh = kv.first;
            Group& g = kv.second;
            openk::RoMat* d_m = nullptr;
            uint32_t *d_z = nullptr, *ro = nullptr;
            TRY(dalloc(ctx, (void**)&d_m, g.mats.size() * sizeof(openk::RoMat)));
            TRY(dalloc(ctx, (void**)&d_z, g.pts.size() * 16));
            TRY(dalloc(ctx, (void**)&ro, (size_t)16 << lh));
            TRY(upload_small(ctx, d_m, g.mats.data(), g.mats.size() * sizeof(openk::RoMat)));
            TRY(upload_small(ctx, d_z, g.pts.data(), g.pts.size() * 16));
            openk::k_reduce_openings<<<((1u << lh) + 127) / 128, 128, 0, ctx->stream>>>(d_m, (uint32_t)g.mats.size(), d_z, (uint32_t)g.pts.size(), d_apow, lh,
                                                                                         gen, ctx->d_tw, ro, 0, 1u << lh);
            LAUNCHED(ctx);
            CU(cudaGetLastError());
            dfree(ctx, d_m);
            dfree(ctx, d_z);
            reduced[lh] = ro;
        }
        dfree(ctx, d_apow);
    }

    // ---- (iii) FRI commit phase ------------------------------------------------------------------------------
    using Layer = FriLayer;
    std::vector<Layer> layers;
    auto release_layers = [&]() {
        for (auto& L : layers) {
            tree_release(L.tree);
            dfree(ctx, L.vec);
        }
        for (auto& kv : reduced) dfree(ctx, kv.second);
    };
    uint32_t final_poly[4];
    const unsigned log_max_height = reduced.begin()->first;
    {
        uint32_t* folded = reduced.begin()->second;
        reduced.begin()->second = nullptr;
        std::vector<std::array<uint32_t, 8>> commits;
        int32_t rc = fri_commit_phase(ctx, ch, folded, 1ull << log_max_height, reduced, layers, commits, final_poly);
        if (rc != BFGPU_OK) { release_layers(); return rc; }
        flat.push_back((uint32_t)commits.size());
        for (auto& c : commits)
            for (int k = 0; k < 8; k++) flat.push_back(out_word(ctx, c[k]));
        for (int k = 0; k < 4; k++) flat.push_back(out_word(ctx, final_poly[k]));
    }

    // ---- (iv) proof of work ----------------------------------------------------------------------------------
    uint32_t witness = 0;
    {
        int32_t rc = pow_grind(ctx, ch, fixed_pow_witness, &witness);
        if (rc != BFGPU_OK) { release_layers(); return rc; }
        flat.push_back(witness);
    }

    // ---- (v) queries: one descriptor template, one kernel (openk::k_answer_queries) -------------------------------------
    {
        Phase ph(ctx, BFGPU_PHASE_QUERY);
        flat.push_back(ctx->num_queries);
        std::vector<openk::QueryWord> tmpl;
        tmpl.push_back({nullptr, 0, 0, 0, 0});  // the query index
        for (int r = 0; r < n_rounds; r++) {
            const bfgpu_tree* t = rounds[r].data->tree;
            const uint32_t down = log_global_max - t->log_max;  // ridx = index >> down
            for (const DMat& m : t->mats)
                for (uint32_t c = 0; c < m.cols; c++)
                    tmpl.push_back({m.d + (uint64_t)c * m.col_stride(), m.rs, log_global_max - ilog2(m.rows), 0, 0});
            for (unsigned l = 0; l < t->log_max; l++)
                for (uint32_t k = 0; k < 8; k++) tmpl.push_back({t->layers[l] + k, 8, down + l, 1, 0});
        }
        for (size_t i = 0; i < layers.size(); i++) {
            for (uint32_t k = 0; k < 4; k++) tmpl.push_back({layers[i].vec + k, 4, (uint32_t)i, 1, 0});  // 8*pair + 4*((idx^1)&1) = 4*(idx^1)
            const bfgpu_tree* t = layers[i].tree;
            for (unsigned l = 0; l < t->log_max; l++)
                for (uint32_t k = 0; k < 8; k++) tmpl.push_back({t->layers[l] + k, 8, (uint32_t)(i + 1 + l), 1, 0});
        }
        std::vector<uint32_t> indices(ctx->num_queries);
        for (uint32_t q = 0; q < ctx->num_queries; q++) indices[q] = ch.sample_bits(log_max_height);
        const uint32_t per_query = (uint32_t)tmpl.size();
        const size_t total = (size_t)per_query * ctx->num_queries;
        Scratch scratch(ctx);
        openk::QueryWord* d_tmpl = nullptr;
        uint32_t *d_idx = nullptr, *d_out = nullptr;
        TRY(scratch.alloc((void**)&d_tmpl, tmpl.size() * sizeof(openk::QueryWord)));
        TRY(scratch.alloc((void**)&d_idx, indices.size() * 4 + 4));
        TRY(scratch.alloc((void**)&d_out, total * 4 + 4));
        TRY(upload_small(ctx, d_tmpl, tmpl.data(), tmpl.size() * sizeof(openk::QueryWord)));
        TRY(upload_small(ctx, d_idx, indices.data(), indices.size() * 4));
        if (total) {
            openk::k_answer_queries<<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(d_tmpl, per_query, d_idx, ctx->num_queries, d_out,
                                                                                             ctx->repr == BFGPU_REPR_CANONICAL);
            LAUNCHED(ctx);
            CU(cudaGetLastError());
            const size_t base = flat.size();
            flat.resize(base + total);
            CU(cudaMemcpyAsync(flat.data() + base, d_out, total * 4, cudaMemcpyDeviceToHost, ctx->stream));
        }
        CU(cudaStreamSynchronize(ctx->stream));
    }
    release_layers();
    guard.keep = true;
    *out = res;
    return BFGPU_OK;
}

// =====================================================================================================
// MachineProver: setup / commit / open over the eight-chip Brainfuck machine
// (reference crates/stark/src/machine.rs:154-224, crates/stark/src/prover.rs:209-236,242-553)
// =====================================================================================================
#include "kernels_air.cuh"

struct bfgpu_pk {
    bfgpu_ctx* ctx = nullptr;
    std::vector<std::string> names;  // sorted by (height desc, name)
    std::vector<int> chip;           // index into air::CHIPS
    std::vector<DMat> traces;        // ingested traces: column-major, bit-reversed rows (read by the LogUp kernel)
    bfgpu_pcs_data* data = nullptr;
    uint32_t commit[8];              // Montgomery
};
struct bfgpu_shard {
    bfgpu_ctx* ctx = nullptr;
    std::vector<std::string> names;
    std::vector<int> chip;
    std::vector<DMat> traces;
    bfgpu_pcs_data* data = nullptr;
    uint32_t commit[8];
};
struct bfgpu_shard_proof {
    std::vector<uint32_t> flat;
};

static int chip_index(const char* name) {
    for (int i = 0; i < air::NUM_CHIPS; i++)
        if (!strcmp(name, air::CHIPS[i].name)) return i;
    return -1;
}

// sort by (Reverse(height), name) (prover.rs:214, machine.rs:182-183), ingest + LDE + Merkle, keep the traces
static int32_t machine_commit(bfgpu_ctx* ctx, const char* const* names, const bfgpu_mat* mats, int32_t n, bool preprocessed,
                              std::vector<std::string>* out_names, std::vector<int>* out_chip, std::vector<DMat>* out_traces,
                              bfgpu_pcs_data** out_data, uint32_t root_mont[8]) {
    std::vector<int> order(n);
    for (int i = 0; i < n; i++) {
        TRY(check_mat(ctx, &mats[i], true));
        int ci = chip_index(names[i]);
        if (ci < 0) return fail(ctx, BFGPU_ERR_INVALID, "unknown chip '%s'", names[i]);
        uint32_t want = preprocessed ? air::CHIPS[ci].prep_w : air::CHIPS[ci].main_w;
        if (mats[i].cols != want) return fail(ctx, BFGPU_ERR_INVALID, "chip %s: trace width %llu, expected %u", names[i], (unsigned long long)mats[i].cols, want);
        order[i] = i;
    }
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        if (mats[a].rows != mats[b].rows) return mats[a].rows > mats[b].rows;
        return strcmp(names[a], names[b]) < 0;
    });
    bfgpu_pcs_data* pd = new bfgpu_pcs_data();
    pd->ctx = ctx;
    pd->ldes.resize(n);
    out_traces->resize(n);
    // copies in commit order, so the first LDE can start as soon as its own matrix has arrived
    std::vector<bfgpu_mat> in_order(n);
    for (int k = 0; k < n; k++) in_order[k] = mats[order[k]];
    int32_t rc = prestage_all(ctx, in_order.data(), n);
    const uint32_t gen = kb::to_mont(kb::GEN);
    std::vector<DMat> coefs(n);
    for (int k = 0; k < n && rc == BFGPU_OK; k++) {  // ingest (+ the copy the LogUp kernel reads later); the LDEs follow in one batch
        int i = order[k];
        out_names->push_back(names[i]);
        out_chip->push_back(chip_index(names[i]));
        if (ilog2(mats[i].rows) + ctx->log_blowup > (unsigned)kb::TWO_ADICITY) rc = fail(ctx, BFGPU_ERR_INVALID, "LDE height exceeds the field's two-adicity");
        if (rc == BFGPU_OK) rc = ingest(ctx, mats[i], /*bitrev=*/true, &coefs[k]);
        if (rc == BFGPU_OK) {
            DMat& keep = (*out_traces)[k];
            keep = coefs[k];
            const size_t bytes = (size_t)keep.rows * keep.cols * 4;
            rc = dalloc(ctx, (void**)&keep.d, bytes);
            if (rc == BFGPU_OK && cudaMemcpyAsync(keep.d, coefs[k].d, bytes, cudaMemcpyDeviceToDevice, ctx->stream) != cudaSuccess)
                rc = fail(ctx, BFGPU_ERR_CUDA, "trace copy failed");
        }
    }
    if (rc == BFGPU_OK) rc = lde_many(ctx, coefs, ctx->log_blowup, std::vector<uint32_t>(n, gen), &pd->ldes);
    for (DMat& c : coefs) dfree(ctx, c.d);  // only non-null after an error
    prestage_clear(ctx);
    if (rc == BFGPU_OK) rc = build_tree(ctx, pd->ldes, false, &pd->tree);
    if (rc == BFGPU_OK) {
        CU(cudaMemcpyAsync(root_mont, pd->tree->layers.back(), 32, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    if (rc != BFGPU_OK) {
        bfgpu_pcs_data_free(pd);
        for (DMat& m : *out_traces) dfree(ctx, m.d);
        return rc;
    }
    *out_data = pd;
    return BFGPU_OK;
}

static int32_t machine_setup_impl(bfgpu_ctx* ctx, const char* const* names, const bfgpu_mat* prep_traces, int32_t n, uint32_t commit[8],
                                       bfgpu_pk** out);
extern "C" int32_t bfgpu_machine_setup(bfgpu_ctx* ctx, const char* const* names, const bfgpu_mat* prep_traces, int32_t n, uint32_t commit[8],
                                       bfgpu_pk** out) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(machine_setup_impl(ctx, names, prep_traces, n, commit, out));
}
static int32_t machine_setup_impl(bfgpu_ctx* ctx, const char* const* names, const bfgpu_mat* prep_traces, int32_t n, uint32_t commit[8],
                                       bfgpu_pk** out) {
    if (!ctx || !names || !prep_traces || n <= 0 || !commit || !out) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    auto* pk = new bfgpu_pk();
    pk->ctx = ctx;
    int32_t rc = machine_commit(ctx, names, prep_traces, n, true, &pk->names, &pk->chip, &pk->traces, &pk->data, pk->commit);
    if (rc != BFGPU_OK) {
        delete pk;
        return rc;
    }
    for (int i = 0; i < 8; i++) commit[i] = out_word(ctx, pk->commit[i]);
    *out = pk;
    return BFGPU_OK;
}
extern "C" void bfgpu_pk_free(bfgpu_pk* pk) {
    if (!pk) return;
    bfgpu_pcs_data_free(pk->data);
    for (DMat& m : pk->traces) dfree(pk->ctx, m.d);
    delete pk;
}
// StarkProvingKey::observe_into (prover.rs:595-601): the commitment then 7 zero elements
extern "C" int32_t bfgpu_pk_observe_into(const bfgpu_pk* pk, bfgpu_challenger* ch) {
    if (!pk || !ch) return BFGPU_ERR_INVALID;
    box(ch)->ch.observe_slice(pk->commit, 8);
    for (int i = 0; i < 7; i++) box(ch)->ch.observe(0);
    return BFGPU_OK;
}

static int32_t machine_commit_impl(bfgpu_ctx* ctx, const char* const* names, const bfgpu_mat* traces, int32_t n, uint32_t root[8],
                                        bfgpu_shard** out);
extern "C" int32_t bfgpu_machine_commit(bfgpu_ctx* ctx, const char* const* names, const bfgpu_mat* traces, int32_t n, uint32_t root[8],
                                        bfgpu_shard** out) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(machine_commit_impl(ctx, names, traces, n, root, out));
}
static int32_t machine_commit_impl(bfgpu_ctx* ctx, const char* const* names, const bfgpu_mat* traces, int32_t n, uint32_t root[8],
                                        bfgpu_shard** out) {
    if (!ctx || !names || !traces || n <= 0 || !root || !out) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    auto* sd = new bfgpu_shard();
    sd->ctx = ctx;
    int32_t rc = machine_commit(ctx, names, traces, n, false, &sd->names, &sd->chip, &sd->traces, &sd->data, sd->commit);
    if (rc != BFGPU_OK) {
        delete sd;
        return rc;
    }
    for (int i = 0; i < 8; i++) root[i] = out_word(ctx, sd->commit[i]);
    *out = sd;
    return BFGPU_OK;
}
extern "C" void bfgpu_shard_free(bfgpu_shard* sd) {
    if (!sd) return;
    bfgpu_pcs_data_free(sd->data);
    for (DMat& m : sd->traces) dfree(sd->ctx, m.d);
    delete sd;
}

// inclusive scan of n ext elements in place (recursive block scan)
static int32_t scan_ext(bfgpu_ctx* ctx, uint32_t* data, uint64_t n) {
    uint64_t nb = (n + air::SCAN_BLOCK - 1) / air::SCAN_BLOCK;
    if (nb <= 1) {
        air::k_scan_blocks<<<1, air::SCAN_THREADS, 0, ctx->stream>>>((uint4*)data, n, nullptr);
        LAUNCHED(ctx);
        CU(cudaGetLastError());
        return BFGPU_OK;
    }
    uint32_t* totals = nullptr;
    TRY(dalloc(ctx, (void**)&totals, nb * 16));
    air::k_scan_blocks<<<(unsigned)nb, air::SCAN_THREADS, 0, ctx->stream>>>((uint4*)data, n, (uint4*)totals);
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    TRY(scan_ext(ctx, totals, nb));
    air::k_scan_add<<<(unsigned)((n + air::SCAN_THREADS - 1) / air::SCAN_THREADS), air::SCAN_THREADS, 0, ctx->stream>>>((uint4*)data, n, (const uint4*)totals);
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    dfree(ctx, totals);
    return BFGPU_OK;
}

// commit to device matrices given column-major with bit-reversed rows (consumed); lde shift per matrix
static int32_t commit_bitrev_device(bfgpu_ctx* ctx, std::vector<DMat>& coefs, const std::vector<uint32_t>& shift_mont, bfgpu_pcs_data** out,
                                    uint32_t root_mont[8]) {
    bfgpu_pcs_data* pd = new bfgpu_pcs_data();
    pd->ctx = ctx;
    int32_t rc = lde_many(ctx, coefs, ctx->log_blowup, shift_mont, &pd->ldes);
    if (rc == BFGPU_OK) rc = build_tree(ctx, pd->ldes, false, &pd->tree);
    if (rc == BFGPU_OK) {
        CU(cudaMemcpyAsync(root_mont, pd->tree->layers.back(), 32, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    if (rc != BFGPU_OK) {
        bfgpu_pcs_data_free(pd);
        return rc;
    }
    *out = pd;
    return BFGPU_OK;
}

// LogUp permutation traces of every chip (prover.rs:280-296 -> permutation.rs:75-148): perm[i] = n x 4*perm_w base columns in the
// prover's layout; the cumulative sums (last running totals) are parked at d_csums[4 i ..] for ONE later copy.
static int32_t perm_traces(bfgpu_ctx* ctx, const bfgpu_pk* pk, const std::vector<int>& pk_idx, const std::vector<int>& chips, const std::vector<DMat>& traces,
                           const air::Challenges& chal, std::vector<DMat>* perm_out, uint32_t* d_csums) {
    std::vector<DMat>& perm = *perm_out;
    const size_t nchips = chips.size();
    Phase ph(ctx, BFGPU_PHASE_PERM);
    for (size_t i = 0; i < nchips; i++) {
        const air::ChipInfo& ci = air::CHIPS[chips[i]];
        const DMat& main = traces[i];
        uint64_t n = main.rows;
        unsigned log_n = ilog2(n);
        perm[i].rows = n;
        perm[i].cols = 4 * ci.perm_w;
        TRY(dalloc(ctx, (void**)&perm[i].d, n * perm[i].cols * 4));
        uint32_t* rowsum = nullptr;
        TRY(dalloc(ctx, (void**)&rowsum, n * 16));
        const uint32_t* prep = pk_idx[i] >= 0 ? pk->traces[pk_idx[i]].d : nullptr;
#define BF_PERM_CASE(C) \
    case C: air::k_perm_rows<C><<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(C, main.d, prep, log_n, chal, ci.perm_w, perm[i].d, rowsum); break;
        switch (chips[i]) {
            BF_PERM_CASE(0) BF_PERM_CASE(1) BF_PERM_CASE(2) BF_PERM_CASE(3) BF_PERM_CASE(4) BF_PERM_CASE(5) BF_PERM_CASE(6) BF_PERM_CASE(7)
        }
#undef BF_PERM_CASE
        LAUNCHED(ctx);
        CU(cudaGetLastError());
        TRY(scan_ext(ctx, rowsum, n));
        air::k_scan_fixup<<<(unsigned)((n + air::SCAN_THREADS - 1) / air::SCAN_THREADS), air::SCAN_THREADS, 0, ctx->stream>>>(
            (const uint4*)rowsum, n, nullptr, log_n, perm[i].d + (uint64_t)4 * (ci.perm_w - 1) * n);
        LAUNCHED(ctx);
        CU(cudaGetLastError());
        // cumulative sum = last running total: parked on the device, fetched with ONE copy after the permutation commit
        // (a device->host copy into pageable memory blocks the host: eight of them plus a synchronisation cost more than
        // the kernels of a small proof)
        CU(cudaMemcpyAsync(d_csums + 4 * i, rowsum + 4 * (n - 1), 16, cudaMemcpyDeviceToDevice, ctx->stream));
        dfree(ctx, rowsum);  // stream-ordered reuse: the copy above is enqueued before any later writer
    }
    return BFGPU_OK;
}

// CpuProver::open (prover.rs:242-553)
static int32_t machine_open_impl(bfgpu_ctx* ctx, const bfgpu_pk* pk, const bfgpu_shard* sd, bfgpu_challenger* chh, int64_t fixed_pow_witness,
                                      bfgpu_shard_proof** out);
extern "C" int32_t bfgpu_machine_open(bfgpu_ctx* ctx, const bfgpu_pk* pk, const bfgpu_shard* sd, bfgpu_challenger* chh, int64_t fixed_pow_witness,
                                      bfgpu_shard_proof** out) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(machine_open_impl(ctx, pk, sd, chh, fixed_pow_witness, out));
}
static int32_t machine_open_impl(bfgpu_ctx* ctx, const bfgpu_pk* pk, const bfgpu_shard* sd, bfgpu_challenger* chh, int64_t fixed_pow_witness,
                                      bfgpu_shard_proof** out) {
    if (!ctx || !pk || !sd || !chh || !out) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    *out = nullptr;
    bfgpu_challenger& ch = box(chh)->ch;
    const size_t nchips = sd->names.size();
    const uint32_t gen = kb::to_mont(kb::GEN);
    if (ctx->log_blowup != 1) return fail(ctx, BFGPU_ERR_INVALID, "the machine prover requires log_blowup = 1 (kb31_poseidon2.rs:63)");
    // pk matrix index of every chip (or -1)
    std::vector<int> pk_idx(nchips, -1);
    for (size_t i = 0; i < nchips; i++)
        for (size_t k = 0; k < pk->names.size(); k++)
            if (pk->names[k] == sd->names[i]) pk_idx[i] = (int)k;
    for (size_t i = 0; i < nchips; i++) {
        const air::ChipInfo& ci = air::CHIPS[sd->chip[i]];
        if (ci.log_quotient_degree != 1) return fail(ctx, BFGPU_ERR_STATE, "chip %s: unsupported quotient degree", ci.name);
        if (ci.prep_w && (pk_idx[i] < 0 || pk->traces[pk_idx[i]].rows != sd->traces[i].rows))
            return fail(ctx, BFGPU_ERR_INVALID, "chip %s: preprocessed trace missing or of a different height", ci.name);
    }
    // ---- transcript: main commitment, LogUp challenges (prover.rs:266-272) ----------------------------------------
    ch.observe_slice(sd->commit, 8);
    air::Challenges chal;
    chal.alpha = ch.sample_ext();
    kb::Ext beta = ch.sample_ext();
    chal.beta_pow[0] = kb::ext_one();
    for (int k = 1; k < 8; k++) chal.beta_pow[k] = kb::ext_mul(chal.beta_pow[k - 1], beta);
    chal.cumulative_sum = kb::ext_zero();

    // ---- permutation traces (prover.rs:280-296 -> permutation.rs:75-148) --------------------------------------------
    std::vector<DMat> perm(nchips);
    std::vector<kb::Ext> csum(nchips);
    Scratch csum_scratch(ctx);
    uint32_t* d_csums = nullptr;
    TRY(csum_scratch.alloc((void**)&d_csums, nchips * 16));
    TRY(perm_traces(ctx, pk, pk_idx, sd->chip, sd->traces, chal, &perm, d_csums));
    bfgpu_pcs_data* perm_data = nullptr;
    uint32_t perm_root[8];
    {
        std::vector<uint32_t> shifts(nchips, gen);
        TRY(commit_bitrev_device(ctx, perm, shifts, &perm_data, perm_root));
    }
    struct Cleanup {
        bfgpu_pcs_data *a = nullptr, *b = nullptr;
        ~Cleanup() { bfgpu_pcs_data_free(a); bfgpu_pcs_data_free(b); }
    } cleanup;
    cleanup.a = perm_data;
    CU(cudaMemcpy(csum.data(), d_csums, nchips * 16, cudaMemcpyDeviceToHost));  // the stream is idle: the commit just returned its root
    ch.observe_slice(perm_root, 8);
    for (size_t i = 0; i < nchips; i++) ch.observe_ext(csum[i]);

    // ---- quotient values (prover.rs:343-388 -> quotient.rs:18-165) ---------------------------------------------------
    const kb::Ext alpha = ch.sample_ext();
    std::vector<DMat> qchunks;
    std::vector<uint32_t> qshifts;
    {
        Phase ph(ctx, BFGPU_PHASE_QUOTIENT);
        std::vector<kb::Ext> apow(air::MAX_CONSTRAINTS);
        apow[0] = kb::ext_one();
        for (int k = 1; k < air::MAX_CONSTRAINTS; k++) apow[k] = kb::ext_mul(apow[k - 1], alpha);
        kb::Ext* d_apow = nullptr;
        TRY(dalloc(ctx, (void**)&d_apow, apow.size() * sizeof(kb::Ext)));
        TRY(upload_small(ctx, d_apow, apow.data(), apow.size() * sizeof(kb::Ext)));
        for (size_t i = 0; i < nchips; i++) {
            const air::ChipInfo& ci = air::CHIPS[sd->chip[i]];
            unsigned log_n = ilog2(sd->traces[i].rows);
            uint64_t n = 1ull << log_n;
            air::QuotientArgs qa;
            qa.chip = sd->chip[i];
            qa.main = sd->data->ldes[i].d;
            qa.prep = pk_idx[i] >= 0 ? pk->data->ldes[pk_idx[i]].d : nullptr;
            qa.perm = perm_data->ldes[i].d;
            qa.log_n = log_n;
            qa.lqd = 1;
            qa.shift = gen;
            qa.g_inv = kb::inv(kb::two_adic_generator(log_n));
            uint32_t sn = kb::pow(gen, n);
            qa.zh[0] = kb::sub(sn, kb::ONE);
            qa.zh[1] = kb::sub(kb::neg(sn), kb::ONE);
            qa.zh_inv[0] = kb::inv(qa.zh[0]);
            qa.zh_inv[1] = kb::inv(qa.zh[1]);
            qa.apow = d_apow;
            qa.tw = ctx->d_tw;
            uint32_t* q = nullptr;
            TRY(dalloc(ctx, (void**)&q, 2 * n * 16));
            qa.out = q;
            air::Challenges c2 = chal;
            c2.cumulative_sum = csum[i];
#define BF_QUOT_CASE(C) \
    case C: air::k_quotient<C><<<(unsigned)((2 * n + 127) / 128), 128, 0, ctx->stream>>>(qa, c2); break;
            switch (qa.chip) {
                BF_QUOT_CASE(0) BF_QUOT_CASE(1) BF_QUOT_CASE(2) BF_QUOT_CASE(3) BF_QUOT_CASE(4) BF_QUOT_CASE(5) BF_QUOT_CASE(6) BF_QUOT_CASE(7)
            }
#undef BF_QUOT_CASE
            LAUNCHED(ctx);
            CU(cudaGetLastError());
            // split_evals / split_domains (prover.rs:391-402): chunk c lives on the coset 3 w_{2n}^c H, LDE shift = GEN / that
            uint32_t w2n = kb::two_adic_generator(log_n + 1);
            for (int c = 0; c < 2; c++) {
                DMat m;
                m.rows = n;
                m.cols = 4;
                TRY(dalloc(ctx, (void**)&m.d, n * 16));
                CU(cudaMemcpyAsync(m.d, q + (uint64_t)c * 4 * n, n * 16, cudaMemcpyDeviceToDevice, ctx->stream));
                qchunks.push_back(m);
                qshifts.push_back(c == 0 ? kb::ONE : kb::inv(w2n));
            }
            dfree(ctx, q);
            (void)ci;
        }
        dfree(ctx, d_apow);  // stream order keeps it alive for the kernels above; no host synchronisation needed
    }
    bfgpu_pcs_data* quot_data = nullptr;
    uint32_t quot_root[8];
    TRY(commit_bitrev_device(ctx, qchunks, qshifts, &quot_data, quot_root));
    cleanup.b = quot_data;
    ch.observe_slice(quot_root, 8);

    // ---- opening points (prover.rs:415-458) and Pcs::open -----------------------------------------------------------------
    const kb::Ext zeta = ch.sample_ext();
    auto push_ext = [&](std::vector<uint32_t>& v, const kb::Ext& e) {
        for (int k = 0; k < 4; k++) v.push_back(out_word(ctx, e.c[k]));
    };
    auto next_point = [&](unsigned log_n) { return kb::ext_scale(zeta, kb::two_adic_generator(log_n)); };
    std::vector<uint32_t> np[4], pts[4];
    for (size_t k = 0; k < pk->names.size(); k++) {
        bool both = !air::CHIPS[pk->chip[k]].local_only;
        np[0].push_back(both ? 2 : 1);
        push_ext(pts[0], zeta);
        if (both) push_ext(pts[0], next_point(ilog2(pk->traces[k].rows)));
    }
    for (size_t i = 0; i < nchips; i++) {
        unsigned log_n = ilog2(sd->traces[i].rows);
        bool both = !air::CHIPS[sd->chip[i]].local_only;
        np[1].push_back(both ? 2 : 1);
        push_ext(pts[1], zeta);
        if (both) push_ext(pts[1], next_point(log_n));
        np[2].push_back(2);
        push_ext(pts[2], zeta);
        push_ext(pts[2], next_point(log_n));
        for (int c = 0; c < 2; c++) {
            np[3].push_back(1);
            push_ext(pts[3], zeta);
        }
    }
    bfgpu_open_round rounds[4] = {{pk->data, np[0].data(), pts[0].data()},
                                  {sd->data, np[1].data(), pts[1].data()},
                                  {perm_data, np[2].data(), pts[2].data()},
                                  {quot_data, np[3].data(), pts[3].data()}};
    bfgpu_opening* op = nullptr;
    TRY(bfgpu_pcs_open(ctx, rounds, 4, chh, fixed_pow_witness, &op));

    // ---- ShardProof (types.rs:32-73): commitments, per-chip (index, log_degree, cumulative sum), opening -------------------
    auto* proof = new bfgpu_shard_proof();
    auto& flat = proof->flat;
    for (int k = 0; k < 8; k++) flat.push_back(out_word(ctx, sd->commit[k]));
    for (int k = 0; k < 8; k++) flat.push_back(out_word(ctx, perm_root[k]));
    for (int k = 0; k < 8; k++) flat.push_back(out_word(ctx, quot_root[k]));
    flat.push_back((uint32_t)nchips);
    for (size_t i = 0; i < nchips; i++) {
        flat.push_back((uint32_t)sd->chip[i]);
        flat.push_back(ilog2(sd->traces[i].rows));
        for (int k = 0; k < 4; k++) flat.push_back(out_word(ctx, csum[i].c[k]));
    }
    flat.insert(flat.end(), op->flat.begin(), op->flat.end());
    bfgpu_opening_free(op);
    *out = proof;
    return BFGPU_OK;
}
extern "C" uint64_t bfgpu_shard_proof_size(const bfgpu_shard_proof* p) { return p ? p->flat.size() : 0; }
extern "C" int32_t bfgpu_shard_proof_read(const bfgpu_shard_proof* p, uint32_t* out) {
    if (!p || !out) return BFGPU_ERR_INVALID;
    memcpy(out, p->flat.data(), p->flat.size() * 4);
    return BFGPU_OK;
}
extern "C" void bfgpu_shard_proof_free(bfgpu_shard_proof* p) { delete p; }
extern "C" int32_t bfgpu_machine_num_chips(void) { return air::NUM_CHIPS; }
extern "C" int32_t bfgpu_machine_chip_info(int32_t i, const char** name, int32_t* main_w, int32_t* prep_w, int32_t* perm_w, int32_t* local_only) {
    if (i < 0 || i >= air::NUM_CHIPS) return BFGPU_ERR_INVALID;
    if (name) *name = air::CHIPS[i].name;
    if (main_w) *main_w = air::CHIPS[i].main_w;
    if (prep_w) *prep_w = air::CHIPS[i].prep_w;
    if (perm_w) *perm_w = air::CHIPS[i].perm_w;
    if (local_only) *local_only = air::CHIPS[i].local_only;
    return BFGPU_OK;
}

// ---- plug point #2: the pieces of CpuProver::open a Plonky3-trait-level integration calls one by one (SURVEY.md §8b) -------------
// Pcs::get_evaluations_on_domain as a DEVICE VIEW (prover.rs:365-373): the committed LDE stays in HBM; the caller gets the pointer
// and the layout (column-major, `col_stride` words between columns, rows in bit-reversed order, Montgomery words).
extern "C" int32_t bfgpu_pcs_lde_device(const bfgpu_pcs_data* d, int32_t idx, const uint32_t** dev, uint64_t* rows, uint64_t* cols, uint64_t* col_stride) {
    if (!d || idx < 0 || (size_t)idx >= d->ldes.size() || !dev) return BFGPU_ERR_INVALID;
    const DMat& m = d->ldes[idx];
    *dev = m.d;
    if (rows) *rows = m.rows;
    if (cols) *cols = m.cols;
    if (col_stride) *col_stride = m.col_stride();
    return BFGPU_OK;
}

// Chip::generate_permutation_trace (chip.rs:117-136 -> permutation.rs:75-148) for ONE chip: main (and preprocessed) trace in, the
// LogUp trace (rows x 4*perm_width base columns, row-major, natural rows: the flattened form prover.rs:318-328 commits) and the
// cumulative sum out.  challenges = alpha (4 words) then beta (4 words).
static int32_t logup_perm_trace_impl(bfgpu_ctx* ctx, const char* chip, const bfgpu_mat* main, const bfgpu_mat* prep, const uint32_t challenges[8],
                                     uint32_t* perm_out, uint32_t cum_sum[4]);
extern "C" int32_t bfgpu_logup_perm_trace(bfgpu_ctx* ctx, const char* chip, const bfgpu_mat* main, const bfgpu_mat* prep, const uint32_t challenges[8],
                                          uint32_t* perm_out, uint32_t cum_sum[4]) {
    AllocScope scope(ctx);
    return scope.ok(logup_perm_trace_impl(ctx, chip, main, prep, challenges, perm_out, cum_sum));
}
static int32_t logup_perm_trace_impl(bfgpu_ctx* ctx, const char* chip, const bfgpu_mat* main, const bfgpu_mat* prep, const uint32_t challenges[8],
                                     uint32_t* perm_out, uint32_t cum_sum[4]) {
    if (!ctx || !chip || !main || !challenges || !perm_out || !cum_sum) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    const int ci = chip_index(chip);
    if (ci < 0) return fail(ctx, BFGPU_ERR_INVALID, "unknown chip '%s'", chip);
    const air::ChipInfo& info = air::CHIPS[ci];
    TRY(check_mat(ctx, main, true));
    if (main->cols != (uint64_t)info.main_w) return fail(ctx, BFGPU_ERR_INVALID, "chip %s: main trace width %llu, expected %d", chip, (unsigned long long)main->cols, info.main_w);
    if (info.prep_w) {
        if (!prep) return fail(ctx, BFGPU_ERR_INVALID, "chip %s needs its preprocessed trace", chip);
        TRY(check_mat(ctx, prep, true));
        if (prep->cols != (uint64_t)info.prep_w || prep->rows != main->rows) return fail(ctx, BFGPU_ERR_INVALID, "chip %s: bad preprocessed trace shape", chip);
    }
    if (info.perm_w == 0) return fail(ctx, BFGPU_ERR_INVALID, "chip %s has no lookups", chip);
    Scratch sc(ctx);
    bfgpu_pk tmp;  // carrier for perm_traces(): just the preprocessed trace
    tmp.ctx = ctx;
    std::vector<DMat> mains(1), perm(1);
    TRY(ingest(ctx, *main, /*bitrev=*/true, &mains[0]));
    sc.bufs.push_back(mains[0].d);
    std::vector<int> pk_idx(1, -1);
    if (info.prep_w) {
        DMat p;
        TRY(ingest(ctx, *prep, /*bitrev=*/true, &p));
        sc.bufs.push_back(p.d);
        tmp.traces.push_back(p);
        pk_idx[0] = 0;
    }
    air::Challenges chal;
    for (int k = 0; k < 4; k++) chal.alpha.c[k] = in_word(ctx, challenges[k]);
    kb::Ext beta;
    for (int k = 0; k < 4; k++) beta.c[k] = in_word(ctx, challenges[4 + k]);
    chal.beta_pow[0] = kb::ext_one();
    for (int k = 1; k < 8; k++) chal.beta_pow[k] = kb::ext_mul(chal.beta_pow[k - 1], beta);
    chal.cumulative_sum = kb::ext_zero();
    uint32_t* d_csum = nullptr;
    TRY(sc.alloc((void**)&d_csum, 16));
    TRY(perm_traces(ctx, &tmp, pk_idx, {ci}, mains, chal, &perm, d_csum));
    sc.bufs.push_back(perm[0].d);
    uint32_t cs[4];
    CU(cudaMemcpyAsync(cs, d_csum, 16, cudaMemcpyDeviceToHost, ctx->stream));
    TRY(egress(ctx, perm[0], /*bitrev=*/true, perm_out));  // synchronises
    for (int k = 0; k < 4; k++) cum_sum[k] = out_word(ctx, cs[k]);
    return BFGPU_OK;
}

// quotient_values (quotient.rs:18-165) for ONE chip from the COMMITTED LDEs (device resident: nothing is copied back to evaluate):
// out = 2^(log_n + 1) extension elements (4 words each), the quotient values over the quotient domain in NATURAL order, exactly the
// Vec<Challenge> the reference then flattens and splits (prover.rs:391-402).  prep_data / prep_idx: -1 / NULL for chips without a
// preprocessed trace.  alpha: constraint-folding challenge; perm_challenges: LogUp alpha, beta; cum_sum: the chip's cumulative sum.
static int32_t quotient_values_impl(bfgpu_ctx* ctx, const char* chip, const bfgpu_pcs_data* prep_data, int32_t prep_idx, const bfgpu_pcs_data* main_data,
                                    int32_t main_idx, const bfgpu_pcs_data* perm_data, int32_t perm_idx, const uint32_t alpha_in[4],
                                    const uint32_t perm_challenges[8], const uint32_t cum_sum[4], uint32_t* out);
extern "C" int32_t bfgpu_quotient_values(bfgpu_ctx* ctx, const char* chip, const bfgpu_pcs_data* prep_data, int32_t prep_idx, const bfgpu_pcs_data* main_data,
                                         int32_t main_idx, const bfgpu_pcs_data* perm_data, int32_t perm_idx, const uint32_t alpha_in[4],
                                         const uint32_t perm_challenges[8], const uint32_t cum_sum[4], uint32_t* out) {
    AllocScope scope(ctx);
    return scope.ok(quotient_values_impl(ctx, chip, prep_data, prep_idx, main_data, main_idx, perm_data, perm_idx, alpha_in, perm_challenges, cum_sum, out));
}
static int32_t quotient_values_impl(bfgpu_ctx* ctx, const char* chip, const bfgpu_pcs_data* prep_data, int32_t prep_idx, const bfgpu_pcs_data* main_data,
                                    int32_t main_idx, const bfgpu_pcs_data* perm_data, int32_t perm_idx, const uint32_t alpha_in[4],
                                    const uint32_t perm_challenges[8], const uint32_t cum_sum[4], uint32_t* out) {
    if (!ctx || !chip || !main_data || !perm_data || !alpha_in || !perm_challenges || !cum_sum || !out) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    const int ci = chip_index(chip);
    if (ci < 0) return fail(ctx, BFGPU_ERR_INVALID, "unknown chip '%s'", chip);
    const air::ChipInfo& info = air::CHIPS[ci];
    if (ctx->log_blowup != 1 || info.log_quotient_degree != 1) return fail(ctx, BFGPU_ERR_INVALID, "quotient degree / blow-up other than 2 is not supported");
    if (main_idx < 0 || (size_t)main_idx >= main_data->ldes.size() || perm_idx < 0 || (size_t)perm_idx >= perm_data->ldes.size())
        return fail(ctx, BFGPU_ERR_INVALID, "bad matrix index");
    const DMat& lm = main_data->ldes[main_idx];
    const DMat& lp = perm_data->ldes[perm_idx];
    if (lm.cols != (uint32_t)info.main_w || lp.cols != 4u * (uint32_t)info.perm_w || lp.rows != lm.rows)
        return fail(ctx, BFGPU_ERR_INVALID, "chip %s: committed matrices have the wrong shape", chip);
    const uint32_t* prep = nullptr;
    if (info.prep_w) {
        if (!prep_data || prep_idx < 0 || (size_t)prep_idx >= prep_data->ldes.size()) return fail(ctx, BFGPU_ERR_INVALID, "chip %s needs its preprocessed commitment", chip);
        const DMat& lq = prep_data->ldes[prep_idx];
        if (lq.cols != (uint32_t)info.prep_w || lq.rows != lm.rows) return fail(ctx, BFGPU_ERR_INVALID, "chip %s: preprocessed LDE has the wrong shape", chip);
        prep = lq.d;
    }
    const uint64_t N = lm.rows, n = N / 2;
    const unsigned log_n = ilog2(n);
    const uint32_t gen = kb::to_mont(kb::GEN);
    kb::Ext alpha;
    for (int k = 0; k < 4; k++) alpha.c[k] = in_word(ctx, alpha_in[k]);
    air::Challenges chal;
    for (int k = 0; k < 4; k++) chal.alpha.c[k] = in_word(ctx, perm_challenges[k]);
    kb::Ext beta;
    for (int k = 0; k < 4; k++) beta.c[k] = in_word(ctx, perm_challenges[4 + k]);
    chal.beta_pow[0] = kb::ext_one();
    for (int k = 1; k < 8; k++) chal.beta_pow[k] = kb::ext_mul(chal.beta_pow[k - 1], beta);
    for (int k = 0; k < 4; k++) chal.cumulative_sum.c[k] = in_word(ctx, cum_sum[k]);
    Phase ph(ctx, BFGPU_PHASE_QUOTIENT);
    Scratch sc(ctx);
    std::vector<kb::Ext> apow(air::MAX_CONSTRAINTS);
    apow[0] = kb::ext_one();
    for (int k = 1; k < air::MAX_CONSTRAINTS; k++) apow[k] = kb::ext_mul(apow[k - 1], alpha);
    kb::Ext* d_apow = nullptr;
    uint32_t* q = nullptr;
    TRY(sc.alloc((void**)&d_apow, apow.size() * sizeof(kb::Ext)));
    TRY(sc.alloc((void**)&q, N * 16));
    TRY(upload_small(ctx, d_apow, apow.data(), apow.size() * sizeof(kb::Ext)));
    air::QuotientArgs qa;
    qa.chip = ci;
    qa.main = lm.d;
    qa.prep = prep;
    qa.perm = lp.d;
    qa.log_n = log_n;
    qa.lqd = 1;
    qa.shift = gen;
    qa.g_inv = kb::inv(kb::two_adic_generator(log_n));
    uint32_t sn = kb::pow(gen, n);
    qa.zh[0] = kb::sub(sn, kb::ONE);
    qa.zh[1] = kb::sub(kb::neg(sn), kb::ONE);
    qa.zh_inv[0] = kb::inv(qa.zh[0]);
    qa.zh_inv[1] = kb::inv(qa.zh[1]);
    qa.apow = d_apow;
    qa.tw = ctx->d_tw;
    qa.out = q;
#define BF_QUOT_CASE(C) \
    case C: air::k_quotient<C><<<(unsigned)((N + 127) / 128), 128, 0, ctx->stream>>>(qa, chal); break;
    switch (ci) { BF_QUOT_CASE(0) BF_QUOT_CASE(1) BF_QUOT_CASE(2) BF_QUOT_CASE(3) BF_QUOT_CASE(4) BF_QUOT_CASE(5) BF_QUOT_CASE(6) BF_QUOT_CASE(7) }
#undef BF_QUOT_CASE
    LAUNCHED(ctx);
    CU(cudaGetLastError());
    // the kernel leaves the two chunk matrices (chunk c = natural index mod 2, column-major, rows bit-reversed): put the values back in
    // natural order of the quotient domain for the caller
    std::vector<uint32_t> h(N * 4);
    CU(cudaMemcpyAsync(h.data(), q, N * 16, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    for (uint64_t i = 0; i < N; i++) {
        const uint64_t c = i & 1, pos = kb::bitrev((uint32_t)(i >> 1), log_n);
        for (int k = 0; k < 4; k++) out[4 * i + k] = out_word(ctx, h[(c * 4 + (uint64_t)k) * n + pos]);
    }
    return BFGPU_OK;
}

// =====================================================================================================
// trace checker: StarkMachine::debug_constraints (machine.rs:288-387, debug.rs:24-105, lookup/debug.rs:59-196)
// =====================================================================================================
#include "kernels_debug.cuh"

struct bfgpu_debug_report {
    std::vector<uint32_t> flat;
};

// Memory: the LogUp traces (16 B x perm_w per row), one 8-byte mask per row, and for the interaction pass R records
// (R <= sum of rows x lookups: 2^26 + 2^23.5 for 2^22 Cpu rows) held as two key/value buffers for the sort (2 x 24 B), the
// per-fingerprint aggregates (36 B) and the imbalanced-group indices (4 B): 88 B per record plus CUB's scratch, about 7 GB at
// 2^22 Cpu rows.  Everything is scratch of this call; only the flat report survives it.
static int32_t machine_debug_impl(bfgpu_ctx* ctx, const bfgpu_pk* pk, const bfgpu_shard* sd, const bfgpu_challenger* chh, uint32_t max_rows,
                                  uint32_t max_keys, bfgpu_debug_report** out);
extern "C" int32_t bfgpu_machine_debug(bfgpu_ctx* ctx, const bfgpu_pk* pk, const bfgpu_shard* sd, const bfgpu_challenger* chh, uint32_t max_rows,
                                       uint32_t max_keys, bfgpu_debug_report** out) {
    AllocScope scope(ctx);  // blocks taken by a failing call go back to the cache (see AllocScope)
    return scope.ok(machine_debug_impl(ctx, pk, sd, chh, max_rows, max_keys, out));
}
static int32_t machine_debug_impl(bfgpu_ctx* ctx, const bfgpu_pk* pk, const bfgpu_shard* sd, const bfgpu_challenger* chh, uint32_t max_rows,
                                  uint32_t max_keys, bfgpu_debug_report** out) {
    if (!ctx || !pk || !sd || !chh || !out) return fail(ctx, BFGPU_ERR_INVALID, "null argument");
    *out = nullptr;
    const size_t nchips = sd->names.size();
    if (nchips > 16) return fail(ctx, BFGPU_ERR_INVALID, "the checker handles at most 16 traces per shard");
    std::vector<int> pk_idx(nchips, -1);
    for (size_t i = 0; i < nchips; i++)
        for (size_t k = 0; k < pk->names.size(); k++)
            if (pk->names[k] == sd->names[i]) pk_idx[i] = (int)k;
    for (size_t i = 0; i < nchips; i++) {
        const air::ChipInfo& ci = air::CHIPS[sd->chip[i]];
        if (ci.prep_w && (pk_idx[i] < 0 || pk->traces[pk_idx[i]].rows != sd->traces[i].rows))
            return fail(ctx, BFGPU_ERR_INVALID, "chip %s: preprocessed trace missing or of a different height", ci.name);
        if (sd->traces[i].rows > (1ull << 24)) return fail(ctx, BFGPU_ERR_INVALID, "chip %s: more than 2^24 rows", ci.name);
    }
    // ---- transcript on a copy: main commitment, LogUp (alpha, beta) as machine_open, then the fingerprint challenges ----------
    bfgpu_challenger ch = box(chh)->ch;
    ch.observe_slice(sd->commit, 8);
    air::Challenges chal;
    chal.alpha = ch.sample_ext();
    const kb::Ext beta = ch.sample_ext();
    chal.beta_pow[0] = kb::ext_one();
    for (int k = 1; k < 8; k++) chal.beta_pow[k] = kb::ext_mul(chal.beta_pow[k - 1], beta);
    chal.cumulative_sum = kb::ext_zero();
    dbg::Fingerprint fp;
    fp.gamma = ch.sample_ext();
    const kb::Ext delta = ch.sample_ext();
    fp.delta_pow[0] = kb::ext_one();
    for (int k = 1; k <= air::MAX_LOOKUP_VALUES; k++) fp.delta_pow[k] = kb::ext_mul(fp.delta_pow[k - 1], delta);

    Scratch sc(ctx);
    // ---- LogUp traces and cumulative sums (the prover's own kernels) ----------------------------------------------------------
    std::vector<DMat> perm(nchips);
    std::vector<kb::Ext> csum(nchips);
    uint32_t* d_csums = nullptr;
    TRY(sc.alloc((void**)&d_csums, nchips * 16));
    TRY(perm_traces(ctx, pk, pk_idx, sd->chip, sd->traces, chal, &perm, d_csums));
    for (DMat& m : perm) sc.bufs.push_back(m.d);
    CU(cudaMemcpyAsync(csum.data(), d_csums, nchips * 16, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));  // the last-row constraint of each chip compares with its cumulative sum

    // ---- constraint pass ----------------------------------------------------------------------------------------------------
    std::vector<uint64_t*> masks(nchips, nullptr);
    std::vector<uint32_t*> bcounts(nchips, nullptr);
    std::vector<uint32_t> totals(nchips * 64);
    {
        Phase ph(ctx, BFGPU_PHASE_DEBUG_ROWS);
        uint32_t* d_totals = nullptr;
        TRY(sc.alloc((void**)&d_totals, nchips * 64 * 4));
        CU(cudaMemsetAsync(d_totals, 0, nchips * 64 * 4, ctx->stream));
        for (size_t i = 0; i < nchips; i++) {
            const uint64_t n = sd->traces[i].rows;
            const unsigned log_n = ilog2(n);
            const uint64_t nb = (n + dbg::MASK_BLOCK - 1) / dbg::MASK_BLOCK;
            TRY(sc.alloc((void**)&masks[i], n * 8));
            TRY(sc.alloc((void**)&bcounts[i], nb * 64 * 4));
            air::Challenges c2 = chal;
            c2.cumulative_sum = csum[i];
            const uint32_t* prep = pk_idx[i] >= 0 ? pk->traces[pk_idx[i]].d : nullptr;
#define BF_DBG_CASE(C) \
    case C: dbg::k_debug_rows<C><<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(sd->traces[i].d, prep, perm[i].d, log_n, c2, masks[i]); break;
            switch (sd->chip[i]) {
                BF_DBG_CASE(0) BF_DBG_CASE(1) BF_DBG_CASE(2) BF_DBG_CASE(3) BF_DBG_CASE(4) BF_DBG_CASE(5) BF_DBG_CASE(6) BF_DBG_CASE(7)
            }
#undef BF_DBG_CASE
            LAUNCHED(ctx);
            CU(cudaGetLastError());
            dbg::k_mask_counts<<<(unsigned)nb, 256, 0, ctx->stream>>>(masks[i], n, bcounts[i], d_totals + 64 * i);
            LAUNCHED(ctx);
            CU(cudaGetLastError());
        }
        CU(cudaMemcpyAsync(totals.data(), d_totals, nchips * 64 * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }

    // ---- interaction pass ---------------------------------------------------------------------------------------------------
    uint64_t rmax = 0;
    for (size_t i = 0; i < nchips; i++) rmax += sd->traces[i].rows * (uint64_t)air::num_lookups(sd->chip[i]);
    if (rmax >= (1ull << 31)) return fail(ctx, BFGPU_ERR_INVALID, "too many interactions for the checker (%llu)", (unsigned long long)rmax);
    uint64_t n_bad = 0;
    std::vector<uint32_t> gathered;
    {
        Phase ph(ctx, BFGPU_PHASE_DEBUG_LOOKUPS);
        dbg::FpKey *keys_a = nullptr, *keys_b = nullptr;
        uint64_t *vals_a = nullptr, *vals_b = nullptr;
        unsigned long long* d_count = nullptr;
        TRY(sc.alloc((void**)&d_count, 16));
        TRY(sc.alloc((void**)&keys_a, std::max<uint64_t>(rmax, 1) * sizeof(dbg::FpKey)));
        TRY(sc.alloc((void**)&vals_a, std::max<uint64_t>(rmax, 1) * 8));
        TRY(sc.alloc((void**)&keys_b, std::max<uint64_t>(rmax, 1) * sizeof(dbg::FpKey)));
        TRY(sc.alloc((void**)&vals_b, std::max<uint64_t>(rmax, 1) * 8));
        CU(cudaMemsetAsync(d_count, 0, 16, ctx->stream));
        for (size_t i = 0; i < nchips; i++) {
            const uint64_t n = sd->traces[i].rows;
            const unsigned log_n = ilog2(n);
            const uint32_t* prep = pk_idx[i] >= 0 ? pk->traces[pk_idx[i]].d : nullptr;
#define BF_REC_CASE(C)                                                                                                                          \
    case C:                                                                                                                                     \
        dbg::k_debug_records<C><<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(sd->traces[i].d, prep, log_n, (uint32_t)i, fp, keys_a, vals_a, \
                                                                                      d_count);                                                 \
        break;
            switch (sd->chip[i]) {
                BF_REC_CASE(0) BF_REC_CASE(1) BF_REC_CASE(2) BF_REC_CASE(3) BF_REC_CASE(4) BF_REC_CASE(5) BF_REC_CASE(6) BF_REC_CASE(7)
            }
#undef BF_REC_CASE
            LAUNCHED(ctx);
            CU(cudaGetLastError());
        }
        unsigned long long nrec = 0;
        CU(cudaMemcpyAsync(&nrec, d_count, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        if (nrec) {
            const int R = (int)nrec;
            size_t sort_bytes = 0, red_bytes = 0;
            CU(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, keys_a, keys_b, vals_a, vals_b, R, dbg::FpDecomposer{}, ctx->stream));
            int* d_chip_of_pos = nullptr;
            int* d_ngroups = nullptr;
            dbg::Group* groups = nullptr;
            uint32_t* bad = nullptr;
            std::vector<int> chip_of_pos(16, 0);
            for (size_t i = 0; i < nchips; i++) chip_of_pos[i] = sd->chip[i];
            TRY(sc.alloc((void**)&d_chip_of_pos, 16 * sizeof(int)));
            TRY(upload_small(ctx, d_chip_of_pos, chip_of_pos.data(), 16 * sizeof(int)));
            const auto grp_in = thrust::make_transform_iterator(vals_b, dbg::RecordToGroup{d_chip_of_pos});
            CU(cub::DeviceReduce::ReduceByKey(nullptr, red_bytes, keys_b, keys_a, grp_in, (dbg::Group*)nullptr, d_ngroups, dbg::GroupSum{}, R, ctx->stream));
            void* temp = nullptr;
            TRY(sc.alloc(&temp, std::max(sort_bytes, red_bytes)));
            TRY(sc.alloc((void**)&groups, (size_t)R * sizeof(dbg::Group)));
            TRY(sc.alloc((void**)&bad, (size_t)R * 4));
            TRY(sc.alloc((void**)&d_ngroups, 16));
            CU(cub::DeviceRadixSort::SortPairs(temp, sort_bytes, keys_a, keys_b, vals_a, vals_b, R, dbg::FpDecomposer{}, ctx->stream));
            LAUNCHED(ctx);
            CU(cub::DeviceReduce::ReduceByKey(temp, red_bytes, keys_b, keys_a, grp_in, groups, d_ngroups, dbg::GroupSum{}, R, ctx->stream));
            LAUNCHED(ctx);
            CU(cudaMemsetAsync(d_count, 0, 8, ctx->stream));
            dbg::k_imbalanced<<<(unsigned)((R + 255) / 256), 256, 0, ctx->stream>>>(groups, d_ngroups, bad, d_count);
            LAUNCHED(ctx);
            CU(cudaGetLastError());
            unsigned long long nb = 0;
            CU(cudaMemcpyAsync(&nb, d_count, 8, cudaMemcpyDeviceToHost, ctx->stream));
            CU(cudaStreamSynchronize(ctx->stream));
            n_bad = nb;
            if (n_bad) {
                dbg::TraceRef tr{};
                for (size_t i = 0; i < nchips; i++) {
                    tr.main[i] = sd->traces[i].d;
                    tr.prep[i] = pk_idx[i] >= 0 ? pk->traces[pk_idx[i]].d : nullptr;
                    tr.log_n[i] = ilog2(sd->traces[i].rows);
                    tr.chip[i] = sd->chip[i];
                }
                uint32_t* d_out = nullptr;
                TRY(sc.alloc((void**)&d_out, n_bad * dbg::GATHER_WORDS * 4));
                dbg::k_gather_values<<<(unsigned)((n_bad + 63) / 64), 64, 0, ctx->stream>>>(tr, groups, bad, n_bad, d_out);
                LAUNCHED(ctx);
                CU(cudaGetLastError());
                gathered.resize(n_bad * dbg::GATHER_WORDS);
                CU(cudaMemcpyAsync(gathered.data(), d_out, gathered.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
            }
        }
    }
    CU(cudaStreamSynchronize(ctx->stream));

    // ---- failing rows: exact counts from the totals, the first max_rows rows from the count blocks that hold them ------------------
    auto* rep = new bfgpu_debug_report();
    std::unique_ptr<bfgpu_debug_report> rep_guard(rep);
    auto& flat = rep->flat;
    flat.push_back((uint32_t)nchips);
    kb::Ext total = kb::ext_zero();
    for (size_t i = 0; i < nchips; i++) {
        const uint64_t n = sd->traces[i].rows;
        const int nk = air::CHIPS[sd->chip[i]].n_constraints;
        flat.push_back((uint32_t)sd->chip[i]);
        flat.push_back(ilog2(n));
        for (int k = 0; k < 4; k++) flat.push_back(out_word(ctx, csum[i].c[k]));
        total = kb::ext_add(total, csum[i]);
        const uint32_t* tot = &totals[64 * i];
        int nfail = 0;
        for (int k = 0; k < nk; k++) nfail += tot[k] != 0;
        flat.push_back((uint32_t)nfail);
        if (!nfail) continue;
        const uint64_t nb = (n + dbg::MASK_BLOCK - 1) / dbg::MASK_BLOCK;
        std::vector<uint32_t> bc(nb * 64);
        CU(cudaMemcpy(bc.data(), bcounts[i], bc.size() * 4, cudaMemcpyDeviceToHost));
        std::vector<char> need(nb, 0);
        for (int k = 0; k < nk; k++) {
            uint64_t want = std::min<uint64_t>(tot[k], max_rows);
            for (uint64_t b = 0; b < nb && want; b++)
                if (bc[b * 64 + k]) {
                    need[b] = 1;
                    want -= std::min<uint64_t>(want, bc[b * 64 + k]);
                }
        }
        std::vector<std::vector<uint32_t>> rows(nk);
        std::vector<uint64_t> blk(dbg::MASK_BLOCK);
        for (uint64_t b = 0; b < nb; b++) {
            if (!need[b]) continue;
            const uint64_t r0 = b * dbg::MASK_BLOCK, cnt = std::min<uint64_t>(dbg::MASK_BLOCK, n - r0);
            CU(cudaMemcpy(blk.data(), masks[i] + r0, cnt * 8, cudaMemcpyDeviceToHost));
            for (uint64_t r = 0; r < cnt; r++)
                for (uint64_t m = blk[r]; m; m &= m - 1) {
                    const int k = __builtin_ctzll(m);
                    if (rows[k].size() < max_rows) rows[k].push_back((uint32_t)(r0 + r));
                }
        }
        for (int k = 0; k < nk; k++) {
            if (!tot[k]) continue;
            flat.push_back((uint32_t)k);
            flat.push_back(tot[k]);
            flat.insert(flat.end(), rows[k].begin(), rows[k].end());
        }
    }
    for (int k = 0; k < 4; k++) flat.push_back(out_word(ctx, total.c[k]));

    // ---- imbalanced keys, ordered by (kind, canonical values) ------------------------------------------------------------------
    std::vector<uint64_t> order(n_bad);
    std::vector<std::vector<uint32_t>> sort_key(n_bad);
    for (uint64_t b = 0; b < n_bad; b++) {
        const uint32_t* g = &gathered[b * dbg::GATHER_WORDS];
        order[b] = b;
        sort_key[b].push_back(g[0]);
        for (uint32_t v = 0; v < g[1]; v++) sort_key[b].push_back(kb::from_mont(g[2 + v]));
    }
    std::sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) { return sort_key[a] < sort_key[b]; });
    flat.push_back((uint32_t)n_bad);
    for (uint64_t j = 0; j < std::min<uint64_t>(n_bad, max_keys); j++) {
        const uint32_t* g = &gathered[order[j] * dbg::GATHER_WORDS];
        const uint32_t* net = g + 2 + air::MAX_LOOKUP_VALUES;
        flat.push_back(g[0]);
        flat.push_back(g[1]);
        for (uint32_t v = 0; v < g[1]; v++) flat.push_back(out_word(ctx, g[2 + v]));
        uint32_t s = 0, nc = 0;
        for (int c = 0; c < air::NUM_CHIPS; c++) {
            s = kb::add(s, net[c]);
            nc += net[c] != 0;
        }
        flat.push_back(out_word(ctx, s));
        flat.push_back(nc);
        for (int c = 0; c < air::NUM_CHIPS; c++)
            if (net[c]) {
                flat.push_back((uint32_t)c);
                flat.push_back(out_word(ctx, net[c]));
            }
    }
    *out = rep_guard.release();
    return BFGPU_OK;
}
extern "C" uint64_t bfgpu_debug_report_size(const bfgpu_debug_report* r) { return r ? r->flat.size() : 0; }
extern "C" int32_t bfgpu_debug_report_read(const bfgpu_debug_report* r, uint32_t* out) {
    if (!r || !out) return BFGPU_ERR_INVALID;
    memcpy(out, r->flat.data(), r->flat.size() * 4);
    return BFGPU_OK;
}
extern "C" void bfgpu_debug_report_free(bfgpu_debug_report* r) { delete r; }

// =====================================================================================================
// one commitment over several GPUs
// =====================================================================================================
#include "dist_commit.cuh"

// =====================================================================================================
// native executor + device-side trace generation
// =====================================================================================================
#include "tracegen.cuh"

// =====================================================================================================
// one shard proof over several GPUs
// =====================================================================================================
#include "dist_prove.cuh"
#include "comm_shm.h"

// =====================================================================================================
// native verifier (host only)
// =====================================================================================================
#include "verifier.h"

// =====================================================================================================
// batch verifier: host stage per proof (verifier::prepare), query checks on the device (kernels_verify.cuh)
// =====================================================================================================
#include <atomic>
#include <thread>

#include "kernels_verify.cuh"

namespace vfy {
// host stage of one batch item: the verdict the host decides by itself (outer: before the shard verifier, the `BfProver::verify`
// checks; inner: the shard verifier's), or the plan the device completes
struct Item {
    std::string outer, inner, cons;
    bool decided = false;
    verifier::Plan pl;
    uint32_t bits = 0;  // first result bit (device items)
    bool device = false;
};
// verifier::walk over the device's result bits
struct BitChecks {
    const uint32_t* bits;
    uint32_t base, nc;
    bool get(uint32_t q, uint32_t c) const {
        const uint32_t b = base + q * nc + c;
        return bits && ((bits[b >> 5] >> (b & 31)) & 1);
    }
    bool input(uint32_t q, int r) const { return get(q, (uint32_t)r); }
    bool commit(uint32_t q, uint32_t k) const { return get(q, 4 + k); }
    bool final_ok(uint32_t q) const { return get(q, nc - 1); }
};
template <class F>
static void parallel_for(int n, F fn) {
    const int nt = std::max(1, std::min<int>({n, (int)std::thread::hardware_concurrency(), 16}));
    std::atomic<int> next{0};
    auto work = [&] {
        for (int i; (i = next.fetch_add(1)) < n;) fn(i);
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nt; t++) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
}
static size_t align16(size_t b) { return (b + 15) & ~(size_t)15; }
}  // namespace vfy

extern "C" int32_t bfgpu_verify_batch(bfgpu_ctx* ctx, const bfgpu_verify_item* items, int32_t n_items, int repr, uint32_t log_blowup,
                                      uint32_t num_queries, uint32_t pow_bits, const uint32_t* options, int32_t n_options, int32_t core,
                                      int32_t* status, char* errs, uint64_t err_len) {
    if (!ctx) return BFGPU_ERR_INVALID;
    if (n_items < 0 || (n_items && (!items || !status || (err_len && !errs)))) return fail(ctx, BFGPU_ERR_INVALID, "bfgpu_verify_batch: null argument");
    if (n_items == 0) return BFGPU_OK;
    AllocScope scope(ctx);
    uint32_t opt[BFGPU_NUM_OPTS];
    verifier::parse_options(options, n_options, opt);
    const bool monty = repr == BFGPU_REPR_MONTY;
    std::vector<vfy::Item> it(n_items);
    // host stage: the checks of bfgpu_verify_core_proof / bfgpu_verify_shard_ex up to the queries, the query plan, the constraints at zeta
    vfy::parallel_for(n_items, [&](int i) {
        auto& x = it[i];
        const auto& a = items[i];
        x.decided = true;
        if (core) {
            if (!a.vk_commit || !a.proof) {
                x.outer = "null argument";
                return;
            }
            if (!(x.outer = verifier::core_precheck(a.proof, a.n_words)).empty()) return;
        }
        if (!a.vk_commit || !a.proof || a.n_prep < 0 || (a.n_prep && (!a.prep_names || !a.prep_log_heights))) {
            x.inner = "null argument";
            return;
        }
        std::vector<std::pair<int, unsigned>> prep;
        if (!(x.inner = verifier::parse_prep(a.prep_names, a.prep_log_heights, a.n_prep, prep)).empty()) return;
        if (!(x.inner = verifier::prepare(a.vk_commit, prep, a.proof, a.n_words, monty, log_blowup, num_queries, pow_bits, opt, x.pl)).empty()) return;
        x.cons = verifier::constraints(x.pl);
        x.decided = false;
        x.device = x.pl.tall_round < 0;  // else the walk stops at query 0 before any check
    });
    // ---- plan -> device records
    std::vector<vfy::VProof> P;
    std::vector<vfy::VMat> M;
    std::vector<uint32_t> aux;
    std::vector<int> owner;
    uint64_t n_words = 0, n_leaf = 0;
    uint32_t n_bits = 0, n_fold = 0, n_merkle = 0;
    for (int i = 0; i < n_items; i++) {
        auto& x = it[i];
        if (x.decided || !x.device) continue;
        const auto& pl = x.pl;
        vfy::VProof v{};
        v.words = n_words;
        v.leaf = n_leaf;
        v.bits = x.bits = n_bits;
        v.task = n_fold;
        v.mtask = n_merkle;
        v.nq = pl.nq_eff;
        v.stride = (uint32_t)pl.stride;
        v.monty = monty;
        v.log_max = pl.log_max;
        v.n_commit = pl.n_commit;
        v.rollin = pl.opt[BFGPU_OPT_FRI_ROLLIN];
        for (int r = 0; r < 4; r++) {
            v.round_off[r] = pl.round_off[r];
            v.sib_off[r] = pl.sib_off[r];
            v.round_lbm[r] = pl.round_lbm[r];
        }
        v.aux = (uint32_t)aux.size();
        aux.insert(aux.end(), pl.index.begin(), pl.index.end());
        aux.insert(aux.end(), pl.cp_off.begin(), pl.cp_off.end());
        for (auto& b : pl.betas) aux.insert(aux.end(), b.c, b.c + 4);
        for (auto& c : pl.fri_commits) aux.insert(aux.end(), c.begin(), c.end());
        for (auto& r : pl.rounds) aux.insert(aux.end(), r.commit, r.commit + 8);
        aux.insert(aux.end(), pl.fri_alpha.c, pl.fri_alpha.c + 4);
        aux.insert(aux.end(), pl.final_poly.c, pl.final_poly.c + 4);
        for (int r = 0; r < 4; r++) {
            v.mat[r] = (uint32_t)M.size();
            for (auto& m : pl.rounds[r].mats) {
                M.push_back(vfy::VMat{m.log_n + pl.log_blowup, m.width, (uint32_t)m.points.size(), (uint32_t)aux.size()});
                for (auto& z : m.points) aux.insert(aux.end(), z.c, z.c + 4);
                for (auto& vals : m.values)
                    for (auto& e : vals) aux.insert(aux.end(), e.c, e.c + 4);
            }
        }
        v.mat[4] = (uint32_t)M.size();
        P.push_back(v);
        owner.push_back(i);
        n_words += (uint64_t)pl.nq_eff * pl.stride;
        n_leaf += (uint64_t)pl.nq_eff * pl.n_commit;
        n_bits += pl.nq_eff * (5 + pl.n_commit);
        n_fold += pl.nq_eff;
        n_merkle += pl.nq_eff * (4 + pl.n_commit);
    }
    std::vector<uint32_t> bits((n_bits + 31) / 32, 0);
    if (!P.empty()) {
        // one page-locked staging buffer: [proofs | matrices | aux words | query words], then the result bits coming back
        const size_t oP = 0, oM = vfy::align16(P.size() * sizeof(vfy::VProof)), oA = oM + vfy::align16(M.size() * sizeof(vfy::VMat)),
                     oW = oA + vfy::align16(aux.size() * 4), in_bytes = oW + vfy::align16(n_words * 4), out_bytes = bits.size() * 4;
        if (ctx->vstage_size < in_bytes + out_bytes) {
            if (ctx->vstage) {
                CU(cudaStreamSynchronize(ctx->stream));
                cudaFreeHost(ctx->vstage);
                ctx->vstage = nullptr;
                ctx->vstage_size = 0;
            }
            const size_t want = std::max<size_t>(in_bytes + out_bytes, 1 << 20) * 5 / 4;
            CU(cudaHostAlloc((void**)&ctx->vstage, want, cudaHostAllocDefault));
            ctx->vstage_size = want;
        }
        uint8_t* st = ctx->vstage;
        memcpy(st + oP, P.data(), P.size() * sizeof(vfy::VProof));
        memcpy(st + oM, M.data(), M.size() * sizeof(vfy::VMat));
        memcpy(st + oA, aux.data(), aux.size() * 4);
        vfy::parallel_for((int)P.size(), [&](int j) {
            const auto& pl = it[owner[j]].pl;
            const auto& a = items[owner[j]];
            uint32_t* dst = (uint32_t*)(st + oW) + P[j].words;
            const uint64_t need = (uint64_t)pl.nq_eff * pl.stride, have = std::min<uint64_t>(need, a.n_words - pl.q_base);
            memcpy(dst, a.proof + pl.q_base, have * 4);
            memset(dst + have, 0, (need - have) * 4);  // past a truncation: stages the walk never reads
        });
        Phase ph(ctx, BFGPU_PHASE_VERIFY);
        Scratch s(ctx);
        uint8_t* d_in;
        uint32_t* d_work;
        TRY(s.alloc((void**)&d_in, in_bytes));
        TRY(s.alloc((void**)&d_work, (n_leaf * 8 + bits.size()) * 4));
        uint32_t* d_bits = d_work + n_leaf * 8;
        CU(cudaMemcpyAsync(d_in, st, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaMemsetAsync(d_bits, 0, bits.size() * 4, ctx->stream));
        const auto* dP = (const vfy::VProof*)(d_in + oP);
        const auto* dM = (const vfy::VMat*)(d_in + oM);
        const auto* dA = (const uint32_t*)(d_in + oA);
        const auto* dW = (const uint32_t*)(d_in + oW);
        vfy::k_verify_fold<<<(n_fold + 127) / 128, 128, 0, ctx->stream>>>(dP, (int)P.size(), dM, dA, dW, n_fold, d_work, d_bits);
        LAUNCHED(ctx);
        vfy::k_verify_merkle<<<(n_merkle + 127) / 128, 128, 0, ctx->stream>>>(dP, (int)P.size(), dM, dA, dW, n_merkle, d_work, d_bits);
        LAUNCHED(ctx);
        CU(cudaGetLastError());
        uint32_t* back = (uint32_t*)(st + in_bytes);
        CU(cudaMemcpyAsync(back, d_bits, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        memcpy(bits.data(), back, out_bytes);
    }
    // ---- the first failing event of every proof, in the host verifier's order
    for (int i = 0; i < n_items; i++) {
        auto& x = it[i];
        std::string e = x.outer;
        if (e.empty()) {
            std::string in = x.inner;
            if (!x.decided) {
                vfy::BitChecks bc{x.device ? bits.data() : nullptr, x.bits, 5 + x.pl.n_commit};
                in = verifier::walk(x.pl, bc);
                if (in.empty()) in = x.cons;
            }
            e = core ? verifier::core_wrap(in) : in;
        }
        status[i] = e.empty() ? BFGPU_OK : BFGPU_ERR_INVALID;
        verifier::say(errs ? errs + (size_t)i * err_len : nullptr, err_len, e);
    }
    return scope.ok();
}
