// kernels_debug.cuh — the trace checker (bfgpu_machine_debug): every constraint on every row, and the balance of every
// interaction, driven by the generated row programs in gen_air_debug.cuh.
//
// Restates `StarkMachine::debug_constraints` (reference crates/stark/src/machine.rs:288-387 -> debug.rs:24-105) and
// `debug_interactions_with_all_chips` (crates/stark/src/lookup/debug.rs:59-196) on the device-resident traces of a shard:
// column-major, Montgomery words, bit-reversed rows (thread t reads stored row t coalesced; natural row i = bitrev(t)).
//
// Constraint pass: k_debug_rows writes one 64-bit mask per natural row (bit k = constraint k of the fold order is nonzero),
// k_mask_counts turns it into exact per-constraint counts, globally and per block of MASK_BLOCK natural rows; the host then copies
// only the blocks that hold the first `max_rows` failing rows of each failing constraint.
//
// Interaction pass: k_debug_records emits one record per (row, lookup) with a nonzero multiplicity: a 4-word fingerprint
// gamma + kind + sum_k delta^(k+1) v_k (the LogUp denominator under fresh challenges), the signed multiplicity and a locator.
// The records are sorted by fingerprint (CUB radix sort, 128-bit key) and reduced per fingerprint (CUB reduce-by-key) into
// per-chip nets; k_imbalanced keeps the groups whose total is nonzero and k_gather_values rebuilds their (kind, values) by running
// the row program again at the group's smallest locator.  Two distinct (kind, values) tuples share a fingerprint only where a
// degree <= 8 polynomial in delta vanishes: probability <= 8 / p^4 per pair, about R^2 * 4 / p^4 over R records.
#pragma once
#include <memory>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_reduce.cuh>
#include <cuda/std/tuple>
#include <thrust/iterator/transform_iterator.h>

#include "kernels_air.cuh"
#include "gen_air_debug.cuh"

namespace dbg {

constexpr int MASK_BLOCK = 1024;  // natural rows per count block (k_mask_counts: 256 threads x 4 rows)

// ---- constraint pass ------------------------------------------------------------------------------------------------------------
// Thread t: stored row t = natural row i = bitrev(t); the next row is natural (i + 1) mod n.  Exact selectors (Montgomery 1 or 0).
template <int CHIP>
__global__ void __launch_bounds__(128) k_debug_rows(const uint32_t* __restrict__ main, const uint32_t* __restrict__ prep, const uint32_t* __restrict__ perm,
                                                    unsigned log_n, air::Challenges ch, uint64_t* __restrict__ mask) {
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint64_t n = 1ull << log_n;
    if (t >= n) return;
    const uint32_t i = kb::bitrev((uint32_t)t, log_n);
    const uint32_t inext = (i + 1) & (uint32_t)(n - 1);
    air::LdeLoader ld{main, prep, perm, n, t, kb::bitrev(inext, log_n)};
    air::Selectors sel;
    sel.is_first = i == 0 ? kb::ONE : 0u;
    sel.is_last = i == n - 1 ? kb::ONE : 0u;
    sel.is_trans = i == n - 1 ? 0u : kb::ONE;
    mask[i] = air::air_constraint_mask(CHIP, ld, sel, ch);
}

// per-constraint failing-row counts: block_counts[b * 64 + k] over natural rows [b * MASK_BLOCK, (b + 1) * MASK_BLOCK), totals[k]
// over the whole trace.  A clean block costs one load per row and no atomics.
__global__ void __launch_bounds__(256) k_mask_counts(const uint64_t* __restrict__ mask, uint64_t n, uint32_t* __restrict__ block_counts,
                                                     uint32_t* __restrict__ totals) {
    __shared__ uint32_t cnt[64];
    if (threadIdx.x < 64) cnt[threadIdx.x] = 0;
    __syncthreads();
    const uint64_t base = (uint64_t)blockIdx.x * MASK_BLOCK;
    for (int r = threadIdx.x; r < MASK_BLOCK; r += blockDim.x) {
        uint64_t m = base + r < n ? mask[base + r] : 0;
        while (m) {
            atomicAdd(&cnt[__ffsll((long long)m) - 1], 1u);
            m &= m - 1;
        }
    }
    __syncthreads();
    if (threadIdx.x < 64) {
        const uint32_t c = cnt[threadIdx.x];
        block_counts[(uint64_t)blockIdx.x * 64 + threadIdx.x] = c;
        if (c) atomicAdd(&totals[threadIdx.x], c);
    }
}

// ---- interaction pass -----------------------------------------------------------------------------------------------------------
struct FpKey {  // fingerprint words (Montgomery, < 2^31) w0 w1 | w2 w3, most significant first
    uint64_t hi, lo;
};
struct FpDecomposer {
    __host__ __device__ cuda::std::tuple<uint64_t&, uint64_t&> operator()(FpKey& k) const { return {k.hi, k.lo}; }
};
__host__ __device__ __forceinline__ bool operator==(const FpKey& a, const FpKey& b) { return a.hi == b.hi && a.lo == b.lo; }
struct Fingerprint {
    kb::Ext gamma;
    kb::Ext delta_pow[air::MAX_LOOKUP_VALUES + 1];  // delta^0 .. delta^MAX_LOOKUP_VALUES
};
// locator: commit position (4 bits) | lookup index (4 bits) | natural row (24 bits)
__host__ __device__ __forceinline__ uint32_t locator(uint32_t pos, uint32_t lookup, uint32_t row) { return pos << 28 | lookup << 24 | row; }
static_assert(air::MAX_LOOKUPS <= 16, "the locator holds a 4-bit lookup index");

// One thread per stored row; records of a warp are appended with one atomic per lookup (warp-aggregated).  The append order
// is not deterministic, the sort and every reduction below are order-independent.
template <int CHIP>
__global__ void __launch_bounds__(128) k_debug_records(const uint32_t* __restrict__ main, const uint32_t* __restrict__ prep, unsigned log_n, uint32_t pos,
                                                       Fingerprint fp, FpKey* __restrict__ keys, uint64_t* __restrict__ vals,
                                                       unsigned long long* __restrict__ count) {
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint64_t n = 1ull << log_n;
    const bool live = t < n;
    const unsigned lane = threadIdx.x & 31;
    air::LookupVals lv[air::MAX_LOOKUPS];
    if (live) {
        air::TraceLoader ld{main, prep, n, t};
        air::air_lookups(CHIP, ld, lv);
    }
    const uint32_t i = live ? kb::bitrev((uint32_t)t, log_n) : 0u;
#pragma unroll
    for (int l = 0; l < air::num_lookups(CHIP); l++) {
        const bool emit = live && lv[l].mult != 0u;
        const unsigned ballot = __ballot_sync(0xffffffffu, emit);
        if (!ballot) continue;
        unsigned long long base = 0;
        const int leader = __ffs(ballot) - 1;
        if ((int)lane == leader) base = atomicAdd(count, (unsigned long long)__popc(ballot));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (!emit) continue;
        const uint64_t slot = base + __popc(ballot & ((1u << lane) - 1u));
        kb::Ext f = fp.gamma;
        f.c[0] = kb::add(f.c[0], kb::to_mont(lv[l].kind));
#pragma unroll
        for (int k = 0; k < air::MAX_LOOKUP_VALUES; k++)
            if (k < (int)lv[l].n_values) f = kb::ext_add(f, kb::ext_scale(fp.delta_pow[k + 1], lv[l].v[k]));
        keys[slot] = FpKey{(uint64_t)f.c[0] << 32 | f.c[1], (uint64_t)f.c[2] << 32 | f.c[3]};
        const uint32_t m = lv[l].is_send ? lv[l].mult : kb::neg(lv[l].mult);
        vals[slot] = (uint64_t)m << 32 | locator(pos, (uint32_t)l, i);
    }
}

// per-fingerprint aggregate: net multiplicity of every chip (air::CHIPS index, Montgomery, mod p) and the smallest locator
struct Group {
    uint32_t net[air::NUM_CHIPS];
    uint32_t loc;
};
struct RecordToGroup {
    const int* chip_of_pos;  // commit position -> air::CHIPS index (device)
    __host__ __device__ Group operator()(uint64_t v) const {
        Group g;
        const uint32_t loc = (uint32_t)v, m = (uint32_t)(v >> 32);
#pragma unroll
        for (int c = 0; c < air::NUM_CHIPS; c++) g.net[c] = 0;
        g.net[chip_of_pos[loc >> 28]] = m;
        g.loc = loc;
        return g;
    }
};
struct GroupSum {
    __host__ __device__ Group operator()(const Group& a, const Group& b) const {
        Group g;
#pragma unroll
        for (int c = 0; c < air::NUM_CHIPS; c++) g.net[c] = kb::add(a.net[c], b.net[c]);
        g.loc = a.loc < b.loc ? a.loc : b.loc;
        return g;
    }
};

// indices of the groups whose total net is nonzero (append order not deterministic: the host orders them by (kind, values))
__global__ void __launch_bounds__(256) k_imbalanced(const Group* __restrict__ groups, const int* __restrict__ n_groups, uint32_t* __restrict__ bad,
                                                    unsigned long long* __restrict__ n_bad) {
    const uint64_t g = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (g >= (uint64_t)*n_groups) return;
    uint32_t s = 0;
#pragma unroll
    for (int c = 0; c < air::NUM_CHIPS; c++) s = kb::add(s, groups[g].net[c]);
    if (s) bad[atomicAdd(n_bad, 1ull)] = (uint32_t)g;
}

// (kind, values) of the imbalanced groups: the row program of the chip at the group's smallest locator
constexpr int GATHER_WORDS = 2 + air::MAX_LOOKUP_VALUES + air::NUM_CHIPS;  // kind, n_values, values, per-chip nets
struct TraceRef {
    const uint32_t* main[16];
    const uint32_t* prep[16];
    uint32_t log_n[16];
    int chip[16];
};
__global__ void __launch_bounds__(64) k_gather_values(TraceRef tr, const Group* __restrict__ groups, const uint32_t* __restrict__ bad, uint64_t n_bad,
                                                      uint32_t* __restrict__ out) {
    const uint64_t b = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (b >= n_bad) return;
    const Group g = groups[bad[b]];
    const uint32_t pos = g.loc >> 28, l = (g.loc >> 24) & 15u, row = g.loc & 0xffffffu;
    const uint64_t n = 1ull << tr.log_n[pos];
    air::TraceLoader ld{tr.main[pos], tr.prep[pos], n, kb::bitrev(row, tr.log_n[pos])};
    air::LookupVals lv[air::MAX_LOOKUPS];
    air::air_lookups(tr.chip[pos], ld, lv);
    uint32_t* o = out + b * GATHER_WORDS;
    o[0] = lv[l].kind;
    o[1] = lv[l].n_values;
    for (int k = 0; k < air::MAX_LOOKUP_VALUES; k++) o[2 + k] = k < (int)lv[l].n_values ? lv[l].v[k] : 0u;
    for (int c = 0; c < air::NUM_CHIPS; c++) o[2 + air::MAX_LOOKUP_VALUES + c] = g.net[c];
}

}  // namespace dbg
