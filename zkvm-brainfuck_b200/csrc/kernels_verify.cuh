// kernels_verify.cuh — device executor of the verifier's query plan (verifier::Plan, csrc/verifier.h) for a batch of proofs.
//
// The host stage has parsed and shape-checked every proof, replayed its transcript and laid out its queries; these kernels compute
// the pass/fail bit of every check of the plan, and verifier::walk reports the first failing one in the host verifier's order.
// Every index a kernel computes is bounded by plan sizes: the word buffer holds nq_eff * stride words per proof (zero padded past
// a truncation), so a stage the reader never reaches computes on padding and its bit is never read.
//
// Result bits of query q of a proof: bits + q * (5 + n_commit) + c, c = r (input round r: MerkleTreeMmcs::verify_batch, InputMmcsError),
// 4 + k (commit-phase round k: CommitPhaseMmcsError), 4 + n_commit (fold chain end == final polynomial, FinalPolyMismatch).  Set = passed.
#pragma once

namespace vfy {

struct VProof {
    uint64_t words;  // first word of query 0 in the word buffer
    uint64_t leaf;   // first commit-phase leaf row (8 words) of this proof: row leaf + q * n_commit + k
    uint32_t bits;   // first result bit
    uint32_t task;   // first fold task: one per (proof, query)
    uint32_t mtask;  // first Merkle task: one per (proof, tree, query)
    uint32_t nq, stride, monty, log_max, n_commit, rollin;
    uint32_t round_off[4], sib_off[4], round_lbm[4];
    uint32_t mat[5];  // VMat records of input round r: [mat[r], mat[r + 1])
    // aux words: index[nq] | cp_off[n_commit] | betas[n_commit][4] | fri commits[n_commit][8] | round commits[4][8] | fri alpha[4] | final poly[4]
    uint32_t aux;
};
struct VMat {
    uint32_t log_h, width, npts;
    uint32_t vals;  // aux index: opening points [npts][4], then opened values [npts][width][4]
};

__device__ __forceinline__ const VProof& find_proof(const VProof* P, int np, uint32_t t, bool merkle) {
    int lo = 0, hi = np - 1;
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if ((merkle ? P[mid].mtask : P[mid].task) <= t) lo = mid;
        else hi = mid - 1;
    }
    return P[lo];
}
__device__ __forceinline__ uint32_t fe(const VProof& pr, const uint32_t* W, uint32_t q, uint32_t o) {
    const uint32_t v = W[pr.words + (uint64_t)q * pr.stride + o];
    return pr.monty ? v : kb::to_mont(v);
}
__device__ __forceinline__ kb::Ext ld_ext(const uint32_t* a) { return kb::Ext{{a[0], a[1], a[2], a[3]}}; }
__device__ __forceinline__ void set_bit(uint32_t* bits, uint32_t b) { atomicOr(&bits[b >> 5], 1u << (b & 31)); }

// One thread per (proof, query): reduced openings per height (fri/two_adic_pcs.rs verify: open_input), the fold chain with the
// FRI_ROLLIN rule (fri/verifier.rs verify_query), every round's 8-word leaf row, and the final-polynomial check.
__global__ void k_verify_fold(const VProof* __restrict__ P, int np, const VMat* __restrict__ M, const uint32_t* __restrict__ aux,
                              const uint32_t* __restrict__ W, uint32_t n_tasks, uint32_t* __restrict__ leaf, uint32_t* __restrict__ bits) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tasks) return;
    const VProof& pr = find_proof(P, np, t, false);
    const uint32_t q = t - pr.task;
    const uint32_t* A = aux + pr.aux;
    const uint32_t index = A[q];
    const uint32_t* cp_off = A + pr.nq;
    const uint32_t* betas = cp_off + pr.n_commit;
    const uint32_t* tail = betas + 12 * pr.n_commit + 32;  // past betas, fri commits and round commits
    const kb::Ext alpha = ld_ext(tail), final_poly = ld_ext(tail + 4);
    const uint32_t gen = kb::to_mont(kb::GEN);
    kb::Ext ro[kb::TWO_ADICITY + 1], ap[kb::TWO_ADICITY + 1];
    uint32_t seen = 0;
    for (int r = 0; r < 4; r++) {
        const uint32_t lbm = pr.round_lbm[r];
        const uint32_t ridx = index >> (pr.log_max - lbm);
        uint32_t o = pr.round_off[r];
        for (uint32_t mi = pr.mat[r]; mi < pr.mat[r + 1]; mi++) {
            const VMat m = M[mi];
            const uint32_t lh = m.log_h;
            const uint32_t x = kb::mul(gen, kb::pow(kb::two_adic_generator(lh), kb::bitrev(ridx >> (lbm - lh), lh)));
            if (!((seen >> lh) & 1)) {
                seen |= 1u << lh;
                ro[lh] = kb::ext_zero();
                ap[lh] = kb::ext_one();
            }
            const uint32_t* pts = aux + m.vals;
            const uint32_t* vals = pts + 4 * m.npts;
            kb::Ext a = ap[lh];
            for (uint32_t p = 0; p < m.npts; p++) {
                kb::Ext d = kb::ext_neg(ld_ext(pts + 4 * p));
                d.c[0] = kb::add(d.c[0], x);  // x - z
                // sum_c alpha^k (p_c(x) - p_c(z)), then one product with 1 / (x - z)
                kb::Ext acc = kb::ext_zero();
                for (uint32_t c = 0; c < m.width; c++) {
                    kb::Ext diff = kb::ext_neg(ld_ext(vals + 4 * (p * m.width + c)));
                    diff.c[0] = kb::add(diff.c[0], fe(pr, W, q, o + c));
                    acc = kb::ext_add(acc, kb::ext_mul(a, diff));
                    a = kb::ext_mul(a, alpha);
                }
                ro[lh] = kb::ext_add(ro[lh], kb::ext_mul(acc, kb::ext_inv(d)));
            }
            ap[lh] = a;
            o += m.width;
        }
    }
    kb::Ext folded = kb::ext_zero();
    uint32_t idx = index;
    for (uint32_t k = 0; k < pr.n_commit; k++) {
        const uint32_t lfh = pr.log_max - 1 - k;
        if ((seen >> (lfh + 1)) & 1) {  // rolled in right after the fold of round k-1 (plain, or scaled by beta_{k-1}^2)
            kb::Ext rv = ro[lfh + 1];
            if (pr.rollin == 1 && k > 0) rv = kb::ext_mul(kb::ext_sqr(ld_ext(betas + 4 * (k - 1))), rv);
            folded = kb::ext_add(folded, rv);
        }
        kb::Ext ev[2] = {folded, folded};
        for (int c = 0; c < 4; c++) ev[(idx ^ 1) & 1].c[c] = fe(pr, W, q, cp_off[k] + c);
        uint32_t* row = leaf + 8 * (pr.leaf + (uint64_t)q * pr.n_commit + k);
        for (int c = 0; c < 4; c++) {
            row[c] = ev[0].c[c];
            row[4 + c] = ev[1].c[c];
        }
        idx >>= 1;
        // fold_row: e0 + (beta - x0) (e1 - e0) / (x1 - x0),  x0 = g_{lfh+1}^{bitrev(idx)}, x1 = -x0
        const uint32_t x0 = kb::pow(kb::two_adic_generator(lfh + 1), kb::bitrev(idx, lfh));
        kb::Ext b = ld_ext(betas + 4 * k);
        b.c[0] = kb::sub(b.c[0], x0);
        const uint32_t den = kb::inv(kb::sub(kb::neg(x0), x0));
        folded = kb::ext_add(ev[0], kb::ext_scale(kb::ext_mul(b, kb::ext_sub(ev[1], ev[0])), den));
    }
    if (folded.c[0] == final_poly.c[0] && folded.c[1] == final_poly.c[1] && folded.c[2] == final_poly.c[2] && folded.c[3] == final_poly.c[3])
        set_bit(bits, pr.bits + q * (5 + pr.n_commit) + 4 + pr.n_commit);
}

__device__ __forceinline__ void compress(uint32_t (&cur)[8], const uint32_t* l, const uint32_t* r) {
    uint32_t s[16];
    for (int j = 0; j < 8; j++) {
        s[j] = l[j];
        s[8 + j] = r[j];
    }
    p2::permute(s);
    for (int j = 0; j < 8; j++) cur[j] = s[j];
}
// PaddingFreeSponge over the concatenated opened rows of the round's matrices of LDE height 2^h (input order); false if there are none
__device__ bool group_digest(const VProof& pr, const VMat* M, const uint32_t* W, int r, uint32_t q, uint32_t h, uint32_t (&out)[8]) {
    uint32_t s[16] = {0};
    uint32_t o = pr.round_off[r], n = 0, c = 0;
    bool any = false;
    for (uint32_t mi = pr.mat[r]; mi < pr.mat[r + 1]; mi++) {
        const uint32_t w = M[mi].width;
        if (M[mi].log_h == h) {
            any = true;
            for (uint32_t j = 0; j < w; j++, n++) {
                s[c++] = fe(pr, W, q, o + j);
                if (c == 8) {
                    p2::permute(s);
                    c = 0;
                }
            }
        }
        o += w;
    }
    if (c || (any && n == 0)) p2::permute(s);
    for (int j = 0; j < 8; j++) out[j] = s[j];
    return any;
}

// One thread per (proof, tree, query), queries fastest so that a warp walks one tree: MerkleTreeMmcs::verify_batch of input round r
// (tree r < 4: sponge the tallest rows, compress upward, inject the shorter heights' rows) or of commit-phase round k (tree 4 + k).
__global__ void k_verify_merkle(const VProof* __restrict__ P, int np, const VMat* __restrict__ M, const uint32_t* __restrict__ aux,
                                const uint32_t* __restrict__ W, uint32_t n_tasks, const uint32_t* __restrict__ leaf, uint32_t* __restrict__ bits) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tasks) return;
    const VProof& pr = find_proof(P, np, t, true);
    const uint32_t tree = (t - pr.mtask) / pr.nq, q = (t - pr.mtask) % pr.nq;
    const uint32_t* A = aux + pr.aux;
    const uint32_t* cp_off = A + pr.nq;
    const uint32_t* fri_commits = cp_off + 5 * pr.n_commit;
    const uint32_t* round_commits = fri_commits + 8 * pr.n_commit;
    uint32_t cur[8], sib[8], idx;
    const uint32_t* root;
    if (tree < 4) {
        const int r = (int)tree;
        const uint32_t lbm = pr.round_lbm[r];
        idx = A[q] >> (pr.log_max - lbm);
        group_digest(pr, M, W, r, q, lbm, cur);
        for (uint32_t l = 0; l < lbm; l++) {
            for (int j = 0; j < 8; j++) sib[j] = fe(pr, W, q, pr.sib_off[r] + 8 * l + j);
            if (idx & 1) compress(cur, sib, cur);
            else compress(cur, cur, sib);
            idx >>= 1;
            uint32_t inj[8];
            if (group_digest(pr, M, W, r, q, lbm - 1 - l, inj)) compress(cur, cur, inj);
        }
        root = round_commits + 8 * r;
    } else {
        const uint32_t k = tree - 4, lfh = pr.log_max - 1 - k;
        uint32_t s[16] = {0};
        const uint32_t* row = leaf + 8 * (pr.leaf + (uint64_t)q * pr.n_commit + k);
        for (int j = 0; j < 8; j++) s[j] = row[j];
        p2::permute(s);
        for (int j = 0; j < 8; j++) cur[j] = s[j];
        idx = A[q] >> (k + 1);
        for (uint32_t l = 0; l < lfh; l++) {
            for (int j = 0; j < 8; j++) sib[j] = fe(pr, W, q, cp_off[k] + 4 + 8 * l + j);
            if (idx & 1) compress(cur, sib, cur);
            else compress(cur, cur, sib);
            idx >>= 1;
        }
        root = fri_commits + 8 * k;
    }
    bool ok = true;
    for (int j = 0; j < 8; j++) ok &= cur[j] == root[j];
    if (ok) set_bit(bits, pr.bits + q * (5 + pr.n_commit) + tree);
}

}  // namespace vfy
