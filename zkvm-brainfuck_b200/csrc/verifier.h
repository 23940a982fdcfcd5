// verifier.h — native (host, no device needed) verifier of a shard proof in the serialisation bfgpu_machine_open emits.
//
// Restates the reference's `Verifier::verify_shard` (crates/stark/src/verifier.rs:27-216: transcript, opening rounds,
// `verify_constraints` :218-292, `recompute_quotient` :294-329, cumulative-sum check :210-213) and, from Plonky3
// p3-fri / p3-commit / p3-merkle-tree v0.1.0 (SURVEY.md Appendix B.9-B.11), `TwoAdicFriPcs::verify`, `fri::verify`
// (commit-phase replay, proof of work, per-query input openings, fold chain) and `MerkleTreeMmcs::verify_batch`.
// SURVEY.md §8f item 2: a Rust-free verifier so that proofs of both backends can be checked without the reference
// toolchain.  The constraint programs over F_p^4 come from gen_air_ext.h (same declarative AIR as the prover kernels).
// Verdict parity (accept / reject, error names) with the CPU restatement is checked in tests/test_native_verifier.py.
#pragma once
#include <cstdarg>
#include <map>
#include <set>
#include <string>
#include <vector>

#include "gen_air_ext.h"

namespace verifier {

using kb::Ext;

struct Reader {
    const uint32_t* p;
    uint64_t n, pos = 0;
    bool monty;  // words already Montgomery; else canonical
    bool ok = true;
    uint32_t raw() {
        if (pos >= n) {
            ok = false;
            return 0;
        }
        return p[pos++];
    }
    uint32_t fe() {  // a field element must be the unique representative in [0, p): anything else is a second encoding of the same proof
        uint32_t v = raw();
        if (v >= kb::P) {
            ok = false;
            return 0;
        }
        return monty ? v : kb::to_mont(v);
    }
    Ext ext() {
        Ext e;
        for (int i = 0; i < 4; i++) e.c[i] = fe();
        return e;
    }
    void digest(uint32_t d[8]) {
        for (int i = 0; i < 8; i++) d[i] = fe();
    }
};

static inline Ext e_pow2k(Ext a, unsigned k) {  // a^(2^k)
    for (unsigned i = 0; i < k; i++) a = kb::ext_sqr(a);
    return a;
}
static inline bool e_eq(const Ext& a, const Ext& b) { return a.c[0] == b.c[0] && a.c[1] == b.c[1] && a.c[2] == b.c[2] && a.c[3] == b.c[3]; }
// sum_k X^k * v[k] for four extension elements v: re-assembles a flattened extension column (verifier.rs:262-281)
static inline Ext unflatten(const Ext* v) {
    // multiplication by X: (c0, c1, c2, c3) -> (3 c3, c0, c1, c2)
    Ext acc = v[3];
    for (int k = 2; k >= 0; k--) {
        Ext t{{kb::mul3(acc.c[3]), acc.c[0], acc.c[1], acc.c[2]}};
        acc = kb::ext_add(t, v[k]);
    }
    return acc;
}

// PaddingFreeSponge<Perm, 16, 8, 8> over a slice of Montgomery words
static inline void sponge(const uint32_t* w, size_t n, uint32_t out[8]) {
    uint32_t s[16] = {0};
    for (size_t i = 0; i < n; i += 8) {
        for (size_t k = 0; k < 8 && i + k < n; k++) s[k] = w[i + k];
        host_p2::permute(s);
    }
    if (n == 0) host_p2::permute(s);  // not reached by this machine (no empty rows)
    for (int k = 0; k < 8; k++) out[k] = s[k];
}
static inline void compress(const uint32_t l[8], const uint32_t r[8], uint32_t out[8]) {
    uint32_t s[16];
    for (int k = 0; k < 8; k++) {
        s[k] = l[k];
        s[8 + k] = r[k];
    }
    host_p2::permute(s);
    for (int k = 0; k < 8; k++) out[k] = s[k];
}

// MerkleTreeMmcs::verify_batch: rows[i] = opened row of matrix i (Montgomery words), heights[i] its height.
static bool verify_batch(const uint32_t root[8], const std::vector<uint64_t>& heights, const std::vector<std::vector<uint32_t>>& rows, uint64_t index,
                         const std::vector<std::array<uint32_t, 8>>& siblings) {
    std::vector<size_t> order(heights.size());
    for (size_t i = 0; i < order.size(); i++) order[i] = i;
    if (order.empty()) return false;  // a round without matrices opens nothing
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return heights[a] > heights[b]; });
    size_t pos = 0;
    auto group_digest = [&](uint64_t h, uint32_t out[8]) -> bool {  // sponge over the concatenated rows of height h
        std::vector<uint32_t> cat;
        bool any = false;
        while (pos < order.size() && heights[order[pos]] == h) {
            const auto& r = rows[order[pos++]];
            cat.insert(cat.end(), r.begin(), r.end());
            any = true;
        }
        if (any) sponge(cat.data(), cat.size(), out);
        return any;
    };
    uint64_t cur_h = heights[order[0]];
    if (cur_h == 0 || (cur_h & (cur_h - 1))) return false;
    uint32_t cur[8];
    group_digest(cur_h, cur);
    for (const auto& sib : siblings) {
        uint32_t nxt[8];
        if (index & 1) compress(sib.data(), cur, nxt);
        else compress(cur, sib.data(), nxt);
        memcpy(cur, nxt, 32);
        index >>= 1;
        cur_h >>= 1;
        uint32_t inj[8];
        if (cur_h && group_digest(cur_h, inj)) {
            compress(cur, inj, nxt);
            memcpy(cur, nxt, 32);
        }
    }
    if (cur_h != 1 || pos != order.size()) return false;
    return memcmp(cur, root, 32) == 0;
}

struct OpenedMat {
    unsigned log_n;              // trace-domain size of the matrix
    uint32_t width;
    std::vector<Ext> points;     // opening points
    std::vector<std::vector<Ext>> values;  // [point][column]
};
struct Round {
    uint32_t commit[8];
    std::vector<OpenedMat> mats;
};

static std::string fmt(const char* f, ...) {
    char buf[256];
    va_list ap;
    va_start(ap, f);
    vsnprintf(buf, sizeof buf, f, ap);
    va_end(ap);
    return buf;
}

struct ChipOpen {
    int chip;
    unsigned log_degree;
    Ext csum;
};

// The query phase of one proof, laid out before any of it is checked.  Where a word sits in the proof depends only on the shape
// words read before the queries, never on whether a check passed, so the host stage (`prepare`) can place every query's words,
// replay the whole transcript and find where the reader would stop; an executor then computes every check of the plan (host:
// HostChecks; device: kernels_verify.cuh) and `walk` reports the first failing event in the order `verify` meets them.
struct Plan {
    bool monty;
    unsigned log_blowup, log_max, n_commit;
    uint32_t nq;      // queries of the proof (= num_queries)
    uint32_t nq_eff;  // queries up to and including the one the reader stops in
    uint32_t opt[BFGPU_NUM_OPTS];
    std::vector<std::pair<int, unsigned>> prep;
    Round rounds[4];
    std::vector<ChipOpen> chips;
    Ext perm_ch[2], alpha, zeta, fri_alpha, final_poly;
    std::vector<std::array<uint32_t, 8>> fri_commits;
    std::vector<Ext> betas;
    std::vector<uint32_t> index;  // sampled query indices (nq_eff)
    uint64_t q_base, stride;      // word position of query 0 and words per query
    // per input round: first opened-row word, first sibling word (both relative to the query's index word), log2 of the tallest LDE
    uint32_t round_off[4], sib_off[4], round_lbm[4];
    std::vector<uint32_t> cp_off;  // per FRI round: first word of the commit-phase opening (sibling value, then path)
    int tall_round = -1;           // first round with a matrix taller than the FRI domain
    bool rollin_bad = false;       // a reduced opening at a height the fold chain never rolls in
    // stage 0: the index word; 1..4: input round stage-1; 5 + k: commit-phase round k.  stop_q == nq: the reader reads every query
    uint32_t stop_q, stop_stage = 0;
    bool index_word_differs = false, trailing = false;
};

// Everything up to the queries: shapes, opened values, transcript, proof of work, and the query plan.  Returns "" when the
// proof reaches its queries, else the error `verify` returns before them.
static std::string prepare(const uint32_t vk_commit_in[8], const std::vector<std::pair<int, unsigned>>& prep /* (chip index, log height), pk order */,
                           const uint32_t* words, uint64_t n_words, bool monty, unsigned log_blowup, unsigned num_queries, unsigned pow_bits,
                           const uint32_t opt[BFGPU_NUM_OPTS], Plan& pl) {
    Reader rd{words, n_words, 0, monty};
    pl.monty = monty;
    pl.log_blowup = log_blowup;
    pl.prep = prep;
    memcpy(pl.opt, opt, sizeof pl.opt);
    uint32_t vk_commit[8];
    for (int i = 0; i < 8; i++) {
        if (vk_commit_in[i] >= kb::P) return "InvalidProofShape: non-canonical verifying key";
        vk_commit[i] = monty ? vk_commit_in[i] : kb::to_mont(vk_commit_in[i]);
    }
    Round* rounds = pl.rounds;
    memcpy(rounds[0].commit, vk_commit, 32);
    rd.digest(rounds[1].commit);
    rd.digest(rounds[2].commit);
    rd.digest(rounds[3].commit);
    const uint32_t n = rd.raw();
    if (!rd.ok || n == 0 || n > (uint32_t)air::NUM_CHIPS) return "ChipOpeningLengthMismatch";
    auto& chips = pl.chips;
    chips.resize(n);
    std::map<int, size_t> where;
    for (auto& c : chips) {
        c.chip = (int)rd.raw();
        c.log_degree = rd.raw();
        c.csum = rd.ext();
        if (!rd.ok || c.chip < 0 || c.chip >= air::NUM_CHIPS || log_blowup > (unsigned)kb::TWO_ADICITY ||
            c.log_degree > (unsigned)kb::TWO_ADICITY - log_blowup || where.count(c.chip))
            return "InvalidProofShape";  // (the sum is not formed: log_degree is an untrusted 32-bit word)
        where[c.chip] = &c - chips.data();
    }
    // ---- transcript (verifier.rs:60-104); the caller's challenger has observed the verifying key --------------------
    bfgpu_challenger ch;
    ch.observe_slice(vk_commit, 8);
    for (int i = 0; i < 7; i++) ch.observe(0);
    ch.observe_slice(rounds[1].commit, 8);
    pl.perm_ch[0] = ch.sample_ext();
    pl.perm_ch[1] = ch.sample_ext();
    ch.observe_slice(rounds[2].commit, 8);
    for (auto& c : chips) ch.observe_ext(c.csum);
    pl.alpha = ch.sample_ext();
    ch.observe_slice(rounds[3].commit, 8);
    const Ext zeta = pl.zeta = ch.sample_ext();
    auto next_point = [&](unsigned log_n) { return kb::ext_scale(zeta, kb::two_adic_generator(log_n)); };
    // ---- opening rounds: shapes, then the opened values in serialisation order ---------------------------------------------
    for (auto& pr : prep) {
        if (!where.count(pr.first)) return "InvalidProofShape: preprocessed chip missing from the proof";
        OpenedMat m{pr.second, (uint32_t)air::CHIPS[pr.first].prep_w, {zeta}, {}};
        if (!air::CHIPS[pr.first].local_only) m.points.push_back(next_point(pr.second));
        rounds[0].mats.push_back(m);
    }
    for (auto& c : chips) {
        const auto& info = air::CHIPS[c.chip];
        OpenedMat mm{c.log_degree, (uint32_t)info.main_w, {zeta}, {}};
        if (!info.local_only) mm.points.push_back(next_point(c.log_degree));
        rounds[1].mats.push_back(mm);
        rounds[2].mats.push_back(OpenedMat{c.log_degree, 4u * (uint32_t)info.perm_w, {zeta, next_point(c.log_degree)}, {}});
        for (int d = 0; d < (1 << info.log_quotient_degree); d++) rounds[3].mats.push_back(OpenedMat{c.log_degree, 4, {zeta}, {}});
    }
    for (int r = 0; r < 4; r++) {
        if (rounds[r].mats.empty()) return "InvalidProofShape: commitment round without matrices";
        for (auto& m : rounds[r].mats)
            if (m.log_n > (unsigned)kb::TWO_ADICITY - log_blowup) return "InvalidProofShape";
    }
    for (int r = 0; r < 4; r++)
        for (auto& m : rounds[r].mats)
            for (size_t t = 0; t < m.points.size(); t++) {
                std::vector<Ext> v(m.width);
                for (auto& e : v) e = rd.ext();
                m.values.push_back(std::move(v));
            }
    if (!rd.ok) return "InvalidProofShape: truncated opened values";
    // ---- TwoAdicFriPcs::verify ------------------------------------------------------------------------------------------------
    for (int r = 0; r < 4; r++)
        for (auto& m : rounds[r].mats)
            for (auto& v : m.values)
                for (auto& e : v)
                    if (opt[BFGPU_OPT_OBSERVE_OPENED_VALUES]) ch.observe_ext(e);
    pl.fri_alpha = ch.sample_ext();
    const uint32_t n_commit = pl.n_commit = rd.raw();
    if (!rd.ok || n_commit == 0 || n_commit > (unsigned)kb::TWO_ADICITY - log_blowup) return "InvalidProofShape";
    for (auto& c : chips)  // every committed LDE must fit under the first FRI layer
        if (c.log_degree > n_commit) return "InvalidProofShape: chip taller than the FRI domain";
    pl.fri_commits.resize(n_commit);
    pl.betas.resize(n_commit);
    for (uint32_t k = 0; k < n_commit; k++) {
        rd.digest(pl.fri_commits[k].data());
        ch.observe_slice(pl.fri_commits[k].data(), 8);
        pl.betas[k] = ch.sample_ext();
    }
    pl.final_poly = rd.ext();
    ch.observe_ext(pl.final_poly);
    const uint32_t pow_witness = rd.raw();  // canonical in the serialisation
    const uint32_t nq = pl.nq = rd.raw();
    if (!rd.ok || nq != num_queries) return "InvalidProofShape: query count";
    // every error of pcs.verify reaches the caller wrapped (verifier.rs: `.map_err(VerificationError::InvalidopeningArgument)`)
    if (pow_witness >= kb::P || !ch.check_witness(pow_bits, kb::to_mont(pow_witness))) return "InvalidOpeningArgument:InvalidPowWitness";
    // ---- query layout: index word, per input round the opened rows then the Merkle path, per FRI round the sibling value then the path
    const unsigned log_max = pl.log_max = n_commit + log_blowup;
    uint64_t off = 1;
    std::set<unsigned, std::greater<unsigned>> heights;
    for (int r = 0; r < 4; r++) {
        unsigned lbm = 0;
        uint64_t w = 0;
        for (auto& m : rounds[r].mats) {
            lbm = std::max(lbm, m.log_n + log_blowup);
            w += m.width;
            heights.insert(m.log_n + log_blowup);
        }
        if (lbm > log_max && pl.tall_round < 0) pl.tall_round = r;
        pl.round_off[r] = (uint32_t)off;
        pl.sib_off[r] = (uint32_t)(off + w);
        pl.round_lbm[r] = lbm;
        off += w + 8ull * lbm;
    }
    pl.cp_off.resize(n_commit);
    for (uint32_t k = 0; k < n_commit; k++) {
        pl.cp_off[k] = (uint32_t)off;
        off += 4 + 8ull * (log_max - 1 - k);
    }
    pl.stride = off;
    pl.q_base = rd.pos;
    // the fold chain rolls in the reduced opening of height log_max - k before folding round k; any other height is left over
    auto hit = heights.begin();
    for (uint32_t k = 0; k < n_commit; k++)
        if (hit != heights.end() && *hit == log_max - k) ++hit;
    pl.rollin_bad = hit != heights.end();
    // the reader's stop: the first word past the end, or a field word (every word of a query but its index) outside [0, p)
    pl.stop_q = nq;
    for (uint64_t q = 0; q < nq && pl.stop_q == nq; q++) {
        const uint64_t base = pl.q_base + q * pl.stride;
        for (uint64_t o = 0; o < pl.stride; o++) {
            if (base + o >= n_words || (o && words[base + o] >= kb::P)) {
                pl.stop_q = (uint32_t)q;
                if (o >= pl.round_off[0]) pl.stop_stage = 1;
                for (int r = 1; r < 4; r++)
                    if (o >= pl.round_off[r]) pl.stop_stage = 1 + r;
                for (uint32_t k = 0; k < n_commit; k++)
                    if (o >= pl.cp_off[k]) pl.stop_stage = 5 + k;
                break;
            }
        }
    }
    pl.nq_eff = pl.stop_q < nq ? pl.stop_q + 1 : nq;
    pl.index.resize(pl.nq_eff);
    for (uint32_t q = 0; q < pl.nq_eff; q++) {
        pl.index[q] = ch.sample_bits(log_max);
        // The serialisation carries the index for the reader's convenience; the reference's QueryProof does not, its verifier uses the
        // sampled one.  So a transcript that went wrong fails where the reference fails (the Merkle openings no longer fit the sampled
        // index: InputMmcsError); a proof that verifies but carries another index word is a second encoding of the same proof and is
        // refused at the end.
        const uint64_t p = pl.q_base + q * pl.stride;
        if (p < n_words && words[p] != pl.index[q]) pl.index_word_differs = true;
    }
    pl.trailing = pl.stop_q == nq && pl.q_base + (uint64_t)nq * pl.stride != n_words;
    return "";
}

// The first failing event of the query phase, in the order `verify` meets them.  Checks: input(q, r), commit(q, k) and
// final_ok(q), called in exactly that order, each only after every earlier event of the walk has passed.
template <class Checks>
static std::string walk(const Plan& pl, Checks& ck) {
    for (uint32_t q = 0; q < pl.nq_eff; q++) {
        if (pl.stop_q == q && pl.stop_stage == 0) return "InvalidProofShape: truncated query";
        for (int r = 0; r < 4; r++) {
            if (pl.tall_round == r) return "InvalidProofShape: matrix taller than the FRI domain";
            if (pl.stop_q == q && pl.stop_stage == 1u + r) return "InvalidProofShape: truncated query";
            if (!ck.input(q, r)) return "InvalidOpeningArgument:InputMmcsError";
        }
        for (uint32_t k = 0; k < pl.n_commit; k++) {
            if (pl.stop_q == q && pl.stop_stage == 5 + k) return "InvalidProofShape: truncated commit-phase opening";
            if (!ck.commit(q, k)) return "InvalidOpeningArgument:CommitPhaseMmcsError";
        }
        if (pl.rollin_bad) return "InvalidOpeningArgument:InvalidProofShape";
        if (!ck.final_ok(q)) return "InvalidOpeningArgument:FinalPolyMismatch";
    }
    if (pl.index_word_differs) return "InvalidProofShape: query index";
    if (pl.trailing) return "InvalidProofShape: trailing words";
    return "";
}

// Host executor of the plan: the per-query reduced openings (fri/two_adic_pcs.rs verify: open_input), MerkleTreeMmcs::verify_batch
// and the fold chain (fri/verifier.rs verify_query), computed in the walk's order.
struct HostChecks {
    const Plan& pl;
    const uint32_t* words;
    std::map<unsigned, Ext, std::greater<unsigned>> ro;
    std::map<unsigned, Ext> apow;
    std::map<unsigned, Ext, std::greater<unsigned>>::iterator it;
    Ext folded;
    uint64_t idx = 0;
    uint32_t fe(uint32_t q, uint64_t o) const {
        const uint32_t v = words[pl.q_base + q * pl.stride + o];
        return pl.monty ? v : kb::to_mont(v);
    }
    void digests(uint32_t q, uint64_t o, size_t n, std::vector<std::array<uint32_t, 8>>& out) const {
        out.resize(n);
        for (size_t l = 0; l < n; l++)
            for (int j = 0; j < 8; j++) out[l][j] = fe(q, o + 8 * l + j);
    }
    bool input(uint32_t q, int r) {
        if (r == 0) {
            ro.clear();
            apow.clear();
        }
        const unsigned log_blowup = pl.log_blowup, log_max = pl.log_max, log_batch_max = pl.round_lbm[r];
        const auto& mats = pl.rounds[r].mats;
        std::vector<uint64_t> heights;
        std::vector<std::vector<uint32_t>> rows;
        uint64_t o = pl.round_off[r];
        for (auto& m : mats) {
            heights.push_back(1ull << (m.log_n + log_blowup));
            std::vector<uint32_t> row(m.width);
            for (auto& w : row) w = fe(q, o++);
            rows.push_back(std::move(row));
        }
        std::vector<std::array<uint32_t, 8>> sib;
        digests(q, pl.sib_off[r], log_batch_max, sib);
        const uint64_t ridx = pl.index[q] >> (log_max - log_batch_max);
        if (!verify_batch(pl.rounds[r].commit, heights, rows, ridx, sib)) return false;
        const uint32_t gen = kb::to_mont(kb::GEN);
        for (size_t mi = 0; mi < mats.size(); mi++) {
            const auto& m = mats[mi];
            const unsigned lh = m.log_n + log_blowup;
            const uint64_t rr = ridx >> (log_batch_max - lh);
            const uint32_t x = kb::mul(gen, kb::pow(kb::two_adic_generator(lh), kb::bitrev((uint32_t)rr, lh)));
            if (!ro.count(lh)) {
                ro[lh] = kb::ext_zero();
                apow[lh] = kb::ext_one();
            }
            for (size_t t = 0; t < m.points.size(); t++) {
                Ext d = kb::ext_neg(m.points[t]);
                d.c[0] = kb::add(d.c[0], x);  // x - z
                const Ext inv = kb::ext_inv(d);
                for (uint32_t c = 0; c < m.width; c++) {
                    Ext diff = kb::ext_neg(m.values[t][c]);
                    diff.c[0] = kb::add(diff.c[0], rows[mi][c]);  // p(x) - p(z)
                    ro[lh] = kb::ext_add(ro[lh], kb::ext_mul(apow[lh], kb::ext_mul(diff, inv)));
                    apow[lh] = kb::ext_mul(apow[lh], pl.fri_alpha);
                }
            }
        }
        if (r == 3) {
            folded = kb::ext_zero();
            it = ro.begin();
            idx = pl.index[q];
        }
        return true;
    }
    bool commit(uint32_t q, uint32_t k) {
        const unsigned lfh = pl.log_max - 1 - k;
        if (it != ro.end() && it->first == lfh + 1) {
            // rolled in right after the fold of round k-1: plain, or scaled by that round's beta^2 (BFGPU_OPT_FRI_ROLLIN)
            Ext r = it->second;
            if (pl.opt[BFGPU_OPT_FRI_ROLLIN] == 1 && k > 0) r = kb::ext_mul(kb::ext_sqr(pl.betas[k - 1]), r);
            folded = kb::ext_add(folded, r);
            ++it;
        }
        Ext ev[2] = {folded, folded};
        for (int c = 0; c < 4; c++) ev[(idx ^ 1) & 1].c[c] = fe(q, pl.cp_off[k] + c);
        std::vector<std::array<uint32_t, 8>> sib;
        digests(q, pl.cp_off[k] + 4, lfh, sib);
        std::vector<uint32_t> row(8);
        for (int e = 0; e < 2; e++)
            for (int c = 0; c < 4; c++) row[4 * e + c] = ev[e].c[c];
        if (!verify_batch(pl.fri_commits[k].data(), {1ull << lfh}, {row}, idx >> 1, sib)) return false;
        idx >>= 1;
        // fold_row: e0 + (beta - x0) (e1 - e0) / (x1 - x0),  x0 = g_{lfh+1}^{bitrev(idx)}, x1 = -x0
        const uint32_t x0 = kb::pow(kb::two_adic_generator(lfh + 1), kb::bitrev((uint32_t)idx, lfh));
        Ext b = pl.betas[k];
        b.c[0] = kb::sub(b.c[0], x0);
        const uint32_t den = kb::inv(kb::sub(kb::neg(x0), x0));
        folded = kb::ext_add(ev[0], kb::ext_scale(kb::ext_mul(b, kb::ext_sub(ev[1], ev[0])), den));
        return true;
    }
    bool final_ok(uint32_t) const { return e_eq(folded, pl.final_poly); }
};

// ---- constraints at zeta (verifier.rs:218-329) -----------------------------------------------------------------------------
static std::string constraints(const Plan& pl) {
    const Round* rounds = pl.rounds;
    const auto& chips = pl.chips;
    const Ext zeta = pl.zeta;
    const uint32_t gen = kb::to_mont(kb::GEN);
    size_t qpos = 0;
    std::map<int, size_t> prep_at;
    for (size_t k = 0; k < pl.prep.size(); k++) prep_at[pl.prep[k].first] = k;
    Ext total = kb::ext_zero();
    for (size_t i = 0; i < chips.size(); i++) {
        const auto& c = chips[i];
        const auto& info = air::CHIPS[c.chip];
        const unsigned ld = c.log_degree, lqd = (unsigned)info.log_quotient_degree;
        // selectors of the trace domain (shift 1) at zeta
        const Ext z_h = kb::ext_sub(e_pow2k(zeta, ld), kb::ext_one());
        const uint32_t ginv = kb::inv(kb::two_adic_generator(ld));
        Ext um1 = zeta, umg = zeta;
        um1.c[0] = kb::sub(um1.c[0], kb::ONE);
        umg.c[0] = kb::sub(umg.c[0], ginv);
        air::ExtRow R;
        R.is_first = kb::ext_mul(z_h, kb::ext_inv(um1));
        R.is_last = kb::ext_mul(z_h, kb::ext_inv(umg));
        R.is_trans = umg;
        const Ext inv_zeroifier = kb::ext_inv(z_h);
        // recompute_quotient: chunk domains = split of the disjoint domain (shift GEN, size 2^(ld+lqd)) into 2^lqd cosets of size 2^ld
        const unsigned nchunk = 1u << lqd;
        std::vector<uint32_t> shifts(nchunk);
        const uint32_t gq = kb::two_adic_generator(ld + lqd);
        for (unsigned d = 0; d < nchunk; d++) shifts[d] = kb::mul(gen, kb::pow(gq, d));
        auto zp = [&](unsigned dom, Ext x) {  // Z of chunk domain `dom` at x: (x / shift)^(2^ld) - 1
            return kb::ext_sub(e_pow2k(kb::ext_scale(x, kb::inv(shifts[dom])), ld), kb::ext_one());
        };
        Ext quotient = kb::ext_zero();
        for (unsigned d = 0; d < nchunk; d++) {
            Ext zps = kb::ext_one();
            for (unsigned o = 0; o < nchunk; o++)
                if (o != d) zps = kb::ext_mul(zps, kb::ext_mul(zp(o, zeta), kb::ext_inv(zp(o, kb::ext_from_base(shifts[d])))));
            quotient = kb::ext_add(quotient, kb::ext_mul(zps, unflatten(rounds[3].mats[qpos + d].values[0].data())));
        }
        qpos += nchunk;
        // opened rows
        std::vector<Ext> zeros_main(info.main_w, kb::ext_zero()), zeros_prep(std::max(info.prep_w, 1), kb::ext_zero());
        const auto& mm = rounds[1].mats[i];
        R.main0 = mm.values[0].data();
        R.main1 = mm.values.size() > 1 ? mm.values[1].data() : zeros_main.data();
        if (info.prep_w) {
            if (!prep_at.count(c.chip)) return "InvalidProofShape: chip needs a preprocessed trace";
            const auto& pm = rounds[0].mats[prep_at[c.chip]];
            R.prep0 = pm.values[0].data();
            R.prep1 = pm.values.size() > 1 ? pm.values[1].data() : zeros_prep.data();
        } else {
            R.prep0 = R.prep1 = zeros_prep.data();
        }
        std::vector<Ext> perm0(info.perm_w), perm1(info.perm_w);
        for (int j = 0; j < info.perm_w; j++) {
            perm0[j] = unflatten(rounds[2].mats[i].values[0].data() + 4 * j);
            perm1[j] = unflatten(rounds[2].mats[i].values[1].data() + 4 * j);
        }
        R.perm0 = perm0.data();
        R.perm1 = perm1.data();
        air::Challenges chal;
        chal.alpha = pl.perm_ch[0];
        chal.beta_pow[0] = kb::ext_one();
        for (int k = 1; k < 8; k++) chal.beta_pow[k] = kb::ext_mul(chal.beta_pow[k - 1], pl.perm_ch[1]);
        chal.cumulative_sum = c.csum;
        std::vector<Ext> apow(info.n_constraints);
        apow[0] = kb::ext_one();
        for (int k = 1; k < info.n_constraints; k++) apow[k] = kb::ext_mul(apow[k - 1], pl.alpha);
        Ext folded = kb::ext_zero();
        air::air_constraints_ext(c.chip, R, chal, apow.data(), folded);
        if (!e_eq(kb::ext_mul(folded, inv_zeroifier), quotient)) return fmt("OodEvaluationMismatch:%s", info.name);
        total = kb::ext_add(total, c.csum);
    }
    if (!e_eq(total, kb::ext_zero())) return "CumulativeSumsError";
    return "";
}

// returns "" when the proof is accepted, else the reference's error name (+ detail)
static std::string verify(const uint32_t vk_commit[8], const std::vector<std::pair<int, unsigned>>& prep /* (chip index, log height), pk order */,
                          const uint32_t* words, uint64_t n_words, bool monty, unsigned log_blowup, unsigned num_queries, unsigned pow_bits,
                          const uint32_t opt[BFGPU_NUM_OPTS]) {
    Plan pl;
    std::string e = prepare(vk_commit, prep, words, n_words, monty, log_blowup, num_queries, pow_bits, opt, pl);
    if (!e.empty()) return e;
    HostChecks hc{pl, words};
    e = walk(pl, hc);
    return e.empty() ? constraints(pl) : e;
}

}  // namespace verifier

namespace verifier {
// (chip index, log height) of every preprocessed trace of the verifying key, pk order; "" or the entry points' argument error
static std::string parse_prep(const char* const* prep_names, const uint32_t* prep_log_heights, int32_t n_prep, std::vector<std::pair<int, unsigned>>& prep) {
    for (int i = 0; i < n_prep; i++) {
        int ci = chip_index(prep_names[i]);
        if (ci < 0) return std::string("unknown chip ") + prep_names[i];
        prep.emplace_back(ci, prep_log_heights[i]);
    }
    return "";
}
static void parse_options(const uint32_t* options, int32_t n_options, uint32_t opt[BFGPU_NUM_OPTS]) {
    opt[0] = 1, opt[1] = 0, opt[2] = 0;
    for (int32_t i = 0; options && i < n_options && i < BFGPU_NUM_OPTS; i++) opt[i] = options[i];
}
// `BfProver::verify` (crates/prover/src/verify.rs:10-36) above `StarkMachine::verify` (crates/stark/src/machine.rs:258-284): the two
// checks the reference makes on the proof before the shard verifier runs — the Cpu chip must be in `chip_ordering`
// (MissingCpuInFirstShard) and its log degree must not exceed MAX_CPU_LOG_DEGREE = 22 (crates/core/machine/src/cpu/mod.rs:8: the LogUp
// multiplicities must not overflow; CpuLogDegreeTooLarge) — then `verify_shard`, whose errors come back as "InvalidShardProof: ...".
static std::string core_precheck(const uint32_t* proof, uint64_t n_words) {
    constexpr uint32_t MAX_CPU_LOG_DEGREE = 22;
    // header of the serialisation: three commitments (24 words), the chip count, then (chip, log_degree, cumulative sum[4]) per chip
    const int cpu = chip_index("Cpu");
    const uint64_t n_chips = n_words > 24 ? proof[24] : 0;
    bool has_cpu = false;
    uint32_t log_degree_cpu = 0;
    for (uint64_t i = 0; i < n_chips && i < (uint64_t)air::NUM_CHIPS && 25 + 6 * i + 1 < n_words; i++)
        if ((int)proof[25 + 6 * i] == cpu && !has_cpu) {
            has_cpu = true;
            log_degree_cpu = proof[25 + 6 * i + 1];
        }
    if (!has_cpu) return "MissingCpuInFirstShard";
    if (log_degree_cpu > MAX_CPU_LOG_DEGREE) return fmt("CpuLogDegreeTooLarge: %u", log_degree_cpu);
    return "";
}
// the shard verifier's error as bfgpu_verify_core_proof reports it (the inner message is held in a 256-byte buffer)
static inline std::string core_wrap(const std::string& inner) { return inner.empty() ? inner : "InvalidShardProof: " + inner.substr(0, 255); }
static void say(char* err, uint64_t err_len, const std::string& s) {
    if (err && err_len) snprintf(err, (size_t)err_len, "%s", s.c_str());
}
}  // namespace verifier

// vk = preprocessed commitment + (chip name, log height) of every preprocessed trace in proving-key order.
// repr: representation of vk_commit and of the proof words (BFGPU_REPR_*).  Returns BFGPU_OK when the proof is accepted;
// otherwise BFGPU_ERR_INVALID with the reference's error name in `err`.
extern "C" int32_t bfgpu_verify_shard_ex(const uint32_t vk_commit[8], const char* const* prep_names, const uint32_t* prep_log_heights, int32_t n_prep,
                                         const uint32_t* proof, uint64_t n_words, int repr, uint32_t log_blowup, uint32_t num_queries, uint32_t pow_bits,
                                         const uint32_t* options, int32_t n_options, char* err, uint64_t err_len) {
    if (!vk_commit || !proof || n_prep < 0 || (n_prep && (!prep_names || !prep_log_heights))) {
        verifier::say(err, err_len, "null argument");
        return BFGPU_ERR_INVALID;
    }
    std::vector<std::pair<int, unsigned>> prep;
    std::string e = verifier::parse_prep(prep_names, prep_log_heights, n_prep, prep);
    if (!e.empty()) {
        verifier::say(err, err_len, e);
        return BFGPU_ERR_INVALID;
    }
    uint32_t opt[BFGPU_NUM_OPTS];
    verifier::parse_options(options, n_options, opt);
    e = verifier::verify(vk_commit, prep, proof, n_words, repr == BFGPU_REPR_MONTY, log_blowup, num_queries, pow_bits, opt);
    verifier::say(err, err_len, e);
    return e.empty() ? BFGPU_OK : BFGPU_ERR_INVALID;
}
extern "C" int32_t bfgpu_verify_shard(const uint32_t vk_commit[8], const char* const* prep_names, const uint32_t* prep_log_heights, int32_t n_prep,
                                      const uint32_t* proof, uint64_t n_words, int repr, uint32_t log_blowup, uint32_t num_queries, uint32_t pow_bits,
                                      char* err, uint64_t err_len) {
    return bfgpu_verify_shard_ex(vk_commit, prep_names, prep_log_heights, n_prep, proof, n_words, repr, log_blowup, num_queries, pow_bits, nullptr, 0, err,
                                 err_len);
}

// bfgpu_verify_shard_ex behind verifier::core_precheck (`BfProver::verify`)
extern "C" int32_t bfgpu_verify_core_proof(const uint32_t vk_commit[8], const char* const* prep_names, const uint32_t* prep_log_heights, int32_t n_prep,
                                           const uint32_t* proof, uint64_t n_words, int repr, uint32_t log_blowup, uint32_t num_queries, uint32_t pow_bits,
                                           const uint32_t* options, int32_t n_options, char* err, uint64_t err_len) {
    if (!vk_commit || !proof) {
        verifier::say(err, err_len, "null argument");
        return BFGPU_ERR_INVALID;
    }
    std::string e = verifier::core_precheck(proof, n_words);
    if (!e.empty()) {
        verifier::say(err, err_len, e);
        return BFGPU_ERR_INVALID;
    }
    char inner[256] = {0};
    int32_t rc = bfgpu_verify_shard_ex(vk_commit, prep_names, prep_log_heights, n_prep, proof, n_words, repr, log_blowup, num_queries, pow_bits, options,
                                       n_options, inner, sizeof inner);
    verifier::say(err, err_len, rc == BFGPU_OK ? std::string() : std::string("InvalidShardProof: ") + inner);
    return rc;
}

// ---- canonical proof serialiser: the bytes `bincode::serialize(&MachineProof)` writes (SURVEY.md §8f.2) ------------------------------
// The reference measures `proofSize` as the length of `bincode::serialize(&proof)` (crates/core/machine/src/utils/prove.rs:47-56) over
// `MachineProof { shard_proof: ShardProof { commitment, opened_values, opening_proof, chip_ordering } }` (crates/stark/src/types.rs:32-73,
// 116-119).  bincode 1.x defaults: little endian, fixed-width integers, u64 for usize / lengths, arrays without a length prefix,
// strings as u64 length + bytes, maps as u64 count + (key, value) pairs.  Plonky3 types inside (P3: restated from the published
// v0.1.0 sources): Hash<F, W, 8> = [W; 8]; BinomialExtensionField = [F; 4]; FriProof { commit_phase_commits, query_proofs, final_poly,
// pow_witness }; QueryProof { input_proof: Vec<BatchOpening { opened_values: Vec<Vec<F>>, opening_proof: Vec<[F; 8]> }>,
// commit_phase_openings: Vec<CommitPhaseProofStep { sibling_value, opening_proof: Vec<[F; 8]> }> }.  A field element is one u32:
// field_repr 1 writes the Montgomery word (p3-monty-31 serialises `self.value` "in monty form"), 0 the canonical residue.
// `chip_ordering` is a hashbrown map whose iteration order is random per process in the reference (SURVEY.md §0.4): here it is
// written in chip order, which makes the encoding canonical; the byte COUNT does not depend on the order.
namespace verifier {
struct ByteSink {
    uint8_t* out;
    uint64_t cap, len = 0;
    void put(const void* p, size_t n) {
        if (out && len + n <= cap) memcpy(out + len, p, n);
        len += n;
    }
    void u64(uint64_t v) { put(&v, 8); }  // little-endian hosts only (x86-64 / aarch64 LE)
    void u32(uint32_t v) { put(&v, 4); }
};
static std::string to_bincode(const std::vector<std::pair<int, unsigned>>& prep, const uint32_t* words, uint64_t n_words, bool monty, unsigned log_blowup,
                              int field_repr, ByteSink& sink) {
    Reader rd{words, n_words, 0, monty};
    auto fe = [&](uint32_t mont) { sink.u32(field_repr == 1 ? mont : kb::from_mont(mont)); };
    auto ext = [&](const Ext& e) { for (int k = 0; k < 4; k++) fe(e.c[k]); };
    uint32_t commits[3][8];
    for (auto& c : commits) rd.digest(c);
    const uint32_t n = rd.raw();
    if (!rd.ok || n == 0 || n > (uint32_t)air::NUM_CHIPS) return "ChipOpeningLengthMismatch";
    struct ChipOpen { int chip; unsigned log_degree; Ext csum; };
    std::vector<ChipOpen> chips(n);
    std::map<int, size_t> where;
    for (auto& c : chips) {
        c.chip = (int)rd.raw();
        c.log_degree = rd.raw();
        c.csum = rd.ext();
        if (!rd.ok || c.chip < 0 || c.chip >= air::NUM_CHIPS || c.log_degree > (unsigned)kb::TWO_ADICITY || where.count(c.chip)) return "InvalidProofShape";
        where[c.chip] = &c - chips.data();
    }
    for (auto& pr : prep)
        if (!where.count(pr.first)) return "InvalidProofShape: preprocessed chip missing from the proof";
    // opened values in serialisation order: preprocessed (pk order), then main, permutation, quotient per chip
    auto read_vals = [&](uint32_t width, bool both, std::vector<Ext>* local, std::vector<Ext>* next) {
        local->resize(width);
        for (auto& e : *local) e = rd.ext();
        next->assign(width, kb::ext_zero());  // local-only chips: `next` is a vector of zeros of the same width (prover.rs:485-487)
        if (both)
            for (auto& e : *next) e = rd.ext();
    };
    std::vector<std::vector<Ext>> pl(n), pn(n), ml(n), mn(n), ql(n), qn(n);
    std::vector<std::vector<std::vector<Ext>>> quot(n);
    for (auto& pr : prep) {
        size_t i = where[pr.first];
        read_vals((uint32_t)air::CHIPS[pr.first].prep_w, !air::CHIPS[pr.first].local_only, &pl[i], &pn[i]);
    }
    for (size_t i = 0; i < n; i++) read_vals((uint32_t)air::CHIPS[chips[i].chip].main_w, !air::CHIPS[chips[i].chip].local_only, &ml[i], &mn[i]);
    for (size_t i = 0; i < n; i++) read_vals(4u * (uint32_t)air::CHIPS[chips[i].chip].perm_w, true, &ql[i], &qn[i]);
    for (size_t i = 0; i < n; i++)
        for (int d = 0; d < (1 << air::CHIPS[chips[i].chip].log_quotient_degree); d++) {
            std::vector<Ext> v(4);
            for (auto& e : v) e = rd.ext();
            quot[i].push_back(v);
        }
    if (!rd.ok) return "InvalidProofShape: truncated opened values";
    // ---- MachineProof.shard_proof.commitment
    for (auto& c : commits)
        for (int k = 0; k < 8; k++) fe(c[k]);
    // ---- opened_values: ShardOpenedValues { chips: Vec<ChipOpenedValues> }
    auto vec_ext = [&](const std::vector<Ext>& v) {
        sink.u64(v.size());
        for (auto& e : v) ext(e);
    };
    sink.u64(n);
    for (size_t i = 0; i < n; i++) {
        vec_ext(pl[i]); vec_ext(pn[i]);   // preprocessed { local, next } (empty vectors for chips without a preprocessed trace)
        vec_ext(ml[i]); vec_ext(mn[i]);   // main
        vec_ext(ql[i]); vec_ext(qn[i]);   // permutation
        sink.u64(quot[i].size());          // quotient: Vec<Vec<Challenge>>
        for (auto& v : quot[i]) vec_ext(v);
        ext(chips[i].csum);
        sink.u64(chips[i].log_degree);
    }
    // ---- opening_proof: FriProof
    const uint32_t n_commit = rd.raw();
    if (!rd.ok || n_commit == 0 || n_commit > (unsigned)kb::TWO_ADICITY) return "InvalidProofShape";
    sink.u64(n_commit);
    for (uint32_t k = 0; k < n_commit; k++) {
        uint32_t d[8];
        rd.digest(d);
        for (int j = 0; j < 8; j++) fe(d[j]);
    }
    const Ext final_poly = rd.ext();
    const uint32_t pow_witness = rd.raw();  // canonical in the flat layout
    const uint32_t nq = rd.raw();
    if (!rd.ok || pow_witness >= kb::P) return "InvalidProofShape";
    const unsigned log_max = n_commit + log_blowup;
    // round shapes: [preprocessed (pk order), main, permutation, quotient]
    struct Shape { std::vector<std::pair<unsigned, uint32_t>> mats; };  // (log LDE height, width)
    Shape rounds[4];
    for (auto& pr : prep) rounds[0].mats.push_back({pr.second + log_blowup, (uint32_t)air::CHIPS[pr.first].prep_w});
    for (auto& c : chips) {
        const auto& info = air::CHIPS[c.chip];
        rounds[1].mats.push_back({c.log_degree + log_blowup, (uint32_t)info.main_w});
        rounds[2].mats.push_back({c.log_degree + log_blowup, 4u * (uint32_t)info.perm_w});
        for (int d = 0; d < (1 << info.log_quotient_degree); d++) rounds[3].mats.push_back({c.log_degree + log_blowup, 4u});
    }
    sink.u64(nq);
    for (uint32_t q = 0; q < nq; q++) {
        (void)rd.raw();  // the query index is not part of QueryProof: the verifier re-derives it from the transcript
        sink.u64(4);      // input_proof: one BatchOpening per commitment round
        for (auto& r : rounds) {
            unsigned lmax = 0;
            sink.u64(r.mats.size());
            for (auto& m : r.mats) {
                lmax = std::max(lmax, m.first);
                sink.u64(m.second);
                for (uint32_t c = 0; c < m.second; c++) fe(rd.fe());
            }
            if (lmax > log_max) return "InvalidProofShape: matrix taller than the FRI domain";
            sink.u64(lmax);
            for (unsigned l = 0; l < lmax; l++) {
                uint32_t d[8];
                rd.digest(d);
                for (int j = 0; j < 8; j++) fe(d[j]);
            }
        }
        sink.u64(n_commit);  // commit_phase_openings
        for (uint32_t k = 0; k < n_commit; k++) {
            ext(rd.ext());
            const unsigned lfh = log_max - 1 - k;
            sink.u64(lfh);
            for (unsigned l = 0; l < lfh; l++) {
                uint32_t d[8];
                rd.digest(d);
                for (int j = 0; j < 8; j++) fe(d[j]);
            }
        }
        if (!rd.ok) return "InvalidProofShape: truncated query";
    }
    ext(final_poly);
    fe(kb::to_mont(pow_witness));
    if (rd.pos != rd.n) return "InvalidProofShape: trailing words";
    // ---- chip_ordering: HashMap<String, usize>, written in chip order
    sink.u64(n);
    for (size_t i = 0; i < n; i++) {
        const char* name = air::CHIPS[chips[i].chip].name;
        sink.u64(strlen(name));
        sink.put(name, strlen(name));
        sink.u64(i);
    }
    return "";
}
}  // namespace verifier

// out == NULL: only the length (the reference's `proofSize`).  Returns BFGPU_ERR_INVALID with a message in err for malformed input,
// BFGPU_ERR_STATE when out_cap is too small (out_len still holds the needed size).
extern "C" int32_t bfgpu_shard_proof_to_bincode(const char* const* prep_names, const uint32_t* prep_log_heights, int32_t n_prep, const uint32_t* proof,
                                                uint64_t n_words, int repr, uint32_t log_blowup, int field_repr, uint8_t* out, uint64_t out_cap,
                                                uint64_t* out_len, char* err, uint64_t err_len) {
    auto say = [&](const std::string& s) {
        if (err && err_len) snprintf(err, (size_t)err_len, "%s", s.c_str());
    };
    if (!proof || !out_len || n_prep < 0 || (n_prep && (!prep_names || !prep_log_heights))) {
        say("null argument");
        return BFGPU_ERR_INVALID;
    }
    std::vector<std::pair<int, unsigned>> prep;
    for (int i = 0; i < n_prep; i++) {
        int ci = chip_index(prep_names[i]);
        if (ci < 0) {
            say(std::string("unknown chip ") + prep_names[i]);
            return BFGPU_ERR_INVALID;
        }
        prep.emplace_back(ci, prep_log_heights[i]);
    }
    verifier::ByteSink sink{out, out_cap};
    std::string e = verifier::to_bincode(prep, proof, n_words, repr == BFGPU_REPR_MONTY, log_blowup, field_repr, sink);
    say(e);
    if (!e.empty()) return BFGPU_ERR_INVALID;
    *out_len = sink.len;
    return (out && sink.len > out_cap) ? BFGPU_ERR_STATE : BFGPU_OK;
}
