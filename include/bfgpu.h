/* bfgpu.h — C ABI of the B200-native proving backend for zkvm-brainfuck.
 *
 * This is the drop-in boundary: a Rust `bf-gpu-sys` crate (see INTEGRATION.md) binds these symbols
 * and implements, on top of them, the traits the reference prover is generic over:
 *
 *   TwoAdicSubgroupDft<KoalaBear>      (alias `Dft`,     reference crates/stark/src/kb31_poseidon2.rs:30)
 *   Mmcs<KoalaBear>                    (alias `ValMmcs`, reference crates/stark/src/kb31_poseidon2.rs:27-28)
 *   Pcs<Challenge, Challenger>         (alias `Pcs`,     reference crates/stark/src/kb31_poseidon2.rs:32;
 *                                       call sites crates/stark/src/prover.rs:227,334,365-373,411,461
 *                                       and crates/stark/src/machine.rs:196)
 *   MachineProver::{commit, open}      (reference crates/stark/src/prover.rs:27-150,209-553)
 *
 * Conventions
 *  - every function returns 0 on success and a negative bfgpu_status on failure;
 *    bfgpu_last_error(ctx) returns a human-readable message for the last failure on that context.
 *    Nothing unwinds across the boundary.  (The reference's error type is the unit struct
 *    `CpuProverError`, prover.rs:166-168; its callers unwrap.)
 *  - host buffers are caller-owned and only borrowed for the duration of the call;
 *    device objects are opaque handles released by the matching *_free.
 *  - field elements cross as raw uint32_t.  `BFGPU_REPR_MONTY` (default for the Rust shim) is the
 *    in-memory representation of `Vec<KoalaBear>` (Montgomery form, R = 2^32);
 *    `BFGPU_REPR_CANONICAL` is the plain residue in [0, p) and is what the Python/ctypes test
 *    harness uses.  Select with bfgpu_set_repr().
 *  - matrices are ROW-MAJOR rows x cols, exactly like Plonky3's RowMajorMatrix<KoalaBear>.
 *  - extension-field elements (BinomialExtensionField<KoalaBear,4>) are 4 consecutive words,
 *    coefficients of X^0..X^3.
 *  - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *    BFGPU_ERR_CUDA.
 */
#ifndef BFGPU_H
#define BFGPU_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    BFGPU_OK = 0,
    BFGPU_ERR_INVALID = -1, /* bad argument (shape not a power of two, null pointer, ...) */
    BFGPU_ERR_CUDA = -2,    /* CUDA runtime error or no device */
    BFGPU_ERR_OOM = -3,     /* device allocation failed */
    BFGPU_ERR_STATE = -4    /* object used in the wrong state */
} bfgpu_status;

enum { BFGPU_REPR_CANONICAL = 0, BFGPU_REPR_MONTY = 1 };
enum { BFGPU_MEM_HOST = 0, BFGPU_MEM_DEVICE = 1 };

typedef struct bfgpu_ctx bfgpu_ctx;
typedef struct bfgpu_tree bfgpu_tree;         /* Mmcs::ProverData  (MerkleTree)            */
typedef struct bfgpu_pcs_data bfgpu_pcs_data; /* Pcs::ProverData   (LDE matrices + MerkleTree) */

/* A row-major matrix of base-field words living in host or device memory. */
typedef struct {
    const uint32_t* data;
    uint64_t rows;
    uint64_t cols;
} bfgpu_mat;

/* ---- context ---------------------------------------------------------------------------------- */
/* Replaces the construction of the config object `KoalaBearPoseidon2::new()`
 * (crates/stark/src/kb31_poseidon2.rs:73-85): builds the Poseidon2 constant bank (my_perm, :35-50),
 * the twiddle table and the FRI parameters (default_fri_config, :54-64: log_blowup 1,
 * num_queries from $FRI_QUERIES or 84, proof_of_work_bits 16). */
int32_t bfgpu_ctx_create(int device, bfgpu_ctx** out);
void bfgpu_ctx_destroy(bfgpu_ctx* ctx);
const char* bfgpu_last_error(const bfgpu_ctx* ctx);
int32_t bfgpu_set_repr(bfgpu_ctx* ctx, int repr);
/* where input matrices passed to the compute entry points live (default BFGPU_MEM_HOST) */
int32_t bfgpu_set_input_space(bfgpu_ctx* ctx, int mem_space);
/* run all work of this context on an existing CUDA stream (cudaStream_t); NULL = own stream */
int32_t bfgpu_set_stream(bfgpu_ctx* ctx, void* cuda_stream);
int32_t bfgpu_synchronize(bfgpu_ctx* ctx);
int32_t bfgpu_set_fri_params(bfgpu_ctx* ctx, uint32_t log_blowup, uint32_t num_queries, uint32_t pow_bits);
/* Transcript options: every choice INSIDE Plonky3 (git dependency pinned at rev 93967fce, not vendored: SURVEY.md "P3" marks) that the
 * restatement could not confirm offline is a switch here, mirrored by the native verifier (bfgpu_verify_shard_ex) and by the
 * CPU oracle, so that pinning against the real Rust prover flips a flag instead of rewriting kernels.  Defaults = Plonky3 of the
 * pinned API era as published.
 *   OBSERVE_OPENED_VALUES 1: TwoAdicFriPcs::open/verify write every opened value into the challenger before sampling alpha; 0: they do not
 *   FRI_ROLLIN            0: a reduced opening joins the folded vector as `folded[i] += ro[i]`; 1: as `folded[i] += beta^2 * ro[i]`
 *   POW_ORDER             0: grind returns the smallest witness; 1: the largest (the reference's rayon find_any returns any valid one) */
enum { BFGPU_OPT_OBSERVE_OPENED_VALUES = 0, BFGPU_OPT_FRI_ROLLIN = 1, BFGPU_OPT_POW_ORDER = 2, BFGPU_NUM_OPTS = 3 };
int32_t bfgpu_set_transcript_option(bfgpu_ctx* ctx, int32_t option, uint32_t value);
/* number of this library's kernels launched on the context since creation (bench evidence) */
uint64_t bfgpu_launch_count(const bfgpu_ctx* ctx);
/* test hooks for the error paths: number of device blocks the context currently has handed out, and "the nth device allocation
 * from now fails with BFGPU_ERR_OOM" (nth < 0 disarms).  A failed entry point must leave live_blocks where it found it. */
uint64_t bfgpu_debug_live_blocks(const bfgpu_ctx* ctx);
int32_t bfgpu_debug_fail_alloc(bfgpu_ctx* ctx, int64_t nth);

/* page-locked host memory for caller matrices: cudaMemcpyAsync from pageable memory is staged by the driver at
 * ~11 GB/s, from pinned memory it runs at PCIe speed (~55 GB/s measured).  Trace generators should write
 * straight into such buffers. */
int32_t bfgpu_host_alloc(bfgpu_ctx* ctx, uint64_t bytes, void** out);
void bfgpu_host_free(void* p);

/* ---- measurement hooks (bench.py): per-phase device time via CUDA events on the context's stream -- */
enum {
    BFGPU_PHASE_H2D = 0,      /* host -> device copies of caller matrices                     */
    BFGPU_PHASE_INGEST = 1,   /* row-major -> column-major Montgomery (+ bit-reversed gather)   */
    BFGPU_PHASE_INTT = 2,     /* inverse NTT passes                                            */
    BFGPU_PHASE_SCALE = 3,    /* coset shift / 1/n scaling and zero-free 2x expansion          */
    BFGPU_PHASE_NTT = 4,      /* forward NTT passes                                            */
    BFGPU_PHASE_LEAF = 5,     /* Poseidon2 sponge over LDE rows (first digest layer)           */
    BFGPU_PHASE_COMPRESS = 6, /* Poseidon2 2-to-1 compression layers (+ injected rows)         */
    BFGPU_PHASE_OTHER = 7,
    BFGPU_PHASE_OPEN_EVAL = 8,   /* barycentric evaluation of all columns at the opening points     */
    BFGPU_PHASE_OPEN_REDUCE = 9, /* per-height reduced openings                                     */
    BFGPU_PHASE_FRI = 10,        /* FRI commit phase: fold + Merkle commit per round                */
    BFGPU_PHASE_POW = 11,        /* proof-of-work grind                                             */
    BFGPU_PHASE_QUERY = 12,      /* query gathers                                                   */
    BFGPU_PHASE_PERM = 13,       /* LogUp permutation trace                                         */
    BFGPU_PHASE_QUOTIENT = 14,   /* quotient values                                                 */
    BFGPU_PHASE_EXCHANGE = 15,   /* multi-GPU commit: launches of the column->row exchange (they run on the copy stream) */
    BFGPU_PHASE_TRACEGEN = 16,   /* device-side trace generation from the execution record                          */
    BFGPU_PHASE_DEBUG_ROWS = 17,    /* trace checker: constraint pass (bfgpu_machine_debug)                          */
    BFGPU_PHASE_DEBUG_LOOKUPS = 18, /* trace checker: interaction pass (records, sort, reduction, gather)            */
    BFGPU_PHASE_VERIFY = 19,        /* batch verifier: plan upload, query checks, result bits back (bfgpu_verify_batch) */
    BFGPU_NUM_PHASES = 20
};
/* start (on != 0, clears the accumulators) or stop collecting per-phase timings */
int32_t bfgpu_profile_enable(bfgpu_ctx* ctx, int on);
/* synchronises, then returns accumulated milliseconds and kernel-launch counts per phase */
int32_t bfgpu_profile_read(bfgpu_ctx* ctx, float ms[BFGPU_NUM_PHASES], uint64_t launches[BFGPU_NUM_PHASES]);
/* register-only integer microbenchmark (IMAD + IADD3/LOP3 mix, no memory traffic): measured
 * thread-level integer instructions per second, the denominator for the Poseidon2 roofline */
int32_t bfgpu_int32_peak_probe(bfgpu_ctx* ctx, double* giops);

/* ---- Poseidon2 primitives (Perm / MyHash / MyCompress, kb31_poseidon2.rs:22-26) -------------- */
/* n independent width-16 permutations, states row-major n x 16, in place */
int32_t bfgpu_poseidon2_permute(bfgpu_ctx* ctx, uint32_t* states, uint64_t n);
/* PaddingFreeSponge::hash_iter over each row of a rows x cols matrix -> rows x 8 digests */
int32_t bfgpu_sponge_hash_rows(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t* digests);
/* TruncatedPermutation::compress on n pairs: left/right n x 8 -> out n x 8 */
int32_t bfgpu_compress(bfgpu_ctx* ctx, const uint32_t* left, const uint32_t* right, uint64_t n, uint32_t* out);

/* ---- TwoAdicSubgroupDft<KoalaBear> ----------------------------------------------------------- */
/* coset_lde_batch(mat, added_bits, shift): evaluations of every column's interpolant (given on the
 * order-`rows` subgroup, natural order) over shift*<w_{rows<<added_bits}>.  out is
 * (rows<<added_bits) x cols; bit_reversed_rows != 0 gives the row order TwoAdicFriPcs::commit
 * stores (`.bit_reverse_rows()`), 0 gives natural order as the trait method returns it. */
int32_t bfgpu_coset_lde_batch(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t added_bits, uint32_t shift,
                              int bit_reversed_rows, uint32_t* out);
int32_t bfgpu_dft_batch(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t* out);  /* natural in / out */
int32_t bfgpu_idft_batch(bfgpu_ctx* ctx, const bfgpu_mat* mat, uint32_t* out); /* natural in / out */

/* ---- Mmcs<KoalaBear> = MerkleTreeMmcs<.., MyHash, MyCompress, 8> ----------------------------- */
/* Mmcs::commit: heights must be powers of two.  root is 8 words. */
int32_t bfgpu_mmcs_commit(bfgpu_ctx* ctx, const bfgpu_mat* mats, int32_t n, uint32_t root[8], bfgpu_tree** out);
/* Mmcs::open_batch(index): opened_rows receives, back to back in input-matrix order, row
 * `index >> (log_max_height - log_height_i)` of each matrix; siblings receives log_max_height
 * digests (8 words each), leaf level first. */
int32_t bfgpu_mmcs_open_batch(bfgpu_tree* tree, uint64_t index, uint32_t* opened_rows, uint32_t* siblings);
/* introspection used by the parity tests */
int32_t bfgpu_tree_num_layers(const bfgpu_tree* tree);
uint64_t bfgpu_tree_layer_len(const bfgpu_tree* tree, int32_t layer);
int32_t bfgpu_tree_get_layer(bfgpu_tree* tree, int32_t layer, uint32_t* digests /* len x 8 */);
void bfgpu_tree_free(bfgpu_tree* tree);

/* ---- Pcs = TwoAdicFriPcs<Val, Dft, ValMmcs, ChallengeMmcs> ----------------------------------- */
/* Pcs::commit(Vec<(Domain, RowMajorMatrix<Val>)>) (prover.rs:227,334,411; machine.rs:196).
 * domain_shifts[i] is the shift of matrix i's two-adic coset domain (NULL = all natural domains,
 * shift 1); the LDE uses shift GENERATOR/domain_shift and the context's log_blowup.  The LDEs
 * and the tree stay on the device inside *out. */
int32_t bfgpu_pcs_commit(bfgpu_ctx* ctx, const bfgpu_mat* evals, const uint32_t* domain_shifts, int32_t n,
                         uint32_t root[8], bfgpu_pcs_data** out);
int32_t bfgpu_pcs_num_matrices(const bfgpu_pcs_data* data);
int32_t bfgpu_pcs_lde_dims(const bfgpu_pcs_data* data, int32_t idx, uint64_t* rows, uint64_t* cols);
/* Pcs::get_evaluations_on_domain(data, idx, domain) for the disjoint domain of size rows<<log_blowup
 * and shift GENERATOR (prover.rs:365-373): the whole LDE, rows in NATURAL order
 * (bit_reversed_rows = 0) or as stored (1).  Test/debug path: the prover kernels read the device
 * copy in place. */
int32_t bfgpu_pcs_get_evaluations(bfgpu_pcs_data* data, int32_t idx, int bit_reversed_rows, uint32_t* out);
bfgpu_tree* bfgpu_pcs_tree(bfgpu_pcs_data* data); /* borrowed; freed with the pcs data */
void bfgpu_pcs_data_free(bfgpu_pcs_data* data);

/* ---- one Pcs::commit over several GPUs (one process / context per GPU) -------------------------------- */
/* Shards `TwoAdicFriPcs::commit` (prover.rs:227,334,411) as SURVEY.md §8e lays out: rank r LDEs columns
 * [W*r/G, W*(r+1)/G) of every matrix, the LDE blocks are stored straight into the peers' row-shard matrices
 * over NVLink (CUDA IPC mappings; no library collective on the data path), rank r hashes LDE rows
 * [r*h/G, (r+1)*h/G) and builds subtree r of the Merkle tree, and the G subtree caps (32 B each) plus the
 * top log2(G) levels give the same root as the single-GPU commit.  The caller's plumbing
 * (torch.distributed in the Python mirror, any byte all-gather + barrier in a Rust shim) moves only the
 * 64-byte buffer handles and the caps.  Call order on every rank:
 *   begin -> recv_handle -> [all-gather handles] -> set_peers -> lde -> bfgpu_synchronize -> [barrier]
 *         -> finish -> [all-gather caps] -> root          (open_batch any time after root)
 * Staged mode (baseline for comparison): set_staging instead of set_peers, then the caller runs an
 * all-to-all of block_words()-sized blocks between lde and unpack. */
typedef struct bfgpu_dist_commit bfgpu_dist_commit;
int32_t bfgpu_dist_commit_begin(bfgpu_ctx* ctx, uint32_t rank, uint32_t world, const uint64_t* rows, const uint32_t* total_cols,
                                int32_t n, bfgpu_dist_commit** out);
/* number of columns of matrix i this rank owns (and the first one's global index) */
uint32_t bfgpu_dist_commit_local_cols(const bfgpu_dist_commit* dc, int32_t i, uint32_t* col0);
int32_t bfgpu_dist_commit_recv_handle(bfgpu_dist_commit* dc, uint8_t handle[64]);
int32_t bfgpu_dist_commit_set_peers(bfgpu_dist_commit* dc, const uint8_t* handles /* world x 64 */);
uint64_t bfgpu_dist_commit_block_words(const bfgpu_dist_commit* dc, uint32_t src_rank);
int32_t bfgpu_dist_commit_set_staging(bfgpu_dist_commit* dc, uint32_t* dev_send /* world x block_words(rank) words */);
/* local[i]: rows[i] x local_cols(i) row-major slice in the context's input space; domain_shifts as bfgpu_pcs_commit */
int32_t bfgpu_dist_commit_lde(bfgpu_dist_commit* dc, const bfgpu_mat* local, const uint32_t* domain_shifts);
int32_t bfgpu_dist_commit_unpack(bfgpu_dist_commit* dc, const uint32_t* dev_recv /* sum_src block_words(src) words */);
int32_t bfgpu_dist_commit_finish(bfgpu_dist_commit* dc, uint32_t cap[8]);
int32_t bfgpu_dist_commit_root(bfgpu_dist_commit* dc, const uint32_t* caps /* world x 8 */, uint32_t root[8]);
/* Mmcs::open_batch for a global leaf index owned by this rank (index / rows_per_rank == rank) */
int32_t bfgpu_dist_commit_open_batch(bfgpu_dist_commit* dc, uint64_t index, uint32_t* opened_rows, uint32_t* siblings);
uint64_t bfgpu_dist_commit_rows_per_rank(const bfgpu_dist_commit* dc);
void bfgpu_dist_commit_free(bfgpu_dist_commit* dc);

/* ---- Challenger = DuplexChallenger<Val, Perm, 16, 8> (kb31_poseidon2.rs:31,126-128) ------------ */
/* Host-side sponge (the transcript is sequential and tiny); the library advances it exactly as the
 * reference's prover does (prover.rs:266-272,337-340,354,412-415,595-601 and inside Pcs::open).  A
 * Rust shim keeps its own DuplexChallenger authoritative by copying the public fields
 * (sponge_state, input_buffer, output_buffer) in and out with the import/export calls. */
typedef struct bfgpu_challenger bfgpu_challenger;
int32_t bfgpu_challenger_create(bfgpu_ctx* ctx, bfgpu_challenger** out);
int32_t bfgpu_challenger_clone(const bfgpu_challenger* ch, bfgpu_challenger** out);
void bfgpu_challenger_free(bfgpu_challenger* ch);
int32_t bfgpu_challenger_observe(bfgpu_challenger* ch, const uint32_t* values, uint64_t n);
int32_t bfgpu_challenger_sample(bfgpu_challenger* ch, uint32_t* out, uint64_t n); /* n base samples (4 = one ext element) */
int32_t bfgpu_challenger_sample_bits(bfgpu_challenger* ch, uint32_t bits, uint32_t* out);
/* state = 16 words, input/output buffers up to 8 words each (caller representation) */
int32_t bfgpu_challenger_export(const bfgpu_challenger* ch, uint32_t state[16], uint32_t input[8], uint32_t* n_input,
                                uint32_t output[8], uint32_t* n_output);
int32_t bfgpu_challenger_import(bfgpu_challenger* ch, const uint32_t state[16], const uint32_t* input, uint32_t n_input,
                                const uint32_t* output, uint32_t n_output);

/* ---- Pcs::open (prover.rs:460-470) ---------------------------------------------------------------- */
/* One entry per commitment ("round"): the prover data and, for every matrix of that commitment in
 * commit order, its opening points (num_points[i] extension elements, 4 words each, concatenated). */
typedef struct {
    bfgpu_pcs_data* data;
    const uint32_t* num_points;
    const uint32_t* points;
} bfgpu_open_round;
typedef struct bfgpu_opening bfgpu_opening; /* OpenedValues + FriProof */
/* Evaluates every column at its points (barycentric, low coset), observes the opened values,
 * samples alpha, builds the per-height reduced openings, runs the FRI commit phase (fold + commit per
 * round, roots observed / betas sampled on `ch`), grinds the proof of work (the smallest witness; any
 * valid one is accepted by the verifier; pass fixed_pow_witness >= 0 to reuse a known one) and answers
 * the queries. */
int32_t bfgpu_pcs_open(bfgpu_ctx* ctx, const bfgpu_open_round* rounds, int32_t n_rounds, bfgpu_challenger* ch,
                       int64_t fixed_pow_witness, bfgpu_opening** out);
/* Flat u32 serialisation (caller representation):
 *   for round, matrix, point: width x 4 words of opened values
 *   n_commit_phase_commits, then 8 words per commit; final_poly (4); pow_witness (1, canonical); n_queries
 *   per query: index; per round: opened row of every matrix (sum of widths), siblings (8 x log2(max height));
 *              per FRI layer i: sibling_value (4), opening proof (8 x log2(layer leaves)) */
uint64_t bfgpu_opening_size(const bfgpu_opening* o);
int32_t bfgpu_opening_read(const bfgpu_opening* o, uint32_t* out);
void bfgpu_opening_free(bfgpu_opening* o);

/* ---- MachineProver<SC, BfAir> (prover.rs:27-150): setup / commit / open ------------------------------ */
/* The eight chips of the machine (crates/core/machine/src/brainfuck/mod.rs:53-81) are compiled into the
 * library as generated constraint / LogUp programs (csrc/gen_air.cuh from air/chips.py). */
int32_t bfgpu_machine_num_chips(void);
int32_t bfgpu_machine_chip_info(int32_t i, const char** name, int32_t* main_width, int32_t* prep_width, int32_t* perm_ext_width,
                                int32_t* local_only);
typedef struct bfgpu_pk bfgpu_pk;                   /* DeviceProvingKey: preprocessed traces + LDE + Merkle tree */
typedef struct bfgpu_shard bfgpu_shard;             /* ShardMainData: main traces + LDE + Merkle tree             */
typedef struct bfgpu_shard_proof bfgpu_shard_proof; /* ShardProof                                                  */
/* StarkMachine::setup (machine.rs:154-224): named preprocessed traces (chip name -> matrix); they are sorted by
 * (height desc, name) and committed.  commit receives the preprocessed commitment. */
int32_t bfgpu_machine_setup(bfgpu_ctx* ctx, const char* const* names, const bfgpu_mat* prep_traces, int32_t n, uint32_t commit[8],
                            bfgpu_pk** out);
/* StarkProvingKey::observe_into (prover.rs:595-601) */
int32_t bfgpu_pk_observe_into(const bfgpu_pk* pk, bfgpu_challenger* ch);
void bfgpu_pk_free(bfgpu_pk* pk);
/* MachineProver::commit (prover.rs:209-236): named main traces of the included chips */
int32_t bfgpu_machine_commit(bfgpu_ctx* ctx, const char* const* names, const bfgpu_mat* traces, int32_t n, uint32_t root[8],
                             bfgpu_shard** out);
void bfgpu_shard_free(bfgpu_shard* shard);
/* MachineProver::open (prover.rs:242-553): LogUp permutation traces, their commitment, quotient values and
 * commitment, and the PCS opening, advancing `ch` exactly like the reference transcript.
 * Serialisation of the proof (flat u32, caller representation):
 *   main root (8), permutation root (8), quotient root (8), n_chips,
 *   per chip in commit order: chip index (bfgpu_machine_chip_info), log_degree, cumulative_sum (4),
 *   then the bfgpu_opening layout for the rounds [preprocessed, main, permutation, quotient]. */
int32_t bfgpu_machine_open(bfgpu_ctx* ctx, const bfgpu_pk* pk, const bfgpu_shard* shard, bfgpu_challenger* ch,
                           int64_t fixed_pow_witness, bfgpu_shard_proof** out);
uint64_t bfgpu_shard_proof_size(const bfgpu_shard_proof* p);
int32_t bfgpu_shard_proof_read(const bfgpu_shard_proof* p, uint32_t* out);
void bfgpu_shard_proof_free(bfgpu_shard_proof* p);

/* Trace checker: StarkMachine::debug_constraints (machine.rs:288-387, debug.rs:24-105, lookup/debug.rs:59-196) on the GPU.  Checks
 * a committed shard without proving it: every constraint of every chip on every row (selectors exact, the next row of the last row
 * is row 0), the LogUp cumulative sums, and the balance of every interaction (sends minus receives per (kind, values) over all
 * chips).  Works on a COPY of `ch` (left unchanged): observes the main commitment and samples the LogUp (alpha, beta) exactly as
 * bfgpu_machine_open does, so for a challenger in the state bfgpu_machine_open would receive the cumulative sums are the ones the
 * proof carries; it then samples two more elements (gamma, delta) for the interaction fingerprints gamma + kind +
 * sum_k delta^(k+1) value_k.  The reference's own sampling order inside debug_constraints cannot be checked offline; it does not
 * affect the verdict, which depends on the challenges only through a fingerprint collision (probability ~ records^2 / p^4).
 * The report is deterministic.  Flat u32 serialisation (caller representation for field elements):
 *   n_chips; per chip in commit order: chip index (bfgpu_machine_chip_info), log_degree, cumulative_sum (4), n_failing,
 *     per failing constraint (ascending index k in fold order: base constraints, one per LogUp batch column, then the LogUp
 *     first-row, transition and last-row constraints): k, failing-row count, the min(count, max_rows) smallest failing natural rows;
 *   total of the cumulative sums (4);
 *   n_imbalanced; for the first min(n_imbalanced, max_keys) keys in (kind, canonical values) order: kind (LookupKind), n_values,
 *     values (n_values), net multiplicity (sends - receives), n_chips with a nonzero net, then (chip index, net) per such chip. */
typedef struct bfgpu_debug_report bfgpu_debug_report;
int32_t bfgpu_machine_debug(bfgpu_ctx* ctx, const bfgpu_pk* pk, const bfgpu_shard* shard, const bfgpu_challenger* ch, uint32_t max_rows,
                            uint32_t max_keys, bfgpu_debug_report** out);
uint64_t bfgpu_debug_report_size(const bfgpu_debug_report* r);
int32_t bfgpu_debug_report_read(const bfgpu_debug_report* r, uint32_t* out);
void bfgpu_debug_report_free(bfgpu_debug_report* r);

/* ---- plug point #2 (SURVEY.md §8b): the steps of CpuProver::open for an integration at the Plonky3 trait level ------------------------- */
/* Pcs::get_evaluations_on_domain (prover.rs:365-373) as a device view: pointer and layout of the committed LDE (column-major,
 * col_stride words between columns, rows bit-reversed, Montgomery words) — the LDE never leaves HBM. */
int32_t bfgpu_pcs_lde_device(const bfgpu_pcs_data* data, int32_t idx, const uint32_t** dev, uint64_t* rows, uint64_t* cols, uint64_t* col_stride);
/* Chip::generate_permutation_trace (chip.rs:117-136 -> permutation.rs:75-148) of one chip: perm_out = rows x 4*perm_ext_width words,
 * row-major, natural row order (the flattened matrix prover.rs:318-328 commits); challenges = LogUp alpha then beta (4 words each);
 * prep may be NULL for chips without a preprocessed trace. */
int32_t bfgpu_logup_perm_trace(bfgpu_ctx* ctx, const char* chip, const bfgpu_mat* main, const bfgpu_mat* prep, const uint32_t challenges[8],
                               uint32_t* perm_out, uint32_t cum_sum[4]);
/* quotient_values (quotient.rs:18-165) of one chip, read from the committed (device-resident) LDEs: out = 2 * trace_rows extension
 * elements (4 words each) over the quotient domain in natural order.  prep_data may be NULL (prep_idx -1). */
int32_t bfgpu_quotient_values(bfgpu_ctx* ctx, const char* chip, const bfgpu_pcs_data* prep_data, int32_t prep_idx, const bfgpu_pcs_data* main_data,
                              int32_t main_idx, const bfgpu_pcs_data* perm_data, int32_t perm_idx, const uint32_t alpha[4],
                              const uint32_t perm_challenges[8], const uint32_t cum_sum[4], uint32_t* out);

/* ---- executor + device-side trace generation (SURVEY.md §8f items 1, 4) -------------------------------------- */
/* `Program::from` + `Executor::run` (crates/core/executor/src/program.rs:22-44, executor.rs:71-79,106-325) as one
 * native pass that emits a 16-byte record per cycle; the eight `MachineAir::generate_trace` implementations and
 * `generate_dependencies` (machine.rs:228-248) run on the GPU from those records (csrc/tracegen.cuh), so only
 * 16 B/cycle cross PCIe.  ctx may be NULL for bfgpu_execute (plain host memory, no device needed).
 * max_cycles 0 = the shard limit 2^23 (clk = 2*cycle must fit the 24-bit range checks). */
typedef struct bfgpu_record bfgpu_record; /* ExecutionRecord */
int32_t bfgpu_execute(bfgpu_ctx* ctx, const char* code, const uint8_t* stdin_bytes, uint64_t n_stdin, uint64_t max_cycles,
                      bfgpu_record** out); /* *out is set even on failure: bfgpu_record_error(), then bfgpu_record_free() */
const char* bfgpu_record_error(const bfgpu_record* rec);
/* counts: cycles, instructions, alu / jump / memory-instruction / io events, touched cells, output bytes */
int32_t bfgpu_record_info(const bfgpu_record* rec, uint64_t counts[8]);
int32_t bfgpu_record_output(const bfgpu_record* rec, uint8_t* out);
/* raw views (tests): (cycles+1) x {pc, mp, prev_ts, mv | prev_value << 8}; cells x {addr, initial ts, initial value,
 * final ts, final value}; program opcodes / jump targets */
const uint32_t* bfgpu_record_cycles(const bfgpu_record* rec);
const uint32_t* bfgpu_record_mem_events(const bfgpu_record* rec);
int32_t bfgpu_record_program(const bfgpu_record* rec, uint32_t* ops, uint32_t* args);
void bfgpu_record_free(bfgpu_record* rec);
/* StarkMachine::setup for the record's program (preprocessed Program + Byte traces) */
int32_t bfgpu_machine_setup_record(bfgpu_ctx* ctx, const bfgpu_record* rec, uint32_t commit[8], bfgpu_pk** out);
/* generate every included chip's main trace on the device and commit (MachineProver::commit, prover.rs:209-236) */
int32_t bfgpu_machine_commit_record(bfgpu_ctx* ctx, const bfgpu_record* rec, uint32_t root[8], bfgpu_shard** out);
/* traces held by a shard, in commit order; get_trace copies one out row-major, natural row order, caller representation */
int32_t bfgpu_shard_num_traces(const bfgpu_shard* shard);
int32_t bfgpu_shard_trace_info(const bfgpu_shard* shard, int32_t i, const char** name, uint64_t* rows, uint64_t* cols);
int32_t bfgpu_shard_get_trace(const bfgpu_shard* shard, int32_t i, uint32_t* out);

/* ---- ONE shard proof over several GPUs (SURVEY.md §8e; one process / context per GPU) ---------------------------------------- */
/* `MachineProver::prove` (crates/stark/src/prover.rs:560-582: commit + open, :209-553) by `world` ranks.  The three commitments go
 * through the sharded commitment above; the LogUp traces are replicated; the quotient is evaluated on each rank's LDE rows (the
 * "next" row read from the peer that holds it, the result stored straight into the rank that owns that quotient column); opened
 * values, reduced openings and FRI folds are row-local with one small exchange per step; queries are answered by the owner of the
 * leaf (csrc/dist_prove.cuh).  The proof is word for word the one bfgpu_machine_open produces on one GPU, returned on EVERY rank.
 * The caller supplies the control plane: an all-gather of equal-sized byte strings between host buffers (recv = world * bytes, rank
 * order) and a barrier — ~30 small all-gathers and ~8 barriers per proof (torch.distributed in the Python mirror, MPI / NCCL in a
 * Rust shim).  Callbacks return 0 on success.  Every rank passes the same proving key, the same record (or the same full set of
 * main traces) and a challenger in the same state (pk observed). */
typedef struct {
    void* user;
    int32_t (*all_gather)(void* user, const void* send, void* recv, uint64_t bytes_per_rank);
    int32_t (*barrier)(void* user);
} bfgpu_comm;
/* A ready-made control plane for one process per GPU on ONE node: bfgpu_comm served from a POSIX shared-memory segment (two atomics
 * and a slot per rank: ~2-5 us per call instead of 150-300 us through a Python / TCP collective).  Every rank calls with the same
 * job-unique name (e.g. "/bfgpu-<port>-<pid of rank 0>"); returns once all ranks are attached (the name is unlinked then). */
int32_t bfgpu_comm_shm_create(const char* name, uint32_t rank, uint32_t world, uint64_t slot_bytes, bfgpu_comm** out);
void bfgpu_comm_shm_destroy(bfgpu_comm* comm);
int32_t bfgpu_dist_prove_record(bfgpu_ctx* ctx, const bfgpu_comm* comm, uint32_t rank, uint32_t world, const bfgpu_pk* pk, const bfgpu_record* rec,
                                bfgpu_challenger* ch, int64_t fixed_pow_witness, bfgpu_shard_proof** out);
int32_t bfgpu_dist_prove(bfgpu_ctx* ctx, const bfgpu_comm* comm, uint32_t rank, uint32_t world, const bfgpu_pk* pk, const char* const* names,
                         const bfgpu_mat* traces, int32_t n, bfgpu_challenger* ch, int64_t fixed_pow_witness, bfgpu_shard_proof** out);

/* ---- native verifier (SURVEY.md §8f item 2) ---------------------------------------------------------------- */
/* `Verifier::verify_shard` (crates/stark/src/verifier.rs:27-216) on the serialisation of bfgpu_machine_open: replays the
 * transcript, verifies the PCS opening (input Merkle openings, reduced openings, FRI fold chain, proof of work), checks
 * C(zeta) = q(zeta) Z_H(zeta) for every chip with the constraint programs over F_p^4, and that the LogUp cumulative sums
 * cancel.  Host code only: no context, no device.  vk = preprocessed commitment + (chip name, log2 height) of the
 * preprocessed traces in proving-key order.  Returns BFGPU_OK (accepted) or BFGPU_ERR_INVALID with the reference's
 * error name (OodEvaluationMismatch:<chip>, InvalidOpeningArgument:..., CumulativeSumsError, ...) in err. */
int32_t bfgpu_verify_shard(const uint32_t vk_commit[8], const char* const* prep_names, const uint32_t* prep_log_heights, int32_t n_prep,
                           const uint32_t* proof, uint64_t n_words, int repr, uint32_t log_blowup, uint32_t num_queries,
                           uint32_t pow_bits, char* err, uint64_t err_len);
/* same with explicit transcript options: options[BFGPU_OPT_*] for the first n_options options (NULL / 0 = all defaults) */
int32_t bfgpu_verify_shard_ex(const uint32_t vk_commit[8], const char* const* prep_names, const uint32_t* prep_log_heights, int32_t n_prep,
                              const uint32_t* proof, uint64_t n_words, int repr, uint32_t log_blowup, uint32_t num_queries,
                              uint32_t pow_bits, const uint32_t* options, int32_t n_options, char* err, uint64_t err_len);

/* `BfProver::verify` (crates/prover/src/verify.rs:10-36) on top of `StarkMachine::verify` (crates/stark/src/machine.rs:258-284): rejects
 * a proof without the Cpu chip (MissingCpuInFirstShard) or with a Cpu log degree above MAX_CPU_LOG_DEGREE = 22
 * (crates/core/machine/src/cpu/mod.rs:8; CpuLogDegreeTooLarge: <n>), then runs bfgpu_verify_shard_ex and reports its errors as
 * "InvalidShardProof: <error>" (MachineVerificationError, machine.rs:391-416).  Host code only. */
int32_t bfgpu_verify_core_proof(const uint32_t vk_commit[8], const char* const* prep_names, const uint32_t* prep_log_heights, int32_t n_prep,
                                const uint32_t* proof, uint64_t n_words, int repr, uint32_t log_blowup, uint32_t num_queries,
                                uint32_t pow_bits, const uint32_t* options, int32_t n_options, char* err, uint64_t err_len);

/* ---- batch verifier on the device ---------------------------------------------------------------------------- */
/* One proof of a batch: its verifying key (as for bfgpu_verify_shard) and its serialised words. */
typedef struct {
    const uint32_t* vk_commit;
    const char* const* prep_names;
    const uint32_t* prep_log_heights;
    int32_t n_prep;
    const uint32_t* proof;
    uint64_t n_words;
} bfgpu_verify_item;
/* `BfProver::verify` (crates/prover/src/verify.rs:10-36) when core is 1, else `Verifier::verify_shard` (crates/stark/src/verifier.rs:27-329),
 * for n_items proofs in one call.  The host parses and shape-checks each proof, replays its transcript, checks the proof of work and
 * evaluates the constraints at zeta; the Merkle openings of every query (input and commit-phase rounds), the reduced openings and the
 * fold chain of every proof run on the device in one pass.  status[i] and the string at errs + i * err_len (truncated to err_len bytes,
 * errs may be NULL when err_len is 0) are exactly what bfgpu_verify_core_proof (core = 1) or bfgpu_verify_shard_ex (core = 0) return for
 * item i under the same repr, FRI parameters and options.  The return value reports only bad arguments or device failures
 * (bfgpu_last_error); n_items = 0 does nothing.  Runs on the context's stream and synchronises it. */
int32_t bfgpu_verify_batch(bfgpu_ctx* ctx, const bfgpu_verify_item* items, int32_t n_items, int repr, uint32_t log_blowup, uint32_t num_queries,
                           uint32_t pow_bits, const uint32_t* options, int32_t n_options, int32_t core, int32_t* status, char* errs,
                           uint64_t err_len);

/* Canonical proof serialiser (SURVEY.md §8f item 2): the bytes `bincode::serialize(&MachineProof { shard_proof })` writes for this proof
 * (crates/stark/src/types.rs:32-73,116-119; bincode 1.x defaults) — what the reference's `proofSize` counts
 * (crates/core/machine/src/utils/prove.rs:47-56) and what a Rust caller can `bincode::deserialize` into a `MachineProof`.  Host code
 * only.  field_repr: 1 = field elements as Montgomery words (p3-monty-31's serde form, P3), 0 = canonical residues.  `chip_ordering`
 * is written in chip order (the reference iterates a randomly seeded hashbrown map: its byte ORDER differs per process, the byte COUNT
 * does not).  out == NULL returns only *out_len. */
int32_t bfgpu_shard_proof_to_bincode(const char* const* prep_names, const uint32_t* prep_log_heights, int32_t n_prep, const uint32_t* proof,
                                     uint64_t n_words, int repr, uint32_t log_blowup, int field_repr, uint8_t* out, uint64_t out_cap,
                                     uint64_t* out_len, char* err, uint64_t err_len);

#ifdef __cplusplus
}
#endif
#endif /* BFGPU_H */
