"""zkvm-brainfuck_b200 — host-side mirror of the reference's proving interfaces over the CUDA C ABI.

The reference (felicityin/zkvm-brainfuck) is Rust and no Rust toolchain exists in this image, so
the production binding is the `extern "C"` surface in include/bfgpu.h (INTEGRATION.md shows the
Rust FFI crate).  This package is the Python/ctypes harness over the SAME symbols, with the same
names and argument meaning as the Plonky3 traits the reference is generic over:

  Radix2Dit       ~ TwoAdicSubgroupDft<KoalaBear>   (kb31_poseidon2.rs:30)
  MerkleTreeMmcs  ~ Mmcs<KoalaBear>                 (kb31_poseidon2.rs:27-28)
  TwoAdicFriPcs   ~ Pcs<Challenge, Challenger>      (kb31_poseidon2.rs:32, prover.rs:227,...)

There is no CPU fallback: importing works anywhere (so the ABI can be checked), but every compute
call raises `BfGpuError` without a CUDA device and the library refuses to load if it was not built.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

P = 2130706433
REPR_CANONICAL, REPR_MONTY = 0, 1
MEM_HOST, MEM_DEVICE = 0, 1

_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)


class BfGpuError(RuntimeError):
    pass


class Mat(C.Structure):
    _fields_ = [("data", C.c_void_p), ("rows", C.c_uint64), ("cols", C.c_uint64)]


_LIB = None
SO_PATH = _build.SO

# every symbol include/bfgpu.h declares: (restype, argtypes)
ABI = {
    "bfgpu_ctx_create": (C.c_int32, [C.c_int, C.POINTER(C.c_void_p)]),
    "bfgpu_ctx_destroy": (None, [C.c_void_p]),
    "bfgpu_last_error": (C.c_char_p, [C.c_void_p]),
    "bfgpu_set_repr": (C.c_int32, [C.c_void_p, C.c_int]),
    "bfgpu_set_input_space": (C.c_int32, [C.c_void_p, C.c_int]),
    "bfgpu_set_stream": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "bfgpu_synchronize": (C.c_int32, [C.c_void_p]),
    "bfgpu_set_fri_params": (C.c_int32, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    "bfgpu_set_transcript_option": (C.c_int32, [C.c_void_p, C.c_int32, C.c_uint32]),
    "bfgpu_launch_count": (C.c_uint64, [C.c_void_p]),
    "bfgpu_debug_live_blocks": (C.c_uint64, [C.c_void_p]),
    "bfgpu_debug_fail_alloc": (C.c_int32, [C.c_void_p, C.c_int64]),
    "bfgpu_host_alloc": (C.c_int32, [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "bfgpu_host_free": (None, [C.c_void_p]),
    "bfgpu_profile_enable": (C.c_int32, [C.c_void_p, C.c_int]),
    "bfgpu_profile_read": (C.c_int32, [C.c_void_p, C.POINTER(C.c_float), _u64p]),
    "bfgpu_int32_peak_probe": (C.c_int32, [C.c_void_p, C.POINTER(C.c_double)]),
    "bfgpu_poseidon2_permute": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "bfgpu_sponge_hash_rows": (C.c_int32, [C.c_void_p, C.POINTER(Mat), C.c_void_p]),
    "bfgpu_compress": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "bfgpu_coset_lde_batch": (C.c_int32, [C.c_void_p, C.POINTER(Mat), C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]),
    "bfgpu_dft_batch": (C.c_int32, [C.c_void_p, C.POINTER(Mat), C.c_void_p]),
    "bfgpu_idft_batch": (C.c_int32, [C.c_void_p, C.POINTER(Mat), C.c_void_p]),
    "bfgpu_mmcs_commit": (C.c_int32, [C.c_void_p, C.POINTER(Mat), C.c_int32, _u32p, C.POINTER(C.c_void_p)]),
    "bfgpu_mmcs_open_batch": (C.c_int32, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "bfgpu_tree_num_layers": (C.c_int32, [C.c_void_p]),
    "bfgpu_tree_layer_len": (C.c_uint64, [C.c_void_p, C.c_int32]),
    "bfgpu_tree_get_layer": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p]),
    "bfgpu_tree_free": (None, [C.c_void_p]),
    "bfgpu_pcs_commit": (C.c_int32, [C.c_void_p, C.POINTER(Mat), _u32p, C.c_int32, _u32p, C.POINTER(C.c_void_p)]),
    "bfgpu_pcs_num_matrices": (C.c_int32, [C.c_void_p]),
    "bfgpu_pcs_lde_dims": (C.c_int32, [C.c_void_p, C.c_int32, _u64p, _u64p]),
    "bfgpu_pcs_get_evaluations": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int, C.c_void_p]),
    "bfgpu_pcs_tree": (C.c_void_p, [C.c_void_p]),
    "bfgpu_pcs_data_free": (None, [C.c_void_p]),
    "bfgpu_pcs_lde_device": (C.c_int32, [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p), _u64p, _u64p, _u64p]),
    "bfgpu_logup_perm_trace": (C.c_int32, [C.c_void_p, C.c_char_p, C.POINTER(Mat), C.POINTER(Mat), _u32p, C.c_void_p, _u32p]),
    "bfgpu_quotient_values": (C.c_int32, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, _u32p, _u32p, _u32p,
                                           C.c_void_p]),
    "bfgpu_execute": (C.c_int32, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(C.c_void_p)]),
    "bfgpu_record_error": (C.c_char_p, [C.c_void_p]),
    "bfgpu_record_info": (C.c_int32, [C.c_void_p, _u64p]),
    "bfgpu_record_output": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "bfgpu_record_cycles": (C.c_void_p, [C.c_void_p]),
    "bfgpu_record_mem_events": (C.c_void_p, [C.c_void_p]),
    "bfgpu_record_program": (C.c_int32, [C.c_void_p, _u32p, _u32p]),
    "bfgpu_record_free": (None, [C.c_void_p]),
    "bfgpu_machine_setup_record": (C.c_int32, [C.c_void_p, C.c_void_p, _u32p, C.POINTER(C.c_void_p)]),
    "bfgpu_machine_commit_record": (C.c_int32, [C.c_void_p, C.c_void_p, _u32p, C.POINTER(C.c_void_p)]),
    "bfgpu_shard_num_traces": (C.c_int32, [C.c_void_p]),
    "bfgpu_shard_trace_info": (C.c_int32, [C.c_void_p, C.c_int32, C.POINTER(C.c_char_p), _u64p, _u64p]),
    "bfgpu_shard_get_trace": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p]),
    "bfgpu_verify_shard": (C.c_int32, [_u32p, C.POINTER(C.c_char_p), _u32p, C.c_int32, _u32p, C.c_uint64, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32,
                           C.c_char_p, C.c_uint64]),
    "bfgpu_verify_shard_ex": (C.c_int32, [_u32p, C.POINTER(C.c_char_p), _u32p, C.c_int32, _u32p, C.c_uint64, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32,
                              _u32p, C.c_int32, C.c_char_p, C.c_uint64]),
    "bfgpu_verify_core_proof": (C.c_int32, [_u32p, C.POINTER(C.c_char_p), _u32p, C.c_int32, _u32p, C.c_uint64, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32,
                                _u32p, C.c_int32, C.c_char_p, C.c_uint64]),
    "bfgpu_verify_batch": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, _u32p, C.c_int32, C.c_int32,
                                       C.POINTER(C.c_int32), C.c_char_p, C.c_uint64]),
    "bfgpu_shard_proof_to_bincode": (C.c_int32, [C.POINTER(C.c_char_p), _u32p, C.c_int32, _u32p, C.c_uint64, C.c_int, C.c_uint32, C.c_int, C.c_void_p,
                                                  C.c_uint64, _u64p, C.c_char_p, C.c_uint64]),
    "bfgpu_dist_commit_begin": (C.c_int32, [C.c_void_p, C.c_uint32, C.c_uint32, _u64p, _u32p, C.c_int32, C.POINTER(C.c_void_p)]),
    "bfgpu_dist_commit_local_cols": (C.c_uint32, [C.c_void_p, C.c_int32, _u32p]),
    "bfgpu_dist_commit_recv_handle": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "bfgpu_dist_commit_set_peers": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "bfgpu_dist_commit_block_words": (C.c_uint64, [C.c_void_p, C.c_uint32]),
    "bfgpu_dist_commit_set_staging": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "bfgpu_dist_commit_lde": (C.c_int32, [C.c_void_p, C.POINTER(Mat), _u32p]),
    "bfgpu_dist_commit_unpack": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "bfgpu_dist_commit_finish": (C.c_int32, [C.c_void_p, _u32p]),
    "bfgpu_dist_commit_root": (C.c_int32, [C.c_void_p, _u32p, _u32p]),
    "bfgpu_dist_commit_open_batch": (C.c_int32, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "bfgpu_dist_commit_rows_per_rank": (C.c_uint64, [C.c_void_p]),
    "bfgpu_dist_commit_free": (None, [C.c_void_p]),
    "bfgpu_comm_shm_create": (C.c_int32, [C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_void_p)]),
    "bfgpu_comm_shm_destroy": (None, [C.c_void_p]),
    "bfgpu_dist_prove_record": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]),
    "bfgpu_dist_prove": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_char_p), C.POINTER(Mat), C.c_int32, C.c_void_p,
                                     C.c_int64, C.POINTER(C.c_void_p)]),
    "bfgpu_challenger_create": (C.c_int32, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "bfgpu_challenger_clone": (C.c_int32, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "bfgpu_challenger_free": (None, [C.c_void_p]),
    "bfgpu_challenger_observe": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "bfgpu_challenger_sample": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "bfgpu_challenger_sample_bits": (C.c_int32, [C.c_void_p, C.c_uint32, _u32p]),
    "bfgpu_challenger_export": (C.c_int32, [C.c_void_p, _u32p, _u32p, _u32p, _u32p, _u32p]),
    "bfgpu_challenger_import": (C.c_int32, [C.c_void_p, _u32p, _u32p, C.c_uint32, _u32p, C.c_uint32]),
    "bfgpu_pcs_open": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]),
    "bfgpu_opening_size": (C.c_uint64, [C.c_void_p]),
    "bfgpu_opening_read": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "bfgpu_opening_free": (None, [C.c_void_p]),
    "bfgpu_machine_num_chips": (C.c_int32, []),
    "bfgpu_machine_chip_info": (C.c_int32, [C.c_int32, C.POINTER(C.c_char_p), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                            C.POINTER(C.c_int32)]),
    "bfgpu_machine_setup": (C.c_int32, [C.c_void_p, C.POINTER(C.c_char_p), C.POINTER(Mat), C.c_int32, _u32p, C.POINTER(C.c_void_p)]),
    "bfgpu_pk_observe_into": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "bfgpu_pk_free": (None, [C.c_void_p]),
    "bfgpu_machine_commit": (C.c_int32, [C.c_void_p, C.POINTER(C.c_char_p), C.POINTER(Mat), C.c_int32, _u32p, C.POINTER(C.c_void_p)]),
    "bfgpu_shard_free": (None, [C.c_void_p]),
    "bfgpu_machine_open": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]),
    "bfgpu_shard_proof_size": (C.c_uint64, [C.c_void_p]),
    "bfgpu_shard_proof_read": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "bfgpu_shard_proof_free": (None, [C.c_void_p]),
    "bfgpu_machine_debug": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]),
    "bfgpu_debug_report_size": (C.c_uint64, [C.c_void_p]),
    "bfgpu_debug_report_read": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "bfgpu_debug_report_free": (None, [C.c_void_p]),
}


class VerifyItem(C.Structure):
    _fields_ = [("vk_commit", _u32p), ("prep_names", C.POINTER(C.c_char_p)), ("prep_log_heights", _u32p), ("n_prep", C.c_int32), ("proof", _u32p),
                ("n_words", C.c_uint64)]


class OpenRound(C.Structure):
    _fields_ = [("data", C.c_void_p), ("num_points", _u32p), ("points", _u32p)]


def lib():
    """Load libbfgpu.so (built in-tree by build.py / __graft_entry__.build()); never falls back."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise BfGpuError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                             "(this backend has no CPU fallback)")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in ABI.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class Context:
    """`KoalaBearPoseidon2::new()` analogue (kb31_poseidon2.rs:73-85): owns the device context."""

    def __init__(self, device=0, repr=REPR_CANONICAL):
        self._h = C.c_void_p()
        rc = lib().bfgpu_ctx_create(device, C.byref(self._h))
        if rc != 0:
            msg = lib().bfgpu_last_error(self._h).decode() if self._h else "context allocation failed"
            if self._h:
                lib().bfgpu_ctx_destroy(self._h)
                self._h = None
            raise BfGpuError(f"bfgpu_ctx_create failed ({rc}): {msg}")
        self.check(lib().bfgpu_set_repr(self._h, repr))

    def check(self, rc):
        if rc != 0:
            raise BfGpuError(f"bfgpu error {rc}: {lib().bfgpu_last_error(self._h).decode()}")

    def set_stream(self, cuda_stream_handle):
        self.check(lib().bfgpu_set_stream(self._h, C.c_void_p(cuda_stream_handle)))

    def set_input_space(self, space):
        self.check(lib().bfgpu_set_input_space(self._h, space))

    def set_repr(self, repr):
        self.check(lib().bfgpu_set_repr(self._h, repr))

    OPTIONS = {"observe_opened_values": 0, "fri_rollin": 1, "pow_order": 2}

    def set_transcript_option(self, name, value):
        """bfgpu_set_transcript_option: the Plonky3-internal choices that cannot be confirmed offline (include/bfgpu.h)."""
        self.check(lib().bfgpu_set_transcript_option(self._h, self.OPTIONS[name], int(value)))

    def set_fri_params(self, log_blowup=1, num_queries=84, pow_bits=16):
        self.check(lib().bfgpu_set_fri_params(self._h, log_blowup, num_queries, pow_bits))

    def synchronize(self):
        self.check(lib().bfgpu_synchronize(self._h))

    def pinned_copy(self, arr):
        """Copy of `arr` in page-locked host memory (uint32), for full-speed host->device transfers."""
        a = _u32(arr)
        p = C.c_void_p()
        self.check(lib().bfgpu_host_alloc(self._h, a.nbytes, C.byref(p)))
        buf = (C.c_uint32 * max(a.size, 1)).from_address(p.value)
        out = np.frombuffer(buf, dtype=np.uint32, count=a.size).reshape(a.shape)
        out[...] = a
        self._pinned = getattr(self, "_pinned", [])
        self._pinned.append(p.value)
        return out

    def free_pinned(self):
        for p in getattr(self, "_pinned", []):
            lib().bfgpu_host_free(C.c_void_p(p))
        self._pinned = []

    PHASES = ["h2d", "ingest", "intt", "scale", "ntt", "leaf_hash", "compress", "other", "open_eval", "open_reduce", "fri",
              "pow", "query", "perm", "quotient", "exchange", "tracegen", "debug_rows", "debug_lookups", "verify"]

    def profile_enable(self, on=True):
        self.check(lib().bfgpu_profile_enable(self._h, 1 if on else 0))

    def profile_read(self):
        """-> {phase: (milliseconds, launches)} accumulated since profile_enable(True)."""
        ms = (C.c_float * 20)()
        ln = (C.c_uint64 * 20)()
        self.check(lib().bfgpu_profile_read(self._h, ms, ln))
        return {n: (float(ms[i]), int(ln[i])) for i, n in enumerate(self.PHASES)}

    def int32_peak_probe(self):
        g = C.c_double()
        self.check(lib().bfgpu_int32_peak_probe(self._h, C.byref(g)))
        return g.value

    @property
    def launch_count(self):
        return int(lib().bfgpu_launch_count(self._h))

    @property
    def live_blocks(self):
        """device blocks currently handed out by the context's allocator (error-path tests)"""
        return int(lib().bfgpu_debug_live_blocks(self._h))

    def fail_alloc(self, nth):
        """test hook: the nth device allocation from now fails with BFGPU_ERR_OOM (nth < 0 disarms)"""
        self.check(lib().bfgpu_debug_fail_alloc(self._h, int(nth)))

    def close(self):
        if getattr(self, "_h", None):
            lib().bfgpu_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # interpreter shutdown: module globals may already be gone
            pass

    # ---- Poseidon2 primitives -----------------------------------------------------------------
    def permute(self, states):
        s = _u32(states).copy()
        assert s.ndim == 2 and s.shape[1] == 16
        self.check(lib().bfgpu_poseidon2_permute(self._h, _ptr(s), s.shape[0]))
        return s

    def hash_rows(self, mat):
        m = _u32(mat)
        out = np.zeros((m.shape[0], 8), np.uint32)
        cm = Mat(m.ctypes.data, m.shape[0], m.shape[1])
        self.check(lib().bfgpu_sponge_hash_rows(self._h, C.byref(cm), _ptr(out)))
        return out

    def compress(self, left, right):
        l, r = _u32(left), _u32(right)
        out = np.zeros_like(l)
        self.check(lib().bfgpu_compress(self._h, _ptr(l), _ptr(r), l.shape[0], _ptr(out)))
        return out


def _mats(mats):
    keep = [_u32(m) for m in mats]
    arr = (Mat * len(keep))()
    for i, m in enumerate(keep):
        if m.ndim != 2:
            raise ValueError("matrices must be 2-D")
        arr[i] = Mat(m.ctypes.data, m.shape[0], m.shape[1])
    return arr, keep


class Radix2Dit:
    """TwoAdicSubgroupDft<KoalaBear> (the reference's `Dft`, kb31_poseidon2.rs:30)."""

    def __init__(self, ctx):
        self.ctx = ctx

    def _call(self, fn, mat, out_rows, *extra):
        m = _u32(mat)
        out = np.zeros((out_rows, m.shape[1]), np.uint32)
        cm = Mat(m.ctypes.data, m.shape[0], m.shape[1])
        self.ctx.check(fn(self.ctx._h, C.byref(cm), *extra, _ptr(out)))
        return out

    def dft_batch(self, mat):
        return self._call(lib().bfgpu_dft_batch, mat, np.shape(mat)[0])

    def idft_batch(self, mat):
        return self._call(lib().bfgpu_idft_batch, mat, np.shape(mat)[0])

    def coset_lde_batch(self, mat, added_bits, shift, bit_reversed_rows=False):
        return self._call(lib().bfgpu_coset_lde_batch, mat, np.shape(mat)[0] << added_bits, added_bits, int(shift),
                          1 if bit_reversed_rows else 0)


class MerkleTree:
    """Mmcs::ProverData."""

    def __init__(self, ctx, handle, dims, owned=True):
        self.ctx, self._h, self.dims, self._owned = ctx, handle, dims, owned
        self.root = None

    def layers(self):
        out = []
        for l in range(lib().bfgpu_tree_num_layers(self._h)):
            n = lib().bfgpu_tree_layer_len(self._h, l)
            a = np.zeros((n, 8), np.uint32)
            self.ctx.check(lib().bfgpu_tree_get_layer(self._h, l, _ptr(a)))
            out.append(a)
        return out

    def free(self):
        if self._owned and self._h:
            lib().bfgpu_tree_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:  # interpreter shutdown: module globals may already be gone
            pass


class MerkleTreeMmcs:
    """Mmcs<KoalaBear> = MerkleTreeMmcs<_, _, MyHash, MyCompress, 8> (kb31_poseidon2.rs:27-28)."""

    def __init__(self, ctx):
        self.ctx = ctx

    def commit(self, mats):
        arr, keep = _mats(mats)
        root = np.zeros(8, np.uint32)
        h = C.c_void_p()
        self.ctx.check(lib().bfgpu_mmcs_commit(self.ctx._h, arr, len(keep), root.ctypes.data_as(_u32p), C.byref(h)))
        t = MerkleTree(self.ctx, h, [m.shape for m in keep])
        t.root = root
        return root, t

    def open_batch(self, index, tree):
        total = sum(c for _, c in tree.dims)
        nl = lib().bfgpu_tree_num_layers(tree._h) - 1
        rows = np.zeros(max(total, 1), np.uint32)
        sib = np.zeros((max(nl, 1), 8), np.uint32)
        self.ctx.check(lib().bfgpu_mmcs_open_batch(tree._h, int(index), _ptr(rows), _ptr(sib)))
        out, o = [], 0
        for _, c in tree.dims:
            out.append(rows[o:o + c].copy())
            o += c
        return out, sib[:nl].copy()


class PcsProverData:
    def __init__(self, ctx, handle):
        self.ctx, self._h = ctx, handle
        n = lib().bfgpu_pcs_num_matrices(handle)
        self.dims = []
        for i in range(n):
            r, c = C.c_uint64(), C.c_uint64()
            lib().bfgpu_pcs_lde_dims(handle, i, C.byref(r), C.byref(c))
            self.dims.append((r.value, c.value))
        self.tree = MerkleTree(ctx, lib().bfgpu_pcs_tree(handle), self.dims, owned=False)

    def free(self):
        if self._h:
            lib().bfgpu_pcs_data_free(self._h)
            self._h = None
            self.tree._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:  # interpreter shutdown: module globals may already be gone
            pass


class Challenger:
    """DuplexChallenger<Val, Perm, 16, 8> (kb31_poseidon2.rs:31); host-side sponge inside the library."""

    def __init__(self, ctx, _handle=None):
        self.ctx = ctx
        if _handle is None:
            _handle = C.c_void_p()
            ctx.check(lib().bfgpu_challenger_create(ctx._h, C.byref(_handle)))
        self._h = _handle

    def clone(self):
        h = C.c_void_p()
        self.ctx.check(lib().bfgpu_challenger_clone(self._h, C.byref(h)))
        return Challenger(self.ctx, h)

    def observe(self, v):
        self.observe_slice([v])

    def observe_slice(self, vs):
        a = _u32(np.asarray(vs).ravel())
        self.ctx.check(lib().bfgpu_challenger_observe(self._h, _ptr(a), a.size))

    observe_digest = observe_slice
    observe_ext = observe_slice

    def sample(self):
        out = np.zeros(1, np.uint32)
        self.ctx.check(lib().bfgpu_challenger_sample(self._h, _ptr(out), 1))
        return int(out[0])

    def sample_ext(self):
        out = np.zeros(4, np.uint32)
        self.ctx.check(lib().bfgpu_challenger_sample(self._h, _ptr(out), 4))
        return out.astype(np.uint64)

    def sample_bits(self, bits):
        out = C.c_uint32()
        self.ctx.check(lib().bfgpu_challenger_sample_bits(self._h, bits, C.byref(out)))
        return out.value

    def export(self):
        st, ib, ob = np.zeros(16, np.uint32), np.zeros(8, np.uint32), np.zeros(8, np.uint32)
        ni, no = C.c_uint32(), C.c_uint32()
        self.ctx.check(lib().bfgpu_challenger_export(self._h, st.ctypes.data_as(_u32p), ib.ctypes.data_as(_u32p), C.byref(ni),
                                                     ob.ctypes.data_as(_u32p), C.byref(no)))
        return st, ib[:ni.value].copy(), ob[:no.value].copy()

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                lib().bfgpu_challenger_free(self._h)
                self._h = None
        except Exception:  # interpreter shutdown: module globals may already be gone
            pass


class TwoAdicFriPcs:
    """Pcs (kb31_poseidon2.rs:32): commit / get_evaluations_on_domain / open."""

    def open(self, rounds, challenger, pow_witness=None):
        """`pcs.open(vec![(&data, points), ...], &mut challenger)` (prover.rs:460-470).
        rounds: [(PcsProverData, [[ext point, ...] per matrix])].  Returns (opened_values, fri_proof) in the
        nested as opened[round][matrix][point] -> (width, 4) and a FriProof-shaped dict."""
        n = len(rounds)
        arr = (OpenRound * n)()
        keep = []
        for i, (data, points) in enumerate(rounds):
            assert len(points) == len(data.dims)
            npts = _u32([len(p) for p in points])
            flat = _u32(np.concatenate([np.asarray(z, np.uint64).ravel() for p in points for z in p]) if any(len(p) for p in points) else np.zeros(0))
            keep += [npts, flat]
            arr[i] = OpenRound(data._h, npts.ctypes.data_as(_u32p), flat.ctypes.data_as(_u32p))
        h = C.c_void_p()
        self.ctx.check(lib().bfgpu_pcs_open(self.ctx._h, arr, n, challenger._h, -1 if pow_witness is None else int(pow_witness), C.byref(h)))
        size = lib().bfgpu_opening_size(h)
        buf = np.zeros(size, np.uint32)
        self.ctx.check(lib().bfgpu_opening_read(h, _ptr(buf)))
        lib().bfgpu_opening_free(h)
        return self._parse_opening(buf, rounds)

    @staticmethod
    def _parse_opening(buf, rounds):
        pos = 0

        def take(k):
            nonlocal pos
            v = buf[pos:pos + k]
            pos += k
            return v

        opened = []
        for data, points in rounds:
            rv = []
            for (rows, cols), pts in zip(data.dims, points):
                rv.append([take(cols * 4).astype(np.uint64).reshape(cols, 4) for _ in pts])
            opened.append(rv)
        ncommit = int(take(1)[0])
        commits = [take(8).copy() for _ in range(ncommit)]
        final_poly = take(4).astype(np.uint64)
        pow_witness = int(take(1)[0])
        nq = int(take(1)[0])
        # FRI folds the tallest LDE down to 2^log_blowup entries, so the commit-phase layers follow from the heights alone
        log_max_height = max(r for data, _ in rounds for r, _ in data.dims).bit_length() - 1
        queries = []
        for _ in range(nq):
            index = int(take(1)[0])
            input_proof = []
            for data, _pts in rounds:
                log_max_h = max(r for r, _ in data.dims).bit_length() - 1
                rows = [take(c).copy() for _, c in data.dims]
                sib = take(8 * log_max_h).reshape(log_max_h, 8).copy()
                input_proof.append(dict(opened_values=rows, opening_proof=sib))
            steps = []
            for i in range(ncommit):
                sv = take(4).astype(np.uint64)
                nl = log_max_height - 1 - i
                steps.append(dict(sibling_value=sv, opening_proof=take(8 * nl).reshape(nl, 8).copy()))
            queries.append(dict(index=index, input_proof=input_proof, commit_phase_openings=steps))
        assert pos == len(buf), (pos, len(buf))
        return opened, dict(commit_phase_commits=commits, query_proofs=queries, final_poly=final_poly, pow_witness=pow_witness)

    def __init__(self, ctx):
        self.ctx = ctx

    def commit(self, evaluations, domain_shifts=None):
        """`pcs.commit(vec![(domain, matrix), ...])`; domain_shifts[i] = domain.shift (default 1)."""
        arr, keep = _mats(evaluations)
        root = np.zeros(8, np.uint32)
        h = C.c_void_p()
        sh = None
        if domain_shifts is not None:
            sh = _u32(domain_shifts)
            assert sh.shape == (len(keep),)
        self.ctx.check(lib().bfgpu_pcs_commit(self.ctx._h, arr, sh.ctypes.data_as(_u32p) if sh is not None else None, len(keep),
                                              root.ctypes.data_as(_u32p), C.byref(h)))
        return root, PcsProverData(self.ctx, h)

    def get_evaluations_on_domain(self, data, idx, bit_reversed_rows=False):
        r, c = data.dims[idx]
        out = np.zeros((r, c), np.uint32)
        self.ctx.check(lib().bfgpu_pcs_get_evaluations(data._h, idx, 1 if bit_reversed_rows else 0, _ptr(out)))
        return out


def generate_permutation_trace(ctx, chip, main, prep, alpha, beta):
    """`Chip::generate_permutation_trace` (chip.rs:117-136): -> (LogUp trace (rows, 4 * perm_width) uint32, cumulative sum (4,))."""
    info = {c[0]: c for c in machine_chips()}.get(chip, (chip, 0, 0, 1, False))  # unknown names are reported by the library
    m = _u32(main)
    cm = Mat(m.ctypes.data, m.shape[0], m.shape[1])
    pm = None
    if prep is not None and np.size(prep):
        pa = _u32(prep)
        pm = Mat(pa.ctypes.data, pa.shape[0], pa.shape[1])
    ch = _u32(np.concatenate([np.asarray(alpha, np.uint64), np.asarray(beta, np.uint64)]))
    out = np.zeros((m.shape[0], 4 * info[3]), np.uint32)
    cs = np.zeros(4, np.uint32)
    ctx.check(lib().bfgpu_logup_perm_trace(ctx._h, chip.encode(), C.byref(cm), C.byref(pm) if pm is not None else None, ch.ctypes.data_as(_u32p),
                                           _ptr(out), cs.ctypes.data_as(_u32p)))
    return out, cs


def quotient_values(ctx, chip, prep_data, prep_idx, main_data, main_idx, perm_data, perm_idx, alpha, perm_challenges, cum_sum):
    """`quotient_values` (quotient.rs:18-165) from committed `PcsProverData` handles -> (2 * rows, 4) uint32, natural order."""
    rows = main_data.dims[main_idx][0]
    out = np.zeros((rows, 4), np.uint32)
    a = _u32(np.asarray(alpha, np.uint64))
    pc = _u32(np.concatenate([np.asarray(x, np.uint64) for x in perm_challenges]))
    cs = _u32(np.asarray(cum_sum, np.uint64))
    ctx.check(lib().bfgpu_quotient_values(ctx._h, chip.encode(), prep_data._h if prep_data is not None else None, prep_idx, main_data._h, main_idx,
                                          perm_data._h, perm_idx, a.ctypes.data_as(_u32p), pc.ctypes.data_as(_u32p), cs.ctypes.data_as(_u32p), _ptr(out)))
    return out


def machine_chips():
    """[(name, main_width, prep_width, perm_ext_width, local_only)] in BfAir::chips() order."""
    out = []
    for i in range(lib().bfgpu_machine_num_chips()):
        name = C.c_char_p()
        mw, pw, ew, lo = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        lib().bfgpu_machine_chip_info(i, C.byref(name), C.byref(mw), C.byref(pw), C.byref(ew), C.byref(lo))
        out.append((name.value.decode(), mw.value, pw.value, ew.value, bool(lo.value)))
    return out


class _Named:
    def __init__(self, ctx, handle, free, names, heights):
        self.ctx, self._h, self._free, self.names, self.heights = ctx, handle, free, names, heights

    def free(self):
        if self._h:
            self._free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:  # interpreter shutdown: module globals may already be gone
            pass


def _named_mats(named):
    names = [k for k, _ in named]
    arr, keep = _mats([v for _, v in named])
    cn = (C.c_char_p * len(names))(*[n.encode() for n in names])
    return cn, arr, keep


def verify_shard(vk_commit, prep_names, prep_heights, proof_words, log_blowup=1, num_queries=84, pow_bits=16, repr=REPR_CANONICAL, options=None, core=False):
    """`Verifier::verify_shard` (crates/stark/src/verifier.rs:27-216) in native host code, on the serialised proof of
    `CudaProver.open_raw` / `prove_program(raw=True)`.  vk = (preprocessed commitment, names and heights of the
    preprocessed traces in proving-key order: `pk.commit, pk.names, pk.heights`).  Returns None when the proof is
    accepted, else the reference's error name.  Needs no GPU."""
    com = _u32(vk_commit)
    words = _u32(proof_words)
    names = (C.c_char_p * len(prep_names))(*[n.encode() for n in prep_names])
    logs = _u32([int(h).bit_length() - 1 for h in prep_heights])
    err = C.create_string_buffer(256)
    opt = _u32([1, 0, 0])  # defaults of bfgpu_set_transcript_option
    for k, v in (options or {}).items():
        opt[Context.OPTIONS[k]] = int(v)
    fn = lib().bfgpu_verify_core_proof if core else lib().bfgpu_verify_shard_ex
    rc = fn(com.ctypes.data_as(_u32p), names, logs.ctypes.data_as(_u32p), len(prep_names), words.ctypes.data_as(_u32p), words.size,
            repr, log_blowup, num_queries, pow_bits, opt.ctypes.data_as(_u32p), 3, err, 256)
    return None if rc == 0 else (err.value.decode() or f"error {rc}")


def verify_core_proof(vk_commit, prep_names, prep_heights, proof_words, log_blowup=1, num_queries=84, pow_bits=16, repr=REPR_CANONICAL, options=None):
    """`BfProver::verify` (crates/prover/src/verify.rs:10-36): the Cpu chip must be present (MissingCpuInFirstShard) with a log degree of
    at most 22 (CpuLogDegreeTooLarge: n), then `StarkMachine::verify` -> `verify_shard`, whose errors read "InvalidShardProof: ...".
    Returns None when accepted.  Needs no GPU."""
    return verify_shard(vk_commit, prep_names, prep_heights, proof_words, log_blowup, num_queries, pow_bits, repr, options, core=True)


def verify_batch(ctx, items, log_blowup=1, num_queries=84, pow_bits=16, repr=REPR_CANONICAL, options=None, core=True):
    """Verify many serialised proofs in one device call (bfgpu_verify_batch).  items: list of (vk_commit, prep_names, prep_heights,
    proof_words).  Returns one entry per item: None when accepted, else exactly the string `verify_core_proof` (core=True) or
    `verify_shard` (core=False) returns for it."""
    keep = []
    arr = (VerifyItem * max(len(items), 1))()
    for i, (com, names, heights, words) in enumerate(items):
        com, words = _u32(com), _u32(words)
        cn = (C.c_char_p * max(len(names), 1))(*[n.encode() for n in names])
        logs = _u32([int(h).bit_length() - 1 for h in heights])
        keep += [com, words, cn, logs]
        arr[i] = VerifyItem(com.ctypes.data_as(_u32p), cn, logs.ctypes.data_as(_u32p), len(names), words.ctypes.data_as(_u32p), words.size)
    opt = _u32([1, 0, 0])  # defaults of bfgpu_set_transcript_option
    for k, v in (options or {}).items():
        opt[Context.OPTIONS[k]] = int(v)
    status = (C.c_int32 * max(len(items), 1))()
    errs = C.create_string_buffer(256 * max(len(items), 1))
    ctx.check(lib().bfgpu_verify_batch(ctx._h, C.byref(arr), len(items), repr, log_blowup, num_queries, pow_bits, opt.ctypes.data_as(_u32p), 3, int(core),
                                       status, errs, 256))
    return [None if status[i] == 0 else (errs.raw[256 * i:256 * (i + 1)].split(b"\0")[0].decode() or f"error {status[i]}") for i in range(len(items))]


def proof_to_bincode(prep_names, prep_heights, proof_words, log_blowup=1, repr=REPR_CANONICAL, field_repr=1):
    """`bincode::serialize(&MachineProof { shard_proof })` (crates/core/machine/src/utils/prove.rs:47) of a serialised proof: the bytes a
    Rust caller deserialises, `len()` of which is the reference's `proofSize`.  field_repr 1 = Montgomery words (p3-monty-31 serde), 0 =
    canonical.  Needs no GPU."""
    words = _u32(proof_words)
    names = (C.c_char_p * len(prep_names))(*[n.encode() for n in prep_names])
    logs = _u32([int(h).bit_length() - 1 for h in prep_heights])
    err = C.create_string_buffer(256)
    n = C.c_uint64()
    args = (names, logs.ctypes.data_as(_u32p), len(prep_names), words.ctypes.data_as(_u32p), words.size, repr, log_blowup, field_repr)
    rc = lib().bfgpu_shard_proof_to_bincode(*args, None, 0, C.byref(n), err, 256)
    if rc != 0:
        raise BfGpuError(f"bfgpu_shard_proof_to_bincode: {err.value.decode()}")
    out = np.zeros(n.value, np.uint8)
    rc = lib().bfgpu_shard_proof_to_bincode(*args, out.ctypes.data_as(C.c_void_p), out.size, C.byref(n), err, 256)
    if rc != 0:
        raise BfGpuError(f"bfgpu_shard_proof_to_bincode: {err.value.decode()}")
    return out.tobytes()


class Record:
    """ExecutionRecord of the native executor (`Program::from` + `Executor::run`, crates/core/executor/src/
    program.rs:22-44, executor.rs:71-79,106-325): one 16-byte record per cycle, kept in page-locked memory when a
    context is given.  ctx=None runs without a device (host logic tests)."""

    def __init__(self, code, stdin=(), ctx=None, max_cycles=0):
        self.ctx = ctx
        self._h = C.c_void_p()
        inp = np.ascontiguousarray(np.asarray(list(stdin), np.uint8))
        rc = lib().bfgpu_execute(ctx._h if ctx is not None else None, code.encode(), _ptr(inp) if inp.size else None, inp.size, max_cycles,
                                 C.byref(self._h))
        if rc != 0:
            msg = lib().bfgpu_record_error(self._h).decode() if self._h else "allocation failed"
            self.free()
            raise BfGpuError(f"bfgpu_execute failed ({rc}): {msg}")
        c = (C.c_uint64 * 8)()
        lib().bfgpu_record_info(self._h, c)
        (self.cycles, self.n_instr, self.n_alu, self.n_jump, self.n_mem_instr, self.n_io, self.n_cells, n_out) = [int(x) for x in c]
        out = np.zeros(max(n_out, 1), np.uint8)
        lib().bfgpu_record_output(self._h, _ptr(out))
        self.output = out[:n_out].tolist()

    def cycle_records(self):
        """(cycles + 1, 4) uint32: pc, mp, previous timestamp of the cell, mv | previous value << 8 (last row = sentinel)."""
        p = lib().bfgpu_record_cycles(self._h)
        return np.ctypeslib.as_array(C.cast(p, _u32p), shape=(self.cycles + 1, 4)).copy()

    def memory_events(self):
        if not self.n_cells:
            return np.zeros((0, 5), np.uint32)
        p = lib().bfgpu_record_mem_events(self._h)
        return np.ctypeslib.as_array(C.cast(p, _u32p), shape=(self.n_cells, 5)).copy()

    def program(self):
        ops, args = np.zeros(self.n_instr, np.uint32), np.zeros(self.n_instr, np.uint32)
        lib().bfgpu_record_program(self._h, ops.ctypes.data_as(_u32p), args.ctypes.data_as(_u32p))
        return ops, args

    def free(self):
        if getattr(self, "_h", None):
            lib().bfgpu_record_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:  # interpreter shutdown: module globals may already be gone
            pass


class CudaProver:
    """`MachineProver<KoalaBearPoseidon2, BfAir>` on the GPU (reference trait: crates/stark/src/prover.rs:27-150;
    CPU implementation it replaces: `CpuProver`, prover.rs:162-582)."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.chips = machine_chips()

    def _sorted(self, traces):
        return sorted(traces.items(), key=lambda kv: (-kv[1].shape[0], kv[0]))

    def setup(self, prep_traces):
        """StarkMachine::setup: {chip name: preprocessed trace} -> (proving key handle, commitment)."""
        named = list(prep_traces.items())
        cn, arr, keep = _named_mats(named)
        commit = np.zeros(8, np.uint32)
        h = C.c_void_p()
        self.ctx.check(lib().bfgpu_machine_setup(self.ctx._h, cn, arr, len(named), commit.ctypes.data_as(_u32p), C.byref(h)))
        srt = self._sorted(prep_traces)
        pk = _Named(self.ctx, h, lib().bfgpu_pk_free, [k for k, _ in srt], [v.shape[0] for _, v in srt])
        pk.commit = commit
        pk.widths = [v.shape[1] for _, v in srt]
        return pk

    def commit(self, traces):
        """MachineProver::commit: {chip name: main trace} -> ShardMainData handle (root in .commit)."""
        named = list(traces.items())
        cn, arr, keep = _named_mats(named)
        root = np.zeros(8, np.uint32)
        h = C.c_void_p()
        self.ctx.check(lib().bfgpu_machine_commit(self.ctx._h, cn, arr, len(named), root.ctypes.data_as(_u32p), C.byref(h)))
        srt = self._sorted(traces)
        sd = _Named(self.ctx, h, lib().bfgpu_shard_free, [k for k, _ in srt], [v.shape[0] for _, v in srt])
        sd.commit = root
        return sd

    def execute(self, code, stdin=()):
        """`Executor::run`: native interpreter writing the cycle records into page-locked memory."""
        return Record(code, stdin, self.ctx)

    def setup_record(self, rec):
        """StarkMachine::setup for the record's program (preprocessed traces are built inside the library)."""
        commit = np.zeros(8, np.uint32)
        h = C.c_void_p()
        self.ctx.check(lib().bfgpu_machine_setup_record(self.ctx._h, rec._h, commit.ctypes.data_as(_u32p), C.byref(h)))
        prows = max(16, 1 << max(rec.n_instr - 1, 0).bit_length())
        srt = sorted([("Program", prows, 6), ("Byte", 65536, 2)], key=lambda t: (-t[1], t[0]))
        pk = _Named(self.ctx, h, lib().bfgpu_pk_free, [t[0] for t in srt], [t[1] for t in srt])
        pk.commit = commit
        pk.widths = [t[2] for t in srt]
        return pk

    def commit_record(self, rec):
        """MachineProver::commit with the main traces generated on the device from the execution record."""
        root = np.zeros(8, np.uint32)
        h = C.c_void_p()
        self.ctx.check(lib().bfgpu_machine_commit_record(self.ctx._h, rec._h, root.ctypes.data_as(_u32p), C.byref(h)))
        names, heights = [], []
        for i in range(lib().bfgpu_shard_num_traces(h)):
            nm, r, c = C.c_char_p(), C.c_uint64(), C.c_uint64()
            lib().bfgpu_shard_trace_info(h, i, C.byref(nm), C.byref(r), C.byref(c))
            names.append(nm.value.decode())
            heights.append(r.value)
        sd = _Named(self.ctx, h, lib().bfgpu_shard_free, names, heights)
        sd.commit = root
        return sd

    def shard_traces(self, shard):
        """{chip: main trace (rows, width)} held by a shard, natural row order (test hook)."""
        out = {}
        for i in range(lib().bfgpu_shard_num_traces(shard._h)):
            nm, r, c = C.c_char_p(), C.c_uint64(), C.c_uint64()
            lib().bfgpu_shard_trace_info(shard._h, i, C.byref(nm), C.byref(r), C.byref(c))
            a = np.zeros((r.value, c.value), np.uint32)
            self.ctx.check(lib().bfgpu_shard_get_trace(shard._h, i, _ptr(a)))
            out[nm.value.decode()] = a
        return out

    def prove_program(self, code, stdin=(), pk=None, pow_witness=None, raw=False):
        """`ProverClient::prove` (sdk/lib.rs, prover/lib.rs:70-90) end to end on the GPU backend: execute, generate the
        traces on the device, commit, open.  Returns (proof | (words, decoder), record)."""
        rec = self.execute(code, stdin)
        own_pk = pk is None
        if own_pk:
            pk = self.setup_record(rec)
        ch = Challenger(self.ctx)
        lib().bfgpu_pk_observe_into(pk._h, ch._h)
        shard = self.commit_record(rec)
        try:
            buf = self.open_raw(pk, shard, ch.clone(), pow_witness)
        finally:  # a failing open must not keep the main LDEs alive until the garbage collector gets to them
            shard.free()
        res = (buf, (lambda: self._parse(buf, pk, None))) if raw else self._parse(buf, pk, None)
        return res, rec

    def prove_many(self, jobs, pk_for=None, prefetch=1):
        """Proofs of a stream of (code, stdin) jobs with the host interpreter of job k+1 running while the GPU proves
        job k (the executor is sequential host code, ~4 ns/cycle; the C call releases the GIL).  Yields
        (serialised proof words, Record) in job order.  pk_for(code) -> proving key (default: one setup per distinct
        program, cached)."""
        import queue
        import threading
        pks = {}

        def get_pk(code, rec):
            if pk_for is not None:
                return pk_for(code)
            if code not in pks:
                pks[code] = self.setup_record(rec)
            return pks[code]

        q = queue.Queue(maxsize=max(1, prefetch))

        def producer():
            try:
                for code, stdin in jobs:
                    q.put((code, self.execute(code, stdin)))
                q.put(None)
            except BaseException as e:  # surface executor errors in the consumer
                q.put(e)

        th = threading.Thread(target=producer, daemon=True)
        th.start()
        while True:
            item = q.get()
            if item is None:
                break
            if isinstance(item, BaseException):
                raise item
            code, rec = item
            pk = get_pk(code, rec)
            ch = Challenger(self.ctx)
            lib().bfgpu_pk_observe_into(pk._h, ch._h)
            shard = self.commit_record(rec)
            try:
                buf = self.open_raw(pk, shard, ch.clone())
            finally:
                shard.free()
            item = None
            yield buf, rec
            del buf, rec  # the record's page-locked buffer goes back to the context's pool for the next execution
        th.join()
        for pk in pks.values():
            pk.free()

    def open(self, pk, shard, challenger, pow_witness=None):
        """MachineProver::open -> ShardProof as nested dicts (commitment, opened_values per chip, opening_proof, chip_ordering)."""
        buf = self.open_raw(pk, shard, challenger, pow_witness)
        return self._parse(buf, pk, shard)

    def open_raw(self, pk, shard, challenger, pow_witness=None):
        """MachineProver::open returning the serialised proof words (layout: include/bfgpu.h, bfgpu_machine_open)."""
        h = C.c_void_p()
        self.ctx.check(lib().bfgpu_machine_open(self.ctx._h, pk._h, shard._h, challenger._h, -1 if pow_witness is None else int(pow_witness), C.byref(h)))
        size = lib().bfgpu_shard_proof_size(h)
        buf = np.zeros(size, np.uint32)
        self.ctx.check(lib().bfgpu_shard_proof_read(h, _ptr(buf)))
        lib().bfgpu_shard_proof_free(h)
        return buf

    def prove(self, pk, traces, challenger, pow_witness=None, raw=False):
        """MachineProver::prove (prover.rs:560-582) minus trace generation: observe pk, commit, open on a clone.
        raw=True returns (serialised proof words, decoder) so that callers can time the prover without the Python decoding."""
        lib().bfgpu_pk_observe_into(pk._h, challenger._h)
        shard = self.commit(traces)
        try:
            if raw:
                buf = self.open_raw(pk, shard, challenger.clone(), pow_witness)
                return buf, (lambda: self._parse(buf, pk, None))
            return self.open(pk, shard, challenger.clone(), pow_witness)
        finally:
            shard.free()

    def debug_constraints(self, pk, shard, challenger, max_rows=5, max_keys=64):
        """`StarkMachine::debug_constraints` (machine.rs:288-387) on the GPU: every constraint on every row and the balance of
        every interaction of a committed shard (bfgpu_machine_debug).  `challenger` is left unchanged; in the state `open` would
        receive (pk observed) the report's cumulative sums are the proof's.  Returns a DebugReport."""
        h = C.c_void_p()
        self.ctx.check(lib().bfgpu_machine_debug(self.ctx._h, pk._h, shard._h, challenger._h, int(max_rows), int(max_keys), C.byref(h)))
        buf = np.zeros(lib().bfgpu_debug_report_size(h), np.uint32)
        rc = lib().bfgpu_debug_report_read(h, _ptr(buf))
        lib().bfgpu_debug_report_free(h)
        self.ctx.check(rc)
        return DebugReport(buf, [c[0] for c in self.chips], max_rows)

    def debug_program(self, code, stdin=(), max_rows=5, max_keys=64):
        """execute -> setup_record -> commit_record -> debug_constraints: checks the device trace generators on a program."""
        rec = self.execute(code, stdin)
        pk = self.setup_record(rec)
        ch = Challenger(self.ctx)
        lib().bfgpu_pk_observe_into(pk._h, ch._h)
        shard = self.commit_record(rec)
        try:
            return self.debug_constraints(pk, shard, ch, max_rows, max_keys)
        finally:
            shard.free()
            pk.free()

    def _parse(self, buf, pk, shard):
        info = {n: (mw, pw, ew, lo) for n, mw, pw, ew, lo in self.chips}
        com = dict(main=buf[0:8].copy(), permutation=buf[8:16].copy(), quotient=buf[16:24].copy())
        n = int(buf[24])
        pos = 25
        meta = []
        for _ in range(n):
            meta.append((self.chips[int(buf[pos])][0], int(buf[pos + 1]), buf[pos + 2:pos + 6].astype(np.uint64)))
            pos += 6

        class _D:  # dims carrier for the opening parser
            pass

        def dims(heights, widths):
            d = _D()
            d.dims = [(2 * h, w) for h, w in zip(heights, widths)]
            return d

        names = [m[0] for m in meta]
        heights = [1 << m[1] for m in meta]
        pts = lambda lo: [None] if lo else [None, None]
        rounds = [
            (dims(pk.heights, pk.widths), [pts(info[k][3]) for k in pk.names]),
            (dims(heights, [info[k][0] for k in names]), [pts(info[k][3]) for k in names]),
            (dims(heights, [4 * info[k][2] for k in names]), [[None, None] for _ in names]),
            (dims([h for h in heights for _ in range(2)], [4] * (2 * n)), [[None] for _ in range(2 * n)]),
        ]
        opened, fri = TwoAdicFriPcs._parse_opening(buf[pos:], rounds)
        prep_v, main_v, perm_v, quot_v = opened
        chips_out = []
        for i, (name, log_degree, csum) in enumerate(meta):
            lo = info[name][3]

            def lv(vals, both):
                return dict(local=vals[0], next=vals[1] if both else np.zeros_like(vals[0]))

            if name in pk.names:
                k = pk.names.index(name)
                prep = lv(prep_v[k], not info[pk.names[k]][3])
            else:
                prep = dict(local=np.zeros((0, 4), np.uint64), next=np.zeros((0, 4), np.uint64))
            chips_out.append(dict(preprocessed=prep, main=lv(main_v[i], not lo), permutation=lv(perm_v[i], True),
                                  quotient=[quot_v[2 * i][0], quot_v[2 * i + 1][0]], cumulative_sum=csum, log_degree=log_degree))
        return dict(commitment=com, opened_values=chips_out, opening_proof=fri, chip_ordering={k: i for i, k in enumerate(names)})


KIND_NAMES = {1: "Memory", 2: "Program", 3: "Alu", 4: "Jump", 5: "MemInstr", 6: "IO", 7: "Byte"}  # LookupKind (lookup.rs:19-41)
_N_BASE = {}  # chip -> (base constraints, LogUp batch columns), from air/chips.py on first use


def constraint_label(chip, k):
    """Name of constraint k of a chip in fold order: "base k", "LogUp batch j", "LogUp first row" / "transition" / "last row"."""
    if not _N_BASE:
        from .air import chips as air_chips
        _N_BASE.update({c.name: (len(c.constraints), c.perm_width - 1) for c in air_chips.machine_chips()})
    n_base, n_batch = _N_BASE[chip]
    if k < n_base:
        return f"base {k}"
    if k < n_base + n_batch:
        return f"LogUp batch {k - n_base}"
    return "LogUp " + ("first row", "transition", "last row")[k - n_base - n_batch]


class DebugReport:
    """Parsed bfgpu_machine_debug report (layout: include/bfgpu.h).
      failures        [(chip, constraint index, label, failing-row count, first rows)] in (commit order, index) order
      cumulative_sums {chip: (4,) words}, total: their sum (zero when the interactions balance)
      imbalances      [(kind name, values tuple, net, {chip: net})] in (kind, values) order, at most max_keys of n_imbalanced
      ok              no failing constraint, no imbalanced key, zero total"""

    def __init__(self, words, chip_names, max_rows):
        w = [int(x) for x in words]
        pos = 0

        def take(k=None):
            nonlocal pos
            pos += 1 if k is None else k
            return w[pos - 1] if k is None else w[pos - k:pos]

        self.words = np.asarray(words, np.uint32)
        self.failures, self.cumulative_sums, self.log_degrees = [], {}, {}
        for _ in range(take()):
            chip = chip_names[take()]
            self.log_degrees[chip] = take()
            self.cumulative_sums[chip] = np.array(take(4), np.uint64)
            for _ in range(take()):
                k, count = take(), take()
                self.failures.append((chip, k, constraint_label(chip, k), count, take(min(count, max_rows))))
        self.total = np.array(take(4), np.uint64)
        self.n_imbalanced = take()
        self.imbalances = []
        while pos < len(w):
            kind, nv = take(), take()
            values, net = tuple(take(nv)), take()
            per_chip = {}
            for _ in range(take()):
                c = take()
                per_chip[chip_names[c]] = take()
            self.imbalances.append((KIND_NAMES[kind], values, net, per_chip))
        self.ok = not self.failures and self.n_imbalanced == 0 and not self.total.any()

    def __str__(self):
        """The report in the reference's terms (debug.rs / lookup/debug.rs)."""
        out = []
        for chip, k, label, count, rows in self.failures:
            more = f" (+{count - len(rows)} more)" if count > len(rows) else ""
            out.append(f"constraint failed: chip {chip}, constraint {k} ({label}), {count} row(s): {', '.join(map(str, rows))}{more}")
        out.append("constraints: ok" if not self.failures else f"constraints: {len(self.failures)} failing")
        for kind, values, net, per_chip in self.imbalances:
            chips = ", ".join(f"{c}: {_signed(v)}" for c, v in per_chip.items())
            out.append(f"interaction imbalance: {kind} {list(values)}: net {_signed(net)} ({chips})")
        if self.n_imbalanced > len(self.imbalances):
            out.append(f"... {self.n_imbalanced - len(self.imbalances)} more imbalanced keys")
        out.append("lookups: ok" if self.n_imbalanced == 0 and not self.total.any() else
                   f"lookups: {self.n_imbalanced} imbalanced key(s), cumulative sums total {self.total.tolist()}")
        return "\n".join(out)


def _signed(v):
    """A multiplicity mod p as the small signed integer it stands for (sends positive, receives negative)."""
    return v - P if v > P // 2 else v


# ---- sdk façade -----------------------------------------------------------------------------------------------------------
class _Action:
    def __init__(self, fn):
        self._fn = fn

    def run(self):
        return self._fn()


class ProofWithPublicValues:
    """`BfProofWithPublicValues` (crates/sdk/src/proof.rs:10-13): the shard proof (serialised words; `.decode()` gives the
    nested form) and the stdin it was produced for; `output` is what the program wrote."""

    def __init__(self, words, decode, stdin, output):
        self.words, self._decode, self.stdin, self.output = words, decode, list(stdin), list(output)

    def decode(self):
        return self._decode()


class ProverClient:
    """`bf_sdk::ProverClient` (crates/sdk/src/lib.rs:19-140) on this backend, same call shapes:
        client = ProverClient(); pk, vk = client.setup(code); proof = client.prove(pk, [17]).run(); client.verify(proof, vk)
    `execute(code, stdin).run()` returns the program's output.  setup / prove need a GPU; execute and verify do not."""

    def __init__(self, device=0):
        self._device, self._ctx, self._prover = device, None, None

    def _gpu(self):
        if self._prover is None:
            self._ctx = Context(self._device)
            self._prover = CudaProver(self._ctx)
        return self._prover

    def execute(self, code, stdin=()):
        return _Action(lambda: Record(code, stdin).output)

    def setup(self, code):
        prover = self._gpu()
        pk = prover.setup_record(_ProgramOnly(code))
        pk.code = code
        vk = dict(commit=pk.commit.copy(), names=list(pk.names), heights=list(pk.heights))
        return pk, vk

    def prove(self, pk, stdin=()):
        def run():
            (words, decode), rec = self._gpu().prove_program(pk.code, stdin, pk=pk, raw=True)
            return ProofWithPublicValues(words, decode, stdin, rec.output)
        return _Action(run)

    def verify(self, proof, vk, log_blowup=1, num_queries=None, pow_bits=16):
        """`BfProver::verify` (crates/prover/src/verify.rs:10-36).  Returns None when accepted, else the reference's error name
        (`MachineVerificationError`: MissingCpuInFirstShard, CpuLogDegreeTooLarge: n, InvalidShardProof: <VerificationError>)."""
        if num_queries is None:
            num_queries = int(os.environ.get("FRI_QUERIES", 84))  # kb31_poseidon2.rs:59-62
        return verify_core_proof(vk["commit"], vk["names"], vk["heights"], proof.words, log_blowup, num_queries, pow_bits)


class _ProgramOnly:
    """Handle for `bfgpu_machine_setup_record` built from the program text alone (no execution)."""

    def __init__(self, code):
        self._h = C.c_void_p()
        rc = lib().bfgpu_execute(None, code.encode(), None, 0, 1, C.byref(self._h))
        # a one-cycle budget: programs longer than one cycle stop with "cycle limit"; the compiled program is kept either way
        if rc != 0:
            msg = lib().bfgpu_record_error(self._h).decode() if self._h else ""
            if "cycle limit" not in msg and "stdin" not in msg:
                lib().bfgpu_record_free(self._h)
                self._h = None
                raise BfGpuError(f"program does not compile: {msg}")
        c = (C.c_uint64 * 8)()
        lib().bfgpu_record_info(self._h, c)
        self.n_instr = int(c[1])

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                lib().bfgpu_record_free(self._h)
                self._h = None
        except Exception:  # interpreter shutdown: module globals may already be gone
            pass
