"""CPU side of the batch verifier (bf.verify_batch, `bfprove.py verify --device`): without a GPU it fails with the library's
no-CPU-fallback error instead of answering from the host, and the CLI refuses a verifying-key count that fits neither form."""
import os
import subprocess
import sys

import pytest

import zkvm_brainfuck_b200 as bf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(bf.BfGpuError, match="no CPU fallback"):
        bf.verify_batch(bf.Context(), [])


def test_cli_needs_one_vk_or_one_per_proof(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bfprove.py"), "verify", "a", "b", "c", "--vk", "x", "--vk", "y"], capture_output=True,
                       text=True, timeout=120)
    assert r.returncode == 2 and "--vk must be given once, or once per proof" in r.stderr
