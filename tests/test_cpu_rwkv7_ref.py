"""The f64 RWKV-7 restatement (tests/rwkv7_ref.py) against the f32 CPU oracle: the GPU deep-parity tests measure the CUDA kernels
against that restatement, so a wrong formula in it would make them fail, or pass, for the wrong reason."""
import os
import sys

import numpy as np
import pytest

import oracle
import parity_util as pu
import rwkv7_ref as rr

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from rwkv7_weights import RWKV7_TINY, long_memory, make_weights  # noqa: E402

# max |logit_oracle_f32 - logit_f64| / std(f64 logits) over 1,024 positions, measured on CPU (x86-64, the oracle built by
# oracle/Makefile): 5.8e-6 with the seed-7 weights, 4.5e-6 with the long-memory decay bias.  The assert allows 2x the larger.
# A formula slip is far above it: group-norm eps 1e-5 instead of 64e-5, or the decay offset -0.49, moves the logits by > 0.02.
TOL_F64_VS_F32_ORACLE = 2 * 5.8e-6


@pytest.mark.parametrize("long_mem", [False, True], ids=["seed7", "long_memory"])
def test_f64_forward_matches_f32_oracle_every_position(long_mem):
    cfg = RWKV7_TINY
    W = make_weights(cfg, 7)
    if long_mem:
        W = long_memory(W, cfg)
    toks = np.random.default_rng(3).integers(0, cfg["vocab"], 1024)
    ref = rr.forward(cfg, W, toks)
    orc = oracle.Session.rwkv7(cfg, W, round_bf16=0)
    got = np.stack([orc.step_logits(int(t)) for t in toks])
    r = pu.logits_parity(got, ref)
    assert r.max() < TOL_F64_VS_F32_ORACLE, (int(r.argmax()), float(r.max()))


def test_kernel_state_layout():
    """element (i, j) of a head's state sits at (j/4)*256 + i*4 + j%4 of the kernel's 4096 floats"""
    S = np.arange(2 * 64 * 64, dtype=np.float64).reshape(2, 64, 64)
    K = rr.state_to_kernel(S)
    i, j = np.meshgrid(np.arange(64), np.arange(64), indexing="ij")
    for h in range(2):
        assert np.array_equal(K[h][(j // 4) * 256 + i * 4 + j % 4], S[h])
    assert np.array_equal(rr.state_from_kernel(K), S)


def test_decay_edges():
    """the decay formula at the edges the scan kernel tests use: overflow of exp(-z) gives exactly 1, large z gives e^-e^-0.5"""
    assert rr.decay(np.array([-800.0]))[0] == 1.0
    assert abs(rr.decay(np.array([60.0]))[0] - np.exp(-np.exp(-0.5))) < 1e-15
    z = np.array([-12.0])
    assert 0 < 1.0 - rr.decay(z)[0] < 1e-4
