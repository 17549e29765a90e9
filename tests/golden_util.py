"""Shared helpers for the fixtures under tests/golden/ (written by oracle/gen_golden.py)."""
import glob
import os

import pytest
import torch

from oracle import msgchn_oracle as O

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
W_SD, W_SM, W_COS = 1.0, 1.0, 0.1
# The reference's fixtures reproduce with torch's CPU kernels on 8 threads.  The thread count (with the cache sizes) decides how a
# reduction is split, hence its summation order, and some stored values follow that rounding: a bias in front of a train-mode
# BatchNorm holds rounding noise that Adam turns into +-lr steps, and the BatchNorm's running mean carries it.  With 1-7 threads, or
# 16 on a CPU with other caches, those values move past the tolerances although the oracle is unchanged.
FIXTURE_THREADS = 8


@pytest.fixture
def fixture_threads():
    """runs a test with torch's CPU kernels on FIXTURE_THREADS threads"""
    saved = torch.get_num_threads()
    torch.set_num_threads(FIXTURE_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(saved)


def golden_names():
    return sorted(os.path.basename(p)[:-3] for p in glob.glob(os.path.join(GOLDEN_DIR, 'msgchn_*.pt')))


def load_golden(name):
    return torch.load(os.path.join(GOLDEN_DIR, name + '.pt'), weights_only=False)


def case_frame(case, t):
    image, sparse, dense = O.synthetic_frame(case['seq_seed'], t, case['n'], case['h'], case['w'], case['dataset'],
                                             depth_scale=case.get('depth_scale', 1.0))
    if case.get('density'):
        g = torch.Generator().manual_seed(77 + t)
        mask = (torch.rand(dense.shape, generator=g) < case['density']).float()
        sparse = dense * mask
    return image, sparse, dense


def case_checkpoint(case):
    """the checkpoint a fixture was generated from: a fitted one (case['ckpt'] names tests/golden/ckpt_*.pt) or the seeded
    randomly initialised stand-in"""
    return O.get_checkpoint(case.get('ckpt', case['ckpt_seed']), case['prepare_mode'])


def rel(a, b):
    return abs(a - b) / max(abs(b), 1e-12)


def nrel(a, b):
    """norm-wise relative error ||a-b|| / ||b||"""
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))
