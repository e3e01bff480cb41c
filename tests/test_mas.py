"""Monotonic alignment search (SURVEY 8 f4): oracle vs the reference's own outputs (golden fixtures, and the compiled
reference when oracle/_ref/ exists), CUDA kernel vs oracle through the C ABI."""
import importlib.util
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
spec = importlib.util.spec_from_file_location("make_golden_mas", os.path.join(ROOT, "scripts", "make_golden_mas.py"))
mg = importlib.util.module_from_spec(spec)
spec.loader.exec_module(mg)

from oracle import build_oracle, mas_oracle  # noqa: E402


def golden(name):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    seed, b, tx, ty = (int(v) for v in g["meta"])
    v, t_xs, t_ys = mg.make_inputs(seed, b, tx, ty, str(g["kind"]))
    assert np.array_equal(t_xs, g["t_xs"]) and np.array_equal(t_ys, g["t_ys"])
    path = np.unpackbits(g["path_bits"], axis=-1)[..., :ty].astype(np.int32)
    return v, t_xs, t_ys, path


def oracle_path(v, t_xs, t_ys):
    p = np.zeros_like(v).astype(np.int32)
    mas_oracle.maximum_path_c(p, v.copy(), t_xs, t_ys)
    return p


@pytest.mark.parametrize("name", list(mg.CASES))
def test_oracle_matches_reference_golden(name):
    v, t_xs, t_ys, want = golden(name)
    assert np.array_equal(oracle_path(v, t_xs, t_ys), want)


def test_oracle_matches_compiled_reference():
    """The seeded sweep against the paths the compiled reference wrote (tests/golden/mas_seeded.npz), and against the
    compiled reference itself where oracle/_ref/ holds it."""
    ref = build_oracle.load_ref()
    g = np.load(os.path.join(GOLD, "mas_seeded.npz"))
    for i, (b, tx, ty, kind, (v, t_xs, t_ys)) in enumerate(mg.seeded_cases()):
        want = np.unpackbits(g["path_bits_%d" % i], axis=-1)[..., :ty].astype(np.int32)
        assert np.array_equal(oracle_path(v, t_xs, t_ys), want), i
        if ref is not None:
            live = np.zeros_like(v).astype(np.int32)
            ref.maximum_path_c(live, v.copy(), t_xs, t_ys)
            assert np.array_equal(live, want), i


def test_path_properties():
    """size-independent properties of a monotonic alignment: one token per frame, non-decreasing, surjective"""
    v, t_xs, t_ys = mg.make_inputs(7, 5, 60, 200, "ragged")
    p = oracle_path(v, t_xs, t_ys)
    for i in range(5):
        tx, ty = int(t_xs[i]), int(t_ys[i])
        assert p[i, :, ty:].sum() == 0 and p[i, tx:].sum() == 0
        assert np.array_equal(p[i, :tx, :ty].sum(0), np.ones(ty, np.int64))
        tok = p[i, :tx, :ty].argmax(0)
        assert tok[0] == 0 and tok[-1] == tx - 1 and np.all(np.diff(tok) >= 0) and np.all(np.diff(tok) <= 1)


def test_python_wrapper_matches_reference_wrapper_semantics():
    """maximum_path(value, mask): lengths come from the mask, value is multiplied by it (__init__.py:13-21)"""
    v, t_xs, t_ys = mg.make_inputs(21, 3, 10, 25, "ragged")
    mask = ((np.arange(10)[None, :, None] < t_xs[:, None, None]) & (np.arange(25)[None, None, :] < t_ys[:, None, None])).astype(np.float32)
    noise = np.random.default_rng(0).standard_normal(v.shape).astype(np.float32)        # garbage outside the mask must not matter
    got = mas_oracle.maximum_path(torch.from_numpy(v + noise * (1 - mask)), torch.from_numpy(mask))
    assert got.dtype == torch.float32 and np.array_equal(got.numpy().astype(np.int32), oracle_path(v, t_xs, t_ys))


# ------------------------------------------------------------------------------------------------ GPU parity
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(mg.CASES))
def test_gpu_matches_reference_golden(name):
    import emojivoice_b200 as ev

    v, t_xs, t_ys, want = golden(name)
    b, tx, ty = v.shape
    mask = ((np.arange(tx)[None, :, None] < t_xs[:, None, None]) & (np.arange(ty)[None, None, :] < t_ys[:, None, None])).astype(np.float32)
    got = ev.maximum_path(torch.from_numpy(v).cuda(), torch.from_numpy(mask).cuda())
    assert got.dtype == torch.float32 and got.is_cuda
    assert np.array_equal(got.cpu().numpy().astype(np.int32), want)


@pytest.mark.gpu
@pytest.mark.parametrize("b,tx,ty,kind", [(32, 181, 668, "ragged"), (8, 300, 2000, "ragged"), (4, 500, 4000, "ties"), (2, 1100, 1500, "full"),
                                          (3, 64, 64, "square")])
def test_gpu_matches_oracle_large(b, tx, ty, kind):
    """full-size batches (config 2 is 32 x 181 x 668), long utterances whose bit matrix spills to the workspace, and more
    text positions than threads per CTA"""
    import emojivoice_b200 as ev

    v, t_xs, t_ys = mg.make_inputs(31, b, tx, ty, kind)
    mask = ((np.arange(tx)[None, :, None] < t_xs[:, None, None]) & (np.arange(ty)[None, None, :] < t_ys[:, None, None])).astype(np.float32)
    got = ev.maximum_path(torch.from_numpy(v).cuda(), torch.from_numpy(mask).cuda()).cpu().numpy().astype(np.int32)
    assert np.array_equal(got, oracle_path(v, t_xs, t_ys))


@pytest.mark.gpu
def test_gpu_rejects_cpu_tensors():
    import emojivoice_b200 as ev

    with pytest.raises(RuntimeError):
        ev.maximum_path(torch.zeros(1, 2, 3), torch.ones(1, 2, 3))
