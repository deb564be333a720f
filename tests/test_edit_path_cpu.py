"""Edit distance paths without a GPU.

* tests/edit_port.c (the CPU restatement of edit_dist with the AT_OUT_EDIT_PATH traceback) against the oracle's edit
  scores and the reference's stored answers, and every step of its path against a full min3 matrix;
* the kernels' pointer derivations (aligntools/c_b200/csrc/at_cell.cuh: edit_bits_ptr for the bit-parallel kernel,
  edit_min3_tagged for the cell-by-cell one) compiled with g++ (tests/edit_model.cpp) against a scalar min3."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

import edit_port
from helpers import load_fuzz

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_build", "libedit_model.so")
SRC = os.path.join(HERE, "edit_model.cpp")
HDR = os.path.join(HERE, "..", "aligntools", "c_b200", "csrc", "at_cell.cuh")


def full_matrix(s1, s2, u, top=None):
    """M as int64 (l1 + 1) x (l2 + 1) and the min3 first-argmin code (LEFT 0, DIAG 1, UP 2) of every inner cell."""
    l1, l2 = len(s1), len(s2)
    M = np.zeros((l1 + 1, l2 + 1), np.int64)
    M[0, :] = np.arange(l2 + 1) if top is None else np.concatenate(([0], np.cumsum(top)))
    M[:, 0] = np.arange(l1 + 1)
    code = np.zeros((l1 + 1, l2 + 1), np.uint8)
    for i in range(1, l1 + 1):
        for j in range(1, l2 + 1):
            c = (M[i, j - 1] + 1, M[i - 1, j - 1] + (0 if s1[i - 1] == s2[j - 1] else u), M[i - 1, j] + 1)
            k = 0
            if c[1] < c[k]:
                k = 1
            if c[2] < c[k]:
                k = 2
            M[i, j], code[i, j] = c[k], k
    return M, code


def path_cost(r1, r2, u):
    return sum(0 if a == b else (u if a != 45 and b != 45 else 1) for a, b in zip(r1, r2))


def rand_pair(rng, l1, l2, alphabet=b"ACGT"):
    s2 = bytes(rng.choice(alphabet) for _ in range(l2))
    s1 = bytearray()
    for ch in s2[:l1]:
        r = rng.random()
        s1 += bytes([rng.choice(alphabet)]) if r < 0.1 else (b"" if r < 0.14 else bytes([ch]))
    while len(s1) < l1:
        s1.append(rng.choice(alphabet))
    return bytes(s1[:l1]), s2


def test_scores_equal_oracle(oracle_mod):
    rng = random.Random(11)
    for k in range(300):
        s1, s2 = rand_pair(rng, rng.randint(1, 70), rng.randint(1, 70), b"ACGT" if k % 3 else b"ACDEFGHIKLMNPQRSTVWY")
        u = rng.choice([1, 2, 3, 0, -2, -1])
        ref = oracle_mod.port_align("edit", s1, s2, oracle_mod.Params(u=u))
        assert edit_port.align(s1, s2, u).score == ref.score, (k, u, s1, s2)


def test_scores_equal_stored_answers():
    cases = [c for c in load_fuzz() if c["mode"] == "edit"]
    assert cases
    for c in cases:
        assert edit_port.align(c["s1"].encode(), c["s2"].encode(), c["u"]).score == c["score"], c


@pytest.mark.parametrize("u", [1, 2, 3, 0, -2])
def test_path_follows_min3(u):
    """Every step of the walk is min3's first argmin at the cell it leaves; the path consumes both sequences; its cost
    (0 per equal column, u per unequal one, 1 per gap) is the score; beg is where the walk met row or column 0."""
    rng = random.Random(100 + u)
    for k in range(120):
        l1, l2 = rng.randint(1, 40), rng.randint(1, 40)
        s1, s2 = rand_pair(rng, l1, l2, b"ACGT" if k % 2 else b"AC")
        res = edit_port.align(s1, s2, u)
        M, code = full_matrix(s1, s2, u)
        assert res.score == M[l1, l2]
        assert res.coords[:2] == (l1, l2)
        assert res.r1.replace(b"-", b"") == s1 and res.r2.replace(b"-", b"") == s2
        assert path_cost(res.r1, res.r2, u) == res.score, (k, s1, s2)
        i, j = l1, l2
        for op in reversed(res.ops):
            if i == 0 or j == 0:
                break
            assert op == b"DMI"[code[i, j]], (k, i, j, s1, s2)
            i, j = i - (op != ord("D")), j - (op != ord("I"))
        assert (i, j) == res.coords[2:] and (i == 0 or j == 0)


@pytest.fixture(scope="module")
def model():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(SRC), os.path.getmtime(HDR)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", "-o", SO, SRC], check=True)
    lib = C.CDLL(SO)
    lib.edit_bits_model.restype = C.c_int
    lib.edit_bits_model.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.edit_cell_model.restype = C.c_int
    lib.edit_cell_model.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_void_p]
    return lib


def test_bit_planes_match_min3(model):
    """Bit-parallel pointer planes (u = 1) on random blocks: reads of 1..100 rows (bits 0 and 31 of several blocks), the
    row above drawn with horizontal differences -1 / 0 / +1 (a stripe's input) or +1 everywhere (row 0)."""
    rng = random.Random(7)
    seen = set()
    for k in range(400):
        l1, l2 = rng.choice([1, 31, 32, 33, 64, 65, rng.randint(1, 100)]), rng.randint(1, 60)
        s1, s2 = rand_pair(rng, l1, l2, b"ACGT" if k % 3 else b"AC")
        top = np.ones(l2, np.int8) if k % 2 else np.array([rng.choice([-1, 0, 1]) for _ in range(l2)], np.int8)
        seen.update(int(x) for x in top)
        code = np.zeros(l1 * l2, np.uint8)
        last = np.zeros(l2 + 1, np.int32)
        model.edit_bits_model(s1, l1, s2, l2, top.ctypes.data, code.ctypes.data, last.ctypes.data)
        M, ref = full_matrix(s1, s2, 1, top.astype(np.int64))
        assert np.array_equal(last, M[l1, :]), (k, s1, s2)
        bad = np.argwhere(code.reshape(l1, l2) != ref[1:, 1:])
        assert bad.size == 0, (k, s1, s2, top.tolist(), bad[:4].tolist())
    assert seen == {-1, 0, 1}


@pytest.mark.parametrize("u", [1, 2, 3, 0, -2])
def test_tagged_min3_matches_min3(model, u):
    rng = random.Random(40 + u)
    for k in range(150):
        l1, l2 = rng.randint(1, 50), rng.randint(1, 50)
        s1, s2 = rand_pair(rng, l1, l2, b"ACGT" if k % 2 else b"ACDEFGHIKLMNPQRSTVWY")
        code = np.zeros(l1 * l2, np.uint8)
        score = model.edit_cell_model(s1, l1, s2, l2, u, code.ctypes.data)
        M, ref = full_matrix(s1, s2, u)
        assert score == M[l1, l2]
        assert np.array_equal(code.reshape(l1, l2), ref[1:, 1:]), (k, s1, s2)
