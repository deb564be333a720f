"""The unbanded traceback pointer-block layouts of aligntools/c_b200/csrc/at_ptr_layout.h, compiled with g++
(tests/ptr_layout_model.cpp): the block sizes and groups keep the numbers the runtime, K1, K2 and K3 have always used,
every cell has its own slot inside its pair's block, the slot K3 reads is the one the fill stores, and the layout class
byte round-trips."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_build", "libptr_layout_model.so")
SRC = os.path.join(HERE, "ptr_layout_model.cpp")
HDRS = [os.path.join(HERE, "..", "aligntools", "c_b200", "csrc", h) for h in ("at_ptr_layout.h", "at_cell.cuh")]

SH_PACKED, SH_NIB, SH_2BIT, SH_JUMP = 2, 3, 4, 5
L1S = [1, 31, 32, 33, 255, 256, 257, 1023, 1024, 1025, 4096, 20000]
L2S = list(range(1, 71)) + [255, 256, 257, 10007]


@pytest.fixture(scope="module")
def lib():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(x) for x in [SRC] + HDRS):
        subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-shared", "-fPIC", "-x", "c++", "-o", SO, SRC], check=True)
    L = C.CDLL(SO)
    u32, u64, i32, vp = C.c_uint32, C.c_uint64, C.c_int, C.c_void_p
    sig = {
        "ptr_model_last_step": ([u32, u32, i32], u32),
        "ptr_model_groups": ([u32, u32], u32),
        "ptr_model_plane_words": ([u32, u32, u32], u64),
        "ptr_model_pair_words": ([u32, u32, u32, u32, i32], u64),
        "ptr_model_packed_job_words": ([u32, u32], u64),
        "ptr_model_edit_bits_groups": ([u32], u32),
        "ptr_model_edit_bits_last_step": ([u32], u32),
        "ptr_model_edit_bits_words": ([u32, u32, u32], u64),
        "ptr_model_class": ([u32, u32], u32),
        "ptr_model_class_r": ([u32], u32),
        "ptr_model_class_half": ([u32], u32),
        "ptr_model_cells": ([u32, u32, u32, u32, u32, u32, vp, vp], u64),
        "ptr_model_edit_bits_cells": ([u32, u32, u32, u32, vp, vp], None),
    }
    for name, (args, res) in sig.items():
        getattr(L, name).argtypes = args
        getattr(L, name).restype = res
    return L


# ---- the formulas each site wrote out before the layout moved into at_ptr_layout.h, copied literally ----

def old_ptr_words_of(mode_2bit, jump, R, l1, l2):          # at_runtime.cu ptr_words_of (R = rclass_of(l1))
    RPP = 32 * R
    stripes = (l1 + RPP - 1) // RPP
    if mode_2bit:
        tl = (l2 + 31) | 15
        return stripes * ((tl >> 4) + 1) * RPP
    tl = (l2 + 31) | (31 if jump else 7)
    w = stripes * ((tl >> 3) + 1) * RPP
    if jump:
        w += stripes * ((tl >> 5) + 1) * RPP
    return w


def old_packed_job_words(R, l2):                            # at_runtime.cu, uniform and general plan
    tl = (l2 + 31) | 3
    return ((tl >> 2) + 1) * R * 32


def old_edit_bits_words(R, l1, l2):                         # at_runtime.cu edit_bits_words
    stripes, G = (l1 + 1024 * R - 1) // (1024 * R), (((l2 + 63) | 15) >> 4) + 1
    return stripes * G * R * 1024


def old_k1(l2, jump, packed):                               # at_fill_affine.cuh: t_last (the loop bound), G
    spw = 4 if packed else 8
    t_last = (l2 + 31) | (31 if jump else spw - 1)
    return t_last, t_last // spw + 1


def old_k3(l2, overlap, half, jump):                        # at_kernels.cuh at_traceback_walk: G, GJ
    if overlap:
        return (((l2 + 31) | 15) >> 4) + 1, 0
    if half:
        return (((l2 + 31) | 3) >> 2) + 1, 0
    tl = (l2 + 31) | (31 if jump else 7)
    return (tl >> 3) + 1, (tl >> 5) + 1


def test_layout_numbers_unchanged(lib):
    for l2 in L2S:
        for jump in (False, True):
            for packed in (False, True):
                if packed and jump:
                    continue
                sh = SH_PACKED if packed else SH_NIB
                t_last, G = old_k1(l2, jump, packed)
                last = lib.ptr_model_last_step(l2, sh, jump)
                assert (last, lib.ptr_model_groups(last, sh)) == (t_last, G), (l2, jump, packed)
            # K2 affine and K3's int32 layout: groups and jump groups from the same last step
            tl = (l2 + 31) | (31 if jump else 7)
            last = lib.ptr_model_last_step(l2, SH_NIB, jump)
            assert (lib.ptr_model_groups(last, SH_NIB), lib.ptr_model_groups(last, SH_JUMP)) == ((tl >> 3) + 1, (tl >> 5) + 1)
            assert (lib.ptr_model_groups(last, SH_NIB), lib.ptr_model_groups(last, SH_JUMP)) == old_k3(l2, False, 0, jump)
        # K2 linear and K3's overlap / cell-by-cell edit layout; K3's packed layout
        g2 = lib.ptr_model_groups(lib.ptr_model_last_step(l2, SH_2BIT, 0), SH_2BIT)
        assert g2 == (((l2 + 31) | 15) >> 4) + 1 == old_k3(l2, True, 0, False)[0]
        assert lib.ptr_model_groups(lib.ptr_model_last_step(l2, SH_PACKED, 0), SH_PACKED) == old_k3(l2, False, 1, False)[0]
        # K2 bit-parallel: loop bound and groups
        assert lib.ptr_model_edit_bits_last_step(l2) == (l2 + 63) | 15
        assert lib.ptr_model_edit_bits_groups(l2) == (((l2 + 63) | 15) >> 4) + 1
        for R in range(1, 9):
            assert lib.ptr_model_packed_job_words(l2, R) == old_packed_job_words(R, l2), (l2, R)
            for l1 in L1S:
                n_stripes = (l1 + 32 * R - 1) // (32 * R)
                for jump in (False, True):
                    assert lib.ptr_model_pair_words(l1, l2, R, SH_NIB, jump) == old_ptr_words_of(False, jump, R, l1, l2), (l1, l2, R, jump)
                    G = old_k3(l2, False, 0, jump)[0]
                    assert lib.ptr_model_plane_words(n_stripes, G, R) == n_stripes * G * 32 * R     # jump-plane base (K2, K3)
                assert lib.ptr_model_pair_words(l1, l2, R, SH_2BIT, 0) == old_ptr_words_of(True, False, R, l1, l2), (l1, l2, R)
        for R in (1, 2, 4):
            for l1 in L1S:
                assert lib.ptr_model_edit_bits_words(l1, l2, R) == old_edit_bits_words(R, l1, l2), (l1, l2, R)


def cells(lib, l1, l2, R, G, sh, bits):
    n = l1 * l2
    word, shift = np.zeros(n, np.uint64), np.zeros(n, np.uint32)
    bad = lib.ptr_model_cells(l1, l2, R, G, sh, bits, word.ctypes.data, shift.ctypes.data)
    assert bad == 0, "K3's word of a cell differs from the one the fill stores"
    assert np.all(shift % bits == 0) and np.all(shift + bits <= 32)
    return word, shift


def assert_distinct(word, shift, bits, n_words, base=0):
    """Every cell's bit range [shift, shift + bits) of its word is its own and inside [base, n_words)."""
    assert word.min() >= base and word.max() < n_words
    key = word * 32 + shift
    assert len(np.unique(key)) == len(key)


def small_cases(R):
    rpp = 32 * R
    for l1 in (1, rpp - 1, rpp, rpp + 1, 2 * rpp + 3):
        for l2 in (1, 7, 8, 9, 33, 70):
            yield l1, l2


def test_cells_have_distinct_in_range_slots(lib):
    for R in range(1, 9):
        for l1, l2 in small_cases(R):
            stripes = (l1 + 32 * R - 1) // (32 * R)
            # 2-bit codes (overlap, cell-by-cell edit paths)
            G = lib.ptr_model_groups(lib.ptr_model_last_step(l2, SH_2BIT, 0), SH_2BIT)
            w, s = cells(lib, l1, l2, R, G, SH_2BIT, 2)
            assert_distinct(w, s, 2, lib.ptr_model_pair_words(l1, l2, R, SH_2BIT, 0))
            for jump in (False, True):
                # int32 nibbles, then the jump plane after them
                last = lib.ptr_model_last_step(l2, SH_NIB, jump)
                G, GJ = lib.ptr_model_groups(last, SH_NIB), lib.ptr_model_groups(last, SH_JUMP)
                total = lib.ptr_model_pair_words(l1, l2, R, SH_NIB, jump)
                plane = lib.ptr_model_plane_words(stripes, G, R)
                w, s = cells(lib, l1, l2, R, G, SH_NIB, 4)
                assert_distinct(w, s, 4, plane)
                if jump:
                    wj, sj = cells(lib, l1, l2, R, GJ, SH_JUMP, 1)
                    assert_distinct(wj + plane, sj, 1, total, base=plane)
                else:
                    assert total == plane
            # packed s16x2: one stripe, pair A in bits 0-15, pair B in bits 16-31 of the same words
            if l1 <= 32 * R:
                G = lib.ptr_model_groups(lib.ptr_model_last_step(l2, SH_PACKED, 0), SH_PACKED)
                w, s = cells(lib, l1, l2, R, G, SH_PACKED, 4)
                assert np.all(s < 16)
                both_w, both_s = np.concatenate([w, w]), np.concatenate([s, s + 16])
                assert_distinct(both_w, both_s, 4, lib.ptr_model_packed_job_words(l2, R))


def test_edit_bits_cells_have_distinct_in_range_slots(lib):
    for R in (1, 2, 4):
        rows = 1024 * R
        for l1 in (1, 33, rows - 1, rows, rows + 1):
            for l2 in (1, 15, 16, 17, 40):
                G = lib.ptr_model_edit_bits_groups(l2)
                n = l1 * l2
                slot, bit = np.zeros(n, np.uint64), np.zeros(n, np.uint32)
                lib.ptr_model_edit_bits_cells(l1, l2, R, G, slot.ctypes.data, bit.ctypes.data)
                assert np.all(bit < 32)
                assert 2 * int(slot.max()) + 1 < lib.ptr_model_edit_bits_words(l1, l2, R)    # a uint2 (LEFT, DIAG) per slot
                key = slot * 32 + bit
                assert len(np.unique(key)) == n, (R, l1, l2)


def test_layout_class_round_trips(lib):
    for R in range(1, 9):
        for half in range(3):
            c = lib.ptr_model_class(R, half)
            assert c < 256 and (lib.ptr_model_class_r(c), lib.ptr_model_class_half(c)) == (R, half)
