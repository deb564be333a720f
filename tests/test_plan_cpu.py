"""The batch plan of aligntools/c_b200/csrc/at_plan.h, compiled with g++ (tests/plan_model.cpp): on seeded random shards
it equals a literal port of the planning loop setup_shard ran before the plan moved into the header, and it keeps the
invariants every kernel relies on -- each pair in one launch of one chunk, disjoint pointer blocks and boundary slabs
within their chunk's totals, class bytes that match the launch, task predecessors queued before their successors.  The
uniform closed form (uniform_pair, what at_plan_uniform writes on the device) matches the general plan, and
cut_by_prefix matches the slicing loop it replaced."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_build", "libplan_model.so")
SRC = os.path.join(HERE, "plan_model.cpp")
CSRC = os.path.join(HERE, "..", "aligntools", "c_b200", "csrc")
HDRS = [os.path.join(CSRC, h) for h in ("at_plan.h", "at_ptr_layout.h", "at_band.h", "at_cell.cuh")] + \
       [os.path.join(HERE, "..", "include", "aligntools_b200.h")]

GLOBAL, LOCAL, FIT, OVERLAP, EDIT = range(5)
LK_INT32, LK_PACKED, LK_WAVE, LK_BITS = range(4)
MAXR = 8
U64MAX = (1 << 64) - 1
NONE32 = (1 << 32) - 1


@pytest.fixture(scope="module")
def lib():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(x) for x in [SRC] + HDRS):
        subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-shared", "-fPIC", "-x", "c++", "-o", SO, SRC], check=True)
    L = C.CDLL(SO)
    u32, u64, i32, vp = C.c_uint32, C.c_uint64, C.c_int, C.c_void_p
    L.plan_model_plan.argtypes = [u32, vp, vp, i32, i32, i32, vp, vp, i32, u32, vp, i32, i32, i32, u64, vp, u64]
    L.plan_model_plan.restype = u64
    L.plan_model_uniform_pair.argtypes = [i32, u32, u64, u64, u32, u32, vp]
    L.plan_model_uniform_pair.restype = None
    L.plan_model_cut.argtypes = [vp, u64, u64, u64, u64, vp]
    L.plan_model_cut.restype = None
    L.plan_model_bits_r.argtypes = [vp, u32, u64]
    L.plan_model_bits_r.restype = u32
    return L


# ---- a shard ----

class Shard:
    def __init__(self, l1, l2, mode, traceback=False, jump=False, band=None, bits=False, bits_r=1, prm=(1, -2, -5, -1),
                 no_p16=False, allow_uniform=True, pair_major=False, budget=U64MAX):
        self.l1, self.l2, self.mode, self.traceback, self.jump = list(l1), list(l2), mode, traceback, jump
        self.band, self.bits, self.bits_r, self.prm, self.no_p16 = band, bits, bits_r, prm, no_p16
        self.allow_uniform, self.pair_major, self.budget = allow_uniform, pair_major, budget

    def __repr__(self):
        return repr(self.__dict__)


def c_plan(L, s):
    n = len(s.l1)
    a1, a2 = np.array(s.l1, np.uint32), np.array(s.l2, np.uint32)
    lo = hi = None
    if s.band is not None:
        lo, hi = np.array([b[0] for b in s.band], np.int32), np.array([b[1] for b in s.band], np.int32)
    prm = np.array(s.prm, np.int32)
    cap = 1 << 16
    while True:
        out = np.zeros(cap, np.uint64)
        need = L.plan_model_plan(n, a1.ctypes.data, a2.ctypes.data, s.mode, int(s.traceback), int(s.jump),
                                 None if lo is None else lo.ctypes.data, None if hi is None else hi.ctypes.data,
                                 int(s.bits), s.bits_r, prm.ctypes.data, int(s.no_p16), int(s.allow_uniform), int(s.pair_major),
                                 s.budget, out.ctypes.data, cap)
        if need <= cap:
            break
        cap = int(need)
    v = [int(x) for x in out[:need]]
    pos = 0

    def take(k=1):
        nonlocal pos
        r = v[pos:pos + k]
        pos += k
        return r

    def vec():
        return take(take()[0])

    need_words = take()[0]
    (uniform, packed, R, wpj, spp, cells, mcw, msw, mbe, mpw, mp, fail_pair, fail_words) = take(13)
    p = dict(need_words=need_words, uniform=uniform, cells=cells, max_chunk_words=mcw, max_scratch_words=msw,
             max_bnd_elems=mbe, max_prog_words=mpw, max_pairs=mp, fail_pair=fail_pair, fail_words=fail_words)
    p["u"] = dict(packed=packed, R=R, words_per_job=wpj, scratch_per_pair=spp) if uniform else None
    p["rclass"] = vec()
    chunks = []
    for _ in range(take()[0]):
        k0, k1, ptr_words, bnd_elems, prog_words, scratch_words, nl = take(7)
        launches = []
        for _ in range(nl):
            kind, r, lcells, ln, prog_base = take(5)
            jobs = [tuple(take(2)) for _ in range(take()[0])]
            tasks = [tuple(take(4)) for _ in range(take()[0])]
            launches.append(dict(kind=kind, r=r, cells=lcells, n=ln, prog_base=prog_base, jobs=jobs, tasks=tasks))
        chunks.append(dict(k0=k0, k1=k1, ptr_words=ptr_words, bnd_elems=bnd_elems, prog_words=prog_words,
                           scratch_words=scratch_words, launches=launches, ptr_off=vec(), bnd_off=vec(), scratch_off=vec()))
    p["chunks"] = chunks
    assert pos == len(v)
    return p


# ---- the geometry the plan reads (at_ptr_layout.h, at_band.h), written out ----

def rclass_of(l1):
    return max(1, min(MAXR, (l1 + 31) // 32))


def ptr_class(R, half):
    return R | (half << 4)


def ptr_pair_words(l1, l2, R, sh, jump):
    RPP = 32 * R
    stripes = (l1 + RPP - 1) // RPP
    last = (l2 + 31) | (31 if jump else (1 << sh) - 1)
    w = stripes * ((last >> sh) + 1) * RPP
    if jump:
        w += stripes * ((last >> 5) + 1) * RPP
    return w


def ptr_packed_job_words(l2, R):
    return ((((l2 + 31) | 3) >> 2) + 1) * 32 * R


def edit_bits_rows(R):
    return 1024 * R


def edit_bits_pair_words(l1, l2, R):
    rows = edit_bits_rows(R)
    return (l1 + rows - 1) // rows * ((((l2 + 63) | 15) >> 4) + 1) * rows


def band_clip(l1, l2, lo, hi):
    a, b = max(lo, 1 - l1), min(hi, l2 - 1)
    return (1, 0) if a > b else (a, b)


def band_stripe(l1, l2, elo, ehi, RPP, s, wsh=4):
    if elo > ehi:
        return None
    ia, ib = s * RPP + 1, min((s + 1) * RPP, l1)
    if ia > ib:
        return None
    a, b = max(ia + elo, 1), min(ib + ehi, l2)
    if a > b:
        return None
    t0 = (a - 1) & ~31
    return (a, b, t0, ((b + 31 - t0) >> wsh) + 1)


def band_pair_words(l1, l2, elo, ehi, RPP, wsh):
    w = 0
    for s in range((l1 + RPP - 1) // RPP):
        win = band_stripe(l1, l2, elo, ehi, RPP, s, wsh)
        if win:
            w += win[3] * RPP
    return w


def band_cells_below(l1, l2, D):
    n = 0
    a, b = max(1 - D, 1), min(l2 - D, l1)
    if a <= b:
        n += (b - a + 1) * (a + b + 2 * D) // 2
    f = max(l2 - D + 1, 1)
    if f <= l1:
        n += (l1 - f + 1) * l2
    return n


def band_cells(l1, l2, elo, ehi):
    if elo > ehi:
        return 0
    return band_cells_below(l1, l2, ehi) - band_cells_below(l1, l2, elo - 1)


# ---- the planning loop of setup_shard (at_runtime.cu) before at_plan.h, copied literally ----

def order_wave_tasks_port(t, pair_major):
    n = len(t)
    if pair_major or n == 0:
        return [(p, s, (x - 1) & 0xffffffff if s else x, 0) for x, (p, s, _, _) in enumerate(t)]      # uint32 prev
    active = []
    x = 0
    while x < n:
        y = x
        while y < n and t[y][0] == t[x][0]:
            y += 1
        active.append([t[x][0], y - x, 0, x])
        x = y
    out = []
    s = 0
    while active:
        keep = []
        for r in active:
            idx = len(out)
            out.append((r[0], t[r[3] + s][1], r[2] if s else idx, 0))
            r[2] = idx
            if s + 1 < r[1]:
                keep.append(r)
        active = keep
        s += 1
    return out


def port_plan(sh):
    n, L1, L2, mode, tb = len(sh.l1), sh.l1, sh.l2, sh.mode, sh.traceback
    jump = sh.jump
    banded = sh.band is not None
    h_band = [band_clip(L1[k], L2[k], *sh.band[k]) for k in range(n)] if banded else None
    band_affine = banded and mode == GLOBAL
    bits_path = sh.bits and tb

    def rclass(l1):
        return MAXR if band_affine else sh.bits_r if bits_path else rclass_of(l1)

    def pair_cells(k, l1, l2):
        return band_cells(l1, l2, *h_band[k]) if banded else l1 * l2

    code_sh = 4 if mode >= OVERLAP else 3

    def pair_ptr_words(k, l1, l2):
        if bits_path:
            return edit_bits_pair_words(l1, l2, sh.bits_r)
        if banded:
            return band_pair_words(l1, l2, h_band[k][0], h_band[k][1], 32 * rclass(l1), code_sh)
        return ptr_pair_words(l1, l2, rclass(l1), code_sh, jump)

    l1u, l2u = L1[0], L2[0]
    uniform = mode <= FIT and l1u <= 32 * MAXR and not band_affine and sh.allow_uniform
    for k in range(1, n):
        uniform = uniform and L1[k] == l1u and L2[k] == l2u
    cells = 0
    h_rclass = []
    if uniform:
        cells = n * l1u * l2u
    else:
        h_rclass = [0] * n
        for k in range(n):
            h_rclass[k] = ptr_class(rclass(L1[k]), 0)
            cells += pair_cells(k, L1[k], L2[k])

    def pair_words(k):
        return pair_ptr_words(k, L1[k], L2[k]) + 64 * rclass(L1[k]) if tb else 0

    need_words = n * pair_words(0) if uniform else sum(pair_words(k) for k in range(n))
    budget_words = sh.budget
    m, u, o, e = sh.prm
    maxabs = max(abs(m), abs(u), abs(o), abs(e), 1)
    p16_local = mode == LOCAL
    p16_mode = (p16_local or mode == GLOBAL or (mode == FIT and not jump)) and abs(m - u) <= 31 and \
               (p16_local or maxabs <= 31) and not sh.no_p16

    def p16_ok(l1, l2):
        return p16_mode and l1 <= 32 * MAXR and l2 <= 60000 and 8 * (l1 + l2 + 42) * maxabs < (32000 if p16_local else 24000)

    plan = dict(need_words=need_words, cells=cells, fail_pair=NONE32, fail_words=0)
    if uniform and need_words and need_words > budget_words:
        uniform = False
        h_rclass = [ptr_class(rclass_of(l1u), 0)] * n
    if uniform:
        packed = p16_ok(l1u, l2u) and n >= 2
        R = rclass_of(l1u)
        words_per_job = 0 if not tb else ptr_packed_job_words(l2u, R) if packed else pair_ptr_words(0, l1u, l2u)
        n_jobs = (n + 1) // 2 if packed else n
        ptr_words = words_per_job * n_jobs
        scratch_words = n * (l1u + l2u) if tb else 0
        launch = dict(kind=LK_PACKED if packed else LK_INT32, r=R, cells=n * l1u * l2u, n=n_jobs, prog_base=0, jobs=[], tasks=[])
        plan.update(uniform=1, u=dict(packed=int(packed), R=R, words_per_job=words_per_job, scratch_per_pair=(l1u + l2u) if tb else 0),
                    rclass=[], max_chunk_words=ptr_words, max_scratch_words=scratch_words, max_bnd_elems=0, max_prog_words=0,
                    max_pairs=n, chunks=[dict(k0=0, k1=n, ptr_words=ptr_words, bnd_elems=0, prog_words=0, scratch_words=scratch_words,
                                              launches=[launch], ptr_off=[], bnd_off=[], scratch_off=[])])
        return plan
    plan.update(uniform=0, u=None)
    max_chunk_words = max_scratch_words = 0
    chunks = []
    cur_k0, words = 0, 0
    for k in range(n):
        w = pair_words(k)
        if w > budget_words:
            plan.update(fail_pair=k, fail_words=w)
            return plan
        if words + w > budget_words and k > cur_k0:
            chunks.append([cur_k0, k])
            cur_k0, words = k, 0
        words += w
    chunks.append([cur_k0, n])
    linear = mode >= OVERLAP
    max_bnd_elems = max_prog_words = 0
    out_chunks = []

    def cells_of(k):
        return L1[k] * L2[k]

    def by_cells(v):
        ragged = any(cells_of(x) != cells_of(v[0]) for x in v[1:])
        if ragged:
            v.sort(key=lambda x: -cells_of(x))      # stable

    def new_launch():
        return dict(kind=0, r=1, cells=0, n=0, prog_base=0, jobs=[], tasks=[])

    for k0, k1 in chunks:
        c = dict(k0=k0, k1=k1, launches=[], bnd_elems=0, prog_words=0)
        nc = k1 - k0
        l32 = [new_launch() for _ in range(MAXR + 1)]
        l16 = [new_launch() for _ in range(MAXR + 1)]
        lwv = [new_launch() for _ in range(MAXR + 1)]
        lbit = [new_launch() for _ in range(MAXR + 1)]
        scalar_pairs, wave_pairs, cand = [], [], []
        for k in range(k0, k1):
            l1, l2 = L1[k], L2[k]
            if linear or band_affine or l1 > 32 * MAXR:
                wave_pairs.append(k)
            elif p16_ok(l1, l2):
                cand.append(k)
            else:
                scalar_pairs.append(k)

        def key(k):
            return ((h_rclass[k] if p16_local else L1[k]) << 32) | L2[k]
        srt = all(key(cand[x - 1]) >= key(cand[x]) for x in range(1, len(cand)))
        if not srt:
            cand.sort(key=lambda x: -key(x))
        x = 0
        while x < len(cand):
            if x + 1 < len(cand) and key(cand[x]) == key(cand[x + 1]):
                r = h_rclass[cand[x]] & 15
                l16[r]["jobs"].append((cand[x], cand[x + 1]))
                l16[r]["cells"] += cells_of(cand[x]) + cells_of(cand[x + 1])
                x += 2
            else:
                scalar_pairs.append(cand[x])
                x += 1
        by_cells(scalar_pairs)
        for k in scalar_pairs:
            r = h_rclass[k] & 15
            l32[r]["jobs"].append((k, k))
            l32[r]["cells"] += cells_of(k)
        by_cells(wave_pairs)
        h_bnd_off = [0] * nc
        for k in wave_pairs:
            l1, l2 = L1[k], L2[k]
            r = sh.bits_r if sh.bits else h_rclass[k] & 15
            rows = edit_bits_rows(r) if sh.bits else 32 * r
            lw = lbit[r] if sh.bits else lwv[r]
            n_stripes = (l1 + rows - 1) // rows
            queued = 0
            for st2 in range(n_stripes):
                if banded and st2 + 1 < n_stripes and not band_stripe(l1, l2, h_band[k][0], h_band[k][1], rows, st2):
                    continue
                lw["tasks"].append((k, st2, 0, 0))
                queued += 1
            lw["cells"] += pair_cells(k, l1, l2) if banded else cells_of(k)
            if queued > 1:
                h_bnd_off[k - k0] = c["bnd_elems"]
                c["bnd_elems"] += 2 * ((l2 + 4) & ~3)
        for r in range(1, MAXR + 1):
            if l32[r]["jobs"]:
                l32[r].update(kind=LK_INT32, r=r, n=len(l32[r]["jobs"]))
                c["launches"].append(l32[r])
            if l16[r]["jobs"]:
                l16[r].update(kind=LK_PACKED, r=r, n=len(l16[r]["jobs"]))
                c["launches"].append(l16[r])
            lwv[r]["tasks"] = order_wave_tasks_port(lwv[r]["tasks"], sh.pair_major)
            lbit[r]["tasks"] = order_wave_tasks_port(lbit[r]["tasks"], sh.pair_major)
            for lw, kind in ((lwv[r], LK_WAVE), (lbit[r], LK_BITS)):
                if lw["tasks"]:
                    lw.update(kind=kind, r=r, n=len(lw["tasks"]), prog_base=c["prog_words"])
                    c["prog_words"] += len(lw["tasks"])
                    c["launches"].append(lw)
        max_bnd_elems = max(max_bnd_elems, c["bnd_elems"])
        max_prog_words = max(max_prog_words, c["prog_words"])
        h_ptr_off = [0] * nc
        words = 0
        if tb:
            for lch in c["launches"]:
                if lch["kind"] == LK_PACKED:
                    for a, b in lch["jobs"]:
                        h_ptr_off[a - k0] = words
                        h_ptr_off[b - k0] = words
                        h_rclass[a] = ptr_class(lch["r"], 1)
                        h_rclass[b] = ptr_class(lch["r"], 2)
                        words += ptr_packed_job_words(L2[a], lch["r"])
                elif lch["kind"] == LK_INT32:
                    for a, _ in lch["jobs"]:
                        h_ptr_off[a - k0] = words
                        words += pair_ptr_words(a, L1[a], L2[a])
                else:
                    placed = [0] * nc
                    for tk in lch["tasks"]:
                        k = tk[0]
                        if placed[k - k0]:
                            continue
                        placed[k - k0] = 1
                        h_ptr_off[k - k0] = words
                        words += pair_ptr_words(k, L1[k], L2[k])
        c["ptr_words"] = words
        max_chunk_words = max(max_chunk_words, words)
        c["ptr_off"], c["bnd_off"] = h_ptr_off, h_bnd_off
        c["scratch_off"], c["scratch_words"] = [], 0
        if tb:
            sw = 0
            for k in range(nc):
                c["scratch_off"].append(sw)
                sw += L1[k0 + k] + L2[k0 + k]
            c["scratch_words"] = sw
            max_scratch_words = max(max_scratch_words, sw)
        out_chunks.append(c)
    plan.update(rclass=h_rclass, chunks=out_chunks, max_chunk_words=max_chunk_words, max_scratch_words=max_scratch_words,
                max_bnd_elems=max_bnd_elems, max_prog_words=max_prog_words, max_pairs=max(k1 - k0 for k0, k1 in chunks))
    return plan


# ---- seeded random shards ----

def random_shard(rng):
    kind = rng.choice(["ragged", "ragged", "long", "uniform", "banded", "bits"])
    mode = rng.choice([GLOBAL, LOCAL, FIT, OVERLAP, EDIT])
    n = rng.randint(1, 24)
    kw = dict(traceback=rng.random() < 0.7, pair_major=rng.random() < 0.2, no_p16=rng.random() < 0.2,
              prm=rng.choice([(1, -2, -5, -1), (1, -4, -6, -1), (2, -3, -5, -2), (5, -4, -10, -1), (1, -40, -5, -1), (1, 1, -1, -1)]))
    if kind == "uniform":
        mode = rng.choice([GLOBAL, LOCAL, FIT])
        l1, l2 = rng.randint(1, 256), rng.randint(1, 700)
        L1, L2 = [l1] * n, [l2] * n
    elif kind == "bits":
        mode = EDIT
        L1 = [rng.choice([rng.randint(1, 300), rng.randint(300, 9000)]) for _ in range(n)]
        L2 = [rng.randint(1, 2000) for _ in range(n)]
        kw.update(bits=True, bits_r=rng.choice([1, 2, 4]))
    else:
        hi1 = 256 if kind == "ragged" else 3000
        L1 = [rng.choice([rng.randint(1, 40), rng.randint(1, hi1), 32 * rng.randint(1, 8), 32 * rng.randint(1, 8) + 1]) for _ in range(n)]
        L2 = [rng.choice([rng.randint(1, 60), rng.randint(1, 1500)]) for _ in range(n)]
        if rng.random() < 0.3:      # a few shapes repeated: packed partners
            L1 = [L1[rng.randrange(min(3, n))] for _ in range(n)]
            L2 = [L2[rng.randrange(min(3, n))] for _ in range(n)]
    if kind == "banded":
        mode = rng.choice([OVERLAP, GLOBAL])
        band = []
        for k in range(n):
            d = L2[k] - L1[k]
            if mode == GLOBAL:
                band.append((min(0, d) - rng.randint(0, 300), max(0, d) + rng.randint(0, 300)))
            else:
                lo = rng.randint(-L1[k] - 50, L2[k] + 50)
                band.append((lo, lo + rng.choice([-1, 0, rng.randint(0, 100), rng.randint(0, 4000)])) if rng.random() < 0.9 else (lo, lo - 5))
                if band[-1][0] > band[-1][1]:
                    band[-1] = (band[-1][0], band[-1][0])      # the runtime rejects lo > hi; an empty band comes from clipping
        kw["band"] = band
    if mode == FIT:
        L2 = [max(a, b, 2) for a, b in zip(L1, L2)]
        kw["jump"] = rng.random() < 0.4
    s = Shard(L1, L2, mode, **kw)
    if rng.random() < 0.35:      # a budget that cuts the shard into many chunks
        w = [x for x in pair_words_of(s)]
        if max(w):
            s.budget = rng.randint(max(w), max(max(w), sum(w) // rng.randint(1, 6)))
    elif rng.random() < 0.05:
        s.budget = 1
    return s


def pair_words_of(s):
    """arena words of every pair, from the port's own plan inputs"""
    saved, s.budget = s.budget, U64MAX
    p = port_plan(s)
    s.budget = saved
    if not s.traceback:
        return [0]
    n = len(s.l1)
    out = []
    for k in range(n):
        one = Shard([s.l1[k]], [s.l2[k]], s.mode, traceback=True, jump=s.jump, band=None if s.band is None else [s.band[k]],
                    bits=s.bits, bits_r=s.bits_r, prm=s.prm, no_p16=True, allow_uniform=False)
        out.append(port_plan(one)["need_words"])
    del p
    return out


def diff(a, b, path="plan"):
    if isinstance(a, dict) and isinstance(b, dict):
        for k in a:
            if k not in b:
                return f"{path}.{k} missing"
            d = diff(a[k], b[k], f"{path}.{k}")
            if d:
                return d
        return None
    if isinstance(a, list) and isinstance(b, list):
        if len(a) != len(b):
            return f"{path}: length {len(a)} != {len(b)}"
        for i, (x, y) in enumerate(zip(a, b)):
            d = diff(x, y, f"{path}[{i}]")
            if d:
                return d
        return None
    return None if a == b else f"{path}: {a} != {b}"


def compare(L, s):
    c, p = c_plan(L, s), port_plan(s)
    assert c["need_words"] == p["need_words"], (s, c["need_words"], p["need_words"])
    if p["fail_pair"] != NONE32:
        assert (c["fail_pair"], c["fail_words"]) == (p["fail_pair"], p["fail_words"]), s
        return c
    d = diff(p, c)
    assert d is None, (d, s)
    return c


def check_invariants(s, p):
    n = len(s.l1)
    if p["fail_pair"] != NONE32:
        return
    assert p["chunks"][0]["k0"] == 0 and p["chunks"][-1]["k1"] == n
    for a, b in zip(p["chunks"], p["chunks"][1:]):
        assert a["k1"] == b["k0"] and a["k0"] < a["k1"]
    if p["uniform"]:
        return
    rcl = p["rclass"]
    for c in p["chunks"]:
        k0, k1 = c["k0"], c["k1"]
        nc = k1 - k0
        seen = {}
        blocks = {}
        prog = 0
        for li, l in enumerate(c["launches"]):
            if l["kind"] >= LK_WAVE:
                assert l["n"] == len(l["tasks"]) and l["prog_base"] == prog
                prog += l["n"]
                pos = {}
                for x, (pair, stripe, prev, _) in enumerate(l["tasks"]):
                    assert k0 <= pair < k1
                    if pair in pos:      # the pair's stripe queued before this one, earlier in the queue
                        assert prev == pos[pair][0] and prev < x and l["tasks"][prev][1] < stripe, (s, l["tasks"])
                    else:
                        assert prev == x or (s.pair_major and stripe > 0)
                        assert seen.setdefault(pair, li) == li
                    pos[pair] = (x, stripe)
                    if s.traceback:
                        assert rcl[pair] == ptr_class(l["r"], 0)
                for pair in pos:
                    if s.traceback and pair not in blocks:
                        blocks[pair] = (c["ptr_off"][pair - k0], None)
            else:
                assert l["n"] == len(l["jobs"])
                for a, b in l["jobs"]:
                    for q in {a, b}:
                        assert k0 <= q < k1 and q not in seen
                        seen[q] = li
                    if l["kind"] == LK_PACKED:
                        assert a != b and c["ptr_off"][a - k0] == c["ptr_off"][b - k0]
                        if s.traceback:
                            assert (rcl[a], rcl[b]) == (ptr_class(l["r"], 1), ptr_class(l["r"], 2))
                            blocks[a] = (c["ptr_off"][a - k0], ptr_packed_job_words(s.l2[a], l["r"]))
                    else:
                        assert a == b
                        if s.traceback:
                            assert rcl[a] == ptr_class(l["r"], 0)
                            blocks[a] = (c["ptr_off"][a - k0], None)
        assert sorted(seen) == list(range(k0, k1)), s
        assert c["prog_words"] == prog
        # pointer blocks: disjoint, inside ptr_words, within budget unless the chunk is one pair
        if s.traceback:
            spans = []
            for pair, (off, words) in blocks.items():
                if words is None:      # the block's size: the distance to the next block, or to the end
                    words = single_words(s, pair)
                spans.append((off, off + words))
            spans.sort()
            for (a0, a1), (b0, b1) in zip(spans, spans[1:]):
                assert a1 <= b0, s
            assert spans[-1][1] <= c["ptr_words"] == sum(e - b for b, e in spans)
            assert c["ptr_words"] <= s.budget or nc == 1
            assert c["scratch_off"] == list(np.cumsum([0] + [s.l1[k] + s.l2[k] for k in range(k0, k1)])[:-1])
        # boundary slabs of the pairs with more than one task
        slabs = []
        for l in c["launches"]:
            if l["kind"] >= LK_WAVE:
                cnt = {}
                for t in l["tasks"]:
                    cnt[t[0]] = cnt.get(t[0], 0) + 1
                for pair, m in cnt.items():
                    if m > 1:
                        off = c["bnd_off"][pair - k0]
                        slabs.append((off, off + 2 * ((s.l2[pair] + 4) & ~3)))
                    else:
                        assert c["bnd_off"][pair - k0] == 0
        slabs.sort()
        for (a0, a1), (b0, b1) in zip(slabs, slabs[1:]):
            assert a1 <= b0
        assert (slabs[-1][1] if slabs else 0) <= c["bnd_elems"]


def single_words(s, k):
    one = Shard([s.l1[k]], [s.l2[k]], s.mode, traceback=True, jump=s.jump, band=None if s.band is None else [s.band[k]],
                bits=s.bits, bits_r=s.bits_r, prm=s.prm, no_p16=True, allow_uniform=False)
    return port_plan(one)["max_chunk_words"]


# ---- tests ----

def test_plan_equals_port_and_keeps_invariants(lib):
    rng = random.Random(20261022)
    kinds = set()
    for _ in range(3000):
        s = random_shard(rng)
        p = compare(lib, s)
        check_invariants(s, p)
        kinds.add((s.mode, s.traceback, s.band is not None, s.bits, p["uniform"], len(p["chunks"]) > 2))
    # the sweep reached every mode with and without traceback, banded, bit-parallel, uniform and many-chunk plans
    assert {m for m, *_ in kinds} == set(range(5))
    assert any(k[2] and k[0] == GLOBAL for k in kinds) and any(k[2] and k[0] == OVERLAP for k in kinds)
    assert any(k[3] for k in kinds) and any(k[4] for k in kinds) and any(k[5] for k in kinds)


@pytest.mark.parametrize("mode", [GLOBAL, LOCAL, FIT])
def test_uniform_shards(lib, mode):
    """even and odd uniform shards, packed and unpacked, within and over budget"""
    for n in (1, 2, 3, 8, 9, 64):
        for l1, l2 in ((1, 1), (31, 40), (150, 500), (256, 257), (100, 3000)):
            for no_p16 in (False, True):
                for tb in (False, True):
                    s = Shard([l1] * n, [max(l1, l2)] * n, mode, traceback=tb, no_p16=no_p16)
                    p = compare(lib, s)
                    check_invariants(s, p)
                    assert p["uniform"] == 1
                    if tb and n > 2:
                        s.budget = p["need_words"] // n * 2      # over budget: the general plan, two pairs per chunk
                        p = compare(lib, s)
                        assert not p["uniform"] and len(p["chunks"]) == (n + 1) // 2
                        check_invariants(s, p)


@pytest.mark.parametrize("mode", [GLOBAL, LOCAL, FIT])
def test_uniform_closed_form_matches_general_plan(lib, mode):
    """uniform_pair (what at_plan_uniform writes) against the general plan of the same even shard"""
    out = np.zeros(7, np.uint64)
    packed_seen = set()
    for n in (2, 8, 64):
        for l1, l2 in ((31, 40), (150, 500), (256, 257)):
            for no_p16 in (False, True):
                s = Shard([l1] * n, [l2] * n, mode, traceback=True, no_p16=no_p16)
                u = c_plan(lib, s)
                s.allow_uniform = False
                g = c_plan(lib, s)
                assert u["uniform"] and not g["uniform"] and len(g["chunks"]) == 1
                uc, gc = u["chunks"][0], g["chunks"][0]
                packed_seen.add(u["u"]["packed"])
                (ul,), (gl,) = uc["launches"], gc["launches"]
                assert (ul["kind"], ul["r"], ul["cells"], ul["n"]) == (gl["kind"], gl["r"], gl["cells"], gl["n"])
                assert (uc["ptr_words"], uc["scratch_words"]) == (gc["ptr_words"], gc["scratch_words"])
                assert u["cells"] == g["cells"] and u["need_words"] == g["need_words"]
                jobs = [None] * ul["n"]
                for k in range(n):
                    q = u["u"]
                    lib.plan_model_uniform_pair(q["packed"], q["R"], q["words_per_job"], q["scratch_per_pair"], n, k, out.ctypes.data)
                    ptr_off, scratch_off, rcl, writes, job, a, b = (int(x) for x in out)
                    assert (ptr_off, scratch_off, rcl) == (gc["ptr_off"][k], gc["scratch_off"][k], g["rclass"][k]), (s, k)
                    if writes:
                        jobs[job] = (a, b)
                assert jobs == gl["jobs"]
    assert packed_seen == {0, 1}


def test_uniform_odd_shard_ends_in_a_lone_packed_job(lib):
    out = np.zeros(7, np.uint64)
    n = 5
    s = Shard([150] * n, [500] * n, LOCAL, traceback=True)
    p = c_plan(lib, s)
    q = p["u"]
    assert q["packed"] and p["chunks"][0]["launches"][0]["n"] == 3
    lib.plan_model_uniform_pair(q["packed"], q["R"], q["words_per_job"], q["scratch_per_pair"], n, n - 1, out.ctypes.data)
    ptr_off, _, rcl, writes, job, a, b = (int(x) for x in out)
    assert writes and job == 2 and (a, b) == (4, 4) and ptr_off == 2 * q["words_per_job"] and rcl == ptr_class(q["R"], 1)
    s.allow_uniform = False      # the general plan runs the odd pair out on int32 lanes
    g = c_plan(lib, s)
    kinds = [(l["kind"], l["jobs"]) for l in g["chunks"][0]["launches"]]
    assert kinds == [(LK_INT32, [(4, 4)]), (LK_PACKED, [(0, 1), (2, 3)])]


def test_single_pair_over_budget_fails(lib):
    s = Shard([100, 3000, 50], [500, 2000, 60], GLOBAL, traceback=True)
    w = pair_words_of(s)
    s.budget = w[1] - 1
    p = compare(lib, s)
    assert (p["fail_pair"], p["fail_words"]) == (1, w[1])


def test_bits_r(lib):
    def port(l1, slots):
        for r in (4, 2):
            if sum((x + 1024 * r - 1) // (1024 * r) for x in l1) >= 2 * slots:
                return r
        return 1
    rng = random.Random(5)
    for _ in range(300):
        l1 = np.array([rng.randint(1, 50000) for _ in range(rng.randint(1, 200))], np.uint32)
        slots = rng.choice([1, 10, 148 * 8 * 4, 100000])
        assert lib.plan_model_bits_r(l1.ctypes.data, len(l1), slots) == port([int(x) for x in l1], slots)


def cut_by_cells_port(cells, lo, hi, parts):
    """at_runtime.cu cut_by_cells, copied literally"""
    cut = [lo] * (parts + 1)
    cut[parts] = hi
    if parts <= 1:
        return cut
    total = sum(cells[lo:hi])
    acc, d = 0, 1
    k = lo
    while k < hi and d < parts:
        acc += cells[k]
        while d < parts and acc * parts >= total * d:
            cut[d] = k + 1
            d += 1
        k += 1
    while d < parts:
        cut[d] = hi
        d += 1
    cut[parts] = hi
    return cut


def test_cut_by_prefix_matches_cut_by_cells(lib):
    rng = random.Random(11)
    for it in range(20000):
        n = rng.randint(0, 40)
        cells = [rng.choice([0, 0, 1, rng.randint(0, 50), rng.randint(0, 1 << 40)]) for _ in range(n)]
        if rng.random() < 0.1:
            cells = [0] * n
        prefix = np.zeros(n + 1, np.uint64)
        prefix[1:] = np.cumsum(np.array(cells, np.uint64), dtype=np.uint64)
        lo = rng.randint(0, n)
        hi = rng.randint(lo, n)
        parts = rng.choice([1, 2, 3, rng.randint(1, 10), rng.randint(1, 100)])
        got = np.zeros(parts + 1, np.uint64)
        lib.plan_model_cut(prefix.ctypes.data, n, lo, hi, parts, got.ctypes.data)
        assert [int(x) for x in got] == cut_by_cells_port(cells, lo, hi, parts), (cells, lo, hi, parts)
