"""Instance helpers for tests and benchmarks: the synthetic generator of SURVEY.md §8(c), a small TSPLIB
NODE_COORD_SECTION reader that mirrors the reference parser's tokenisation (reference
src/utility.c:351-453: separators " :\\n\\t\\r", atoi/atof, 1-based ids), and tour conversions."""
from __future__ import annotations

import random

import numpy as np

WEIGHT_TYPES = {"EUC_2D": 0, "MAX_2D": 1, "MAN_2D": 2, "CEIL_2D": 3, "GEO": 4, "ATT": 5}


def uniform_instance(n: int, seed: int | None = None, hi: int = 10000) -> np.ndarray:
    """uni<n>: rng = random.Random(n); x then y drawn with randint(0, hi) per node; EUC_2D.
    The range mirrors the reference's generator cap (other_codes/generate_tsp_istances.py:3-4,26-27)."""
    rng = random.Random(n if seed is None else seed)
    xy = np.empty((n, 2), dtype=np.float64)
    for i in range(n):
        xy[i, 0] = rng.randint(0, hi)
        xy[i, 1] = rng.randint(0, hi)
    return xy


def read_tsplib(path: str):
    """Returns (xy, weight_type). Unknown / missing EDGE_WEIGHT_TYPE -> -1 (the reference then falls back
    to EUC_2D in calc_dist, src/distutil.c:91)."""
    import re
    n, wt, xy, section = -1, -1, None, 0
    with open(path) as f:
        for line in f:
            if len(line) <= 1:
                continue
            tok = [t for t in re.split(r"[ :\n\t\r]+", line) if t]
            if not tok:
                continue
            key = tok[0]
            if key.startswith("NAME") or key.startswith("COMMENT") or key.startswith("TYPE"):
                section = 0
            elif key.startswith("DIMENSION"):
                n = int(tok[1]); xy = np.zeros((n, 2), dtype=np.float64); section = 0
            elif key.startswith("EOF"):
                break
            elif key.startswith("EDGE_WEIGHT_TYPE"):
                for name, val in WEIGHT_TYPES.items():
                    if tok[1].startswith(name):
                        wt = val
                if tok[1].startswith("EXPLICIT"):
                    raise ValueError("EXPLICIT instances are rejected by the reference parser (utility.c:418)")
                section = 0
            elif key.startswith("NODE_COORD_SECTION"):
                section = 1
            elif key.startswith("EDGE_WEIGHT_SECTION"):
                section = 2
            elif section == 1:
                i = int(key) - 1
                xy[i] = (float(tok[1]), float(tok[2]))
    return xy, wt


def order_to_succ(order) -> np.ndarray:
    order = np.asarray(order, dtype=np.int32)
    succ = np.empty_like(order)
    succ[order] = np.roll(order, -1)
    return succ


def succ_to_order(succ, start: int = 0) -> np.ndarray:
    succ = np.asarray(succ)
    out = np.empty(len(succ), dtype=np.int32)
    at = start
    for p in range(len(succ)):
        out[p] = at
        at = succ[at]
    return out


def random_tours(n: int, batch: int, seed: int) -> np.ndarray:
    """`batch` random Hamiltonian cycles as successor arrays (GA-style random population)."""
    rng = np.random.default_rng(seed)
    out = np.empty((batch, n), dtype=np.int32)
    for b in range(batch):
        out[b] = order_to_succ(rng.permutation(n).astype(np.int32))
    return out


def is_tour(succ) -> bool:
    succ = np.asarray(succ)
    n = len(succ)
    seen = np.zeros(n, dtype=bool)
    at = 0
    for _ in range(n):
        if at < 0 or at >= n or seen[at]:
            return False
        seen[at] = True
        at = succ[at]
    return at == 0


class GlibcRandom:
    """glibc's random() / srandom() (TYPE_3 additive feedback generator, r[i] = r[i-3] + r[i-31]) restated, so that
    populations can be generated exactly like the reference does (reference include/utility.h:36 URAND() =
    random() / RAND_MAX, src/utility.c:752-754 rand_choice) without touching the process-wide libc state.
    tests/test_host_logic.py checks it against libc itself."""

    RAND_MAX = 2147483647

    def __init__(self, seed: int):
        seed = seed & 0xFFFFFFFF
        if seed == 0:
            seed = 1
        r = [0] * 34
        r[0] = seed
        for i in range(1, 31):
            # 16807 * r[i-1] % 2147483647 on the signed 32-bit value, as glibc computes it (Schrage)
            prev = r[i - 1] if r[i - 1] < 0x80000000 else r[i - 1] - 0x100000000
            hi, lo = int(prev / 127773), int(prev - 127773 * int(prev / 127773))
            word = 16807 * lo - 2836 * hi
            if word < 0:
                word += 2147483647
            r[i] = word & 0xFFFFFFFF
        for i in range(31, 34):
            r[i] = r[i - 31]
        self._r = r
        for _ in range(310):
            self._step()

    def _step(self) -> int:
        r = self._r
        v = (r[-31] + r[-3]) & 0xFFFFFFFF
        r.append(v)
        del r[0]
        return v

    def random(self) -> int:
        return self._step() >> 1

    def urand(self) -> float:
        return self.random() / 2147483647.0

    def rand_choice(self, lo: int, hi: int) -> int:
        return lo + int(self.urand() * (hi - lo))


def vns_kick_indices(g: GlibcRandom, n: int):
    """The three tour indices of one kick() of the reference's VNS, drawn from `g` like src/vns.c:25-31 (the loop of
    examples/vns_resident.c): idx1, then idx2 until it is neither idx1 nor next to it, then idx3 likewise."""
    i1 = g.rand_choice(0, n)
    i2 = i3 = i1
    while i2 == i1 or abs(i1 - i2) <= 1:
        i2 = g.rand_choice(0, n)
    while i3 == i1 or i3 == i2 or abs(i1 - i3) <= 1 or abs(i2 - i3) <= 1:
        i3 = g.rand_choice(0, n)
    return i1, i2, i3


def reference_random_population(n: int, batch: int, seed: int) -> np.ndarray:
    """`batch` chromosomes generated exactly like reference src/genetic.c:349-364 random_generation(): identity, then n
    random transpositions (idx1, idx2 drawn with rand_choice(0, n) in that order), one generator stream (srandom(seed),
    reference src/solver.c:264) for the whole population.  Returns visiting orders [batch, n]."""
    g = GlibcRandom(seed)
    draws = np.empty(2 * n * batch, dtype=np.int64)
    r = g._r
    out = draws
    for k in range(len(out)):  # the recurrence has lag 3: a plain loop (about a second for 1024 x 1000)
        v = (r[-31] + r[-3]) & 0xFFFFFFFF
        r.append(v)
        del r[0]
        out[k] = v >> 1
    idx = ((draws / 2147483647.0) * n).astype(np.int64)
    pop = np.empty((batch, n), dtype=np.int32)
    p = 0
    for b in range(batch):
        c = list(range(n))
        for _ in range(n):
            i1, i2 = idx[p], idx[p + 1]
            p += 2
            c[i1], c[i2] = c[i2], c[i1]
        pop[b] = c
    return pop


def apply_moves(succ0, moves) -> np.ndarray:
    """Applies 2-opt moves (i, j[, delta]) to a successor array exactly as the reference does (src/tabusearch.c:161-165,
    src/heuristics.c:476-483): a = i, b = j, succ[a] = b, succ[a1] = b1, forward path a1..b reversed.  Host-side helper for
    checking a downloaded tour against a committed move log (bench.py)."""
    succ0 = np.asarray(succ0, dtype=np.int32)
    n = len(succ0)
    order = succ_to_order_fast(succ0)
    pos = np.empty(n, dtype=np.int64)
    pos[order] = np.arange(n)
    for mv in moves:
        a, b = int(mv[0]), int(mv[1])
        pa, pb = int(pos[a]), int(pos[b])
        s = (pa + 1) % n
        length = (pb - pa) % n
        if length <= 1:
            continue
        if s + length <= n:
            seg = order[s:s + length][::-1].copy()
            order[s:s + length] = seg
            pos[seg] = np.arange(s, s + length)
        else:
            idx = (s + np.arange(length)) % n
            seg = order[idx][::-1].copy()
            order[idx] = seg
            pos[seg] = idx
    return order_to_succ(order)


def succ_to_order_fast(succ) -> np.ndarray:
    """succ_to_order from node 0 with list arithmetic (the numpy scalar loop is ~10x slower at n = 100 000)."""
    s = np.asarray(succ).tolist()
    out = [0] * len(s)
    at = 0
    for p in range(len(s)):
        out[p] = at
        at = s[at]
    return np.asarray(out, dtype=np.int32)
