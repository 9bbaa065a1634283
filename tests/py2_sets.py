"""Random down-sampling draws for comparing smc_py2rand.h (host harness and device) with smcounter_b200/downsample.py:
barcode sets of 1 to 120 000 distinct keys in insertion order, 2-bit codes of 0 to 31 nt mixed with dictionary-coded
barcodes (top bit set), real 1-based positions as seeds, and k at the edges of random.sample's two branches."""
from __future__ import annotations

import numpy as np

from smcounter_b200.downsample import py2_dict_key_order, py2_seeded_sample, py2_string_hash
from smcounter_b200.soa import umi_code, umi_string

SIZES_LARGE = (50001, 60000, 120000)        # beyond 50 000 keys a dict grows x2 instead of x4


def _barcodes(rng, n, names, table):
    """n distinct barcodes: (codes, strings)."""
    seen, codes, strs = set(), [], []
    while len(codes) < n:
        r = rng.random()
        if r < 0.03:                                               # not ACGT or longer than 31 nt: dictionary code
            s = "".join(rng.choice(list("ACGTN"), size=int(rng.integers(1, 40))))
            if "N" not in s and len(s) <= 31:
                s += "N"
        elif r < 0.06:
            s = "".join(rng.choice(list("ACGT"), size=int(rng.integers(0, 9))))
        else:
            s = "".join(rng.choice(list("ACGT"), size=int(rng.integers(9, 32))))
        if s in seen:
            continue
        seen.add(s)
        c = umi_code(s, table)
        if c >> 63:
            names[c] = s
        codes.append(c)
        strs.append(s)
    return codes, strs


def make_sets(seed: int = 7, n_small: int = 2000, n_medium: int = 24, large: bool = True):
    """[(codes, strings, pos1, k)] and the {code: string} table of the dictionary-coded barcodes."""
    rng = np.random.default_rng(seed)
    names, table = {}, {}
    sizes = [int(rng.integers(1, 400)) for _ in range(n_small)] + [int(rng.integers(400, 9000)) for _ in range(n_medium)]
    if large:
        sizes += list(SIZES_LARGE)
    sets = []
    for t, n in enumerate(sizes):
        codes, strs = _barcodes(rng, n, names, table)
        choice = t % 7
        k = (0, 1, 5, 6, n - 1, n, int(rng.integers(0, n + 1)))[choice]
        k = min(max(k, 0), n)
        pos1 = int(rng.integers(1, 250_000_000))
        sets.append((codes, strs, pos1, k))
    return sets, names


def reference_draw(strs, pos1, k):
    """downsample.py's draw as insertion indices."""
    index = {s: i for i, s in enumerate(strs)}
    return [index[s] for s in py2_seeded_sample(str(pos1), py2_dict_key_order(strs), k)]


def hashes_of(strs):
    return np.asarray([py2_string_hash(s) for s in strs], dtype=np.int64)


def code_hash(code: int, names) -> int:
    return py2_string_hash(umi_string(code, names))
