"""The shanten and agari lookup tables are generated from first principles (tools/gen_shanten_tables.cc,
tools/gen_agari_table.py); this pins the generators. libriichi's own data files are held in tests/golden/ref_tables.json
as a digest of their whole content plus a sample of rows (written by tools/extract_ref_fixtures.py)."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
with open(os.path.join(ROOT, "tests", "golden", "ref_tables.json")) as _f:
    REF_TABLES = json.load(_f)


@pytest.fixture(scope="module")
def generated():
    import build_tables

    return build_tables.generate_shanten_tables()


def nibbles(row5):
    out = []
    for b in row5:
        out += [b & 15, b >> 4]
    return out


def test_generated_rows_known_answers(generated):
    suhai = np.frombuffer(generated["shanten_suhai.bin"], dtype=np.uint8).reshape(-1, 5)
    jihai = np.frombuffer(generated["shanten_jihai.bin"], dtype=np.uint8).reshape(-1, 5)
    assert suhai.shape[0] == 1_940_777 and jihai.shape[0] == 78_032
    # empty suit: m melds cost 3m tiles, a pair 2 more (max nibble 14)
    assert nibbles(suhai[0]) == [0, 3, 6, 9, 12, 2, 5, 8, 11, 14]
    assert nibbles(jihai[0]) == [0, 3, 6, 9, 12, 2, 5, 8, 11, 14]
    idx = lambda counts: int(sum(c * 5 ** (len(counts) - 1 - i) for i, c in enumerate(counts)))
    # 123 456 789: three complete runs; a pair beside two runs borrows one tile, beside all three it needs two new ones
    assert nibbles(suhai[idx([1] * 9)]) == [0, 0, 0, 0, 3, 1, 1, 1, 2, 5]
    # 1112345678999 (the nine-gates shape): four melds + pair missing exactly one tile
    assert nibbles(suhai[idx([3, 1, 1, 1, 1, 1, 1, 1, 3])])[9] == 1
    # honours: a triplet is a meld, a pair is a pair, singles only save one tile each
    assert nibbles(jihai[idx([3, 2, 1, 0, 0, 0, 0])]) == [0, 0, 1, 3, 6, 0, 0, 2, 5, 8]


def test_generated_tables_equal_reference_data(generated):
    for name in ("shanten_suhai.bin", "shanten_jihai.bin"):
        ref, raw = REF_TABLES[name], generated[name]
        rows = np.frombuffer(raw, dtype=np.uint8).reshape(-1, 5)
        for i, want in ref["sample_rows"].items():
            assert rows[int(i)].tobytes().hex() == want, (name, i)
        assert len(raw) == ref["bytes"] and hashlib.sha256(raw).hexdigest() == ref["sha256"], name


def test_installed_tables_are_the_generated_ones(generated):
    for name in ("shanten_suhai.bin", "shanten_jihai.bin"):
        with open(os.path.join(ROOT, "mortal_b200", "data", name), "rb") as f:
            assert f.read() == generated[name], name


@pytest.fixture(scope="module")
def agari_table():
    import gen_agari_table

    return gen_agari_table.generate()


def test_agari_table_known_answers(agari_table):
    import gen_agari_table as g

    assert len(agari_table) == 9_362
    # 123 456 789 + 123 + 11-pair in another suit: one split, four runs, straight flag, pair is the last kind
    key = g.shape_key([[1] * 9, [1, 1, 1], [2]])
    (div,) = agari_table[key]
    assert div & 7 == 0 and (div >> 3) & 7 == 4 and (div >> 6) & 15 == 12 and div & g.F_ITTSUU
    # seven separate pairs: the seven-pairs flag alone; 11223344556677: three splits with two double runs each, no seven-pairs flag
    assert agari_table[g.shape_key([[2]] * 7)] == [g.F_CHITOI]
    divs = agari_table[g.shape_key([[2] * 7])]
    assert len(divs) == 3 and all(d & g.F_RYANPEIKOU and not d & g.F_CHITOI for d in divs)
    # nine gates on its 9th tile: 1112345678999 + 5
    assert all(d & g.F_CHUUREN for d in agari_table[g.shape_key([[3, 1, 1, 1, 2, 1, 1, 1, 3]])])
    # 45556 (five concealed tiles beside three called melds): the one split is the pair 55 + the run 456
    assert agari_table[g.shape_key([[1, 3, 1]])] == [0 | 1 << 3 | 1 << 6 | 0 << 10]
    # 111222333444 + pair: {four triplets} and {123 123 123 + 444}; the table never lists {111 + 234 234 234}
    divs = agari_table[g.shape_key([[3, 3, 3, 3], [2]])]
    assert [(d & 7, (d >> 3) & 7) for d in divs] == [(4, 0), (1, 3)] and (divs[1] >> 10) & 15 == 3
    # every div decodes to as many melds as the hand holds
    for key, divs in agari_table.items():
        for d in divs:
            if d & g.F_CHITOI:
                continue
            assert (d & 7) + ((d >> 3) & 7) <= 4


def test_agari_table_equals_reference_data(agari_table):
    from extract_ref_fixtures import agari_digest

    # key -> ordered list of divs; the record order of the file is not content (agari.rs:22-51)
    ref = REF_TABLES["agari.bin"]
    for key, divs in ref["sample"].items():
        assert agari_table.get(int(key, 16)) == divs, key
    assert len(agari_table) == ref["keys"] and agari_digest(agari_table) == ref["sha256"]


def test_installed_agari_table_is_the_generated_one(agari_table):
    import gen_agari_table as g

    with open(os.path.join(ROOT, "mortal_b200", "data", "agari.bin"), "rb") as f:
        assert f.read() == g.serialize(agari_table)


def _decode_shape(key: int):
    """inverse of gen_agari_table.shape_key: a kind is a run of r one-bits from its position (count = r // 2 + 1, r odd = the
    block ends here), the next kind starts r + 1 bits further"""
    blocks, cur, b, top = [], [], 0, key.bit_length()
    while b < top:
        r = 0
        while (key >> (b + r)) & 1:
            r += 1
        cur.append(r // 2 + 1)
        if r & 1:
            blocks.append(cur)
            cur = []
        b += r + 1
    assert not cur
    return blocks


def test_agari_table_every_split_rebuilds_its_shape(agari_table):
    """Reference-independent: the key decodes to a shape of 3n+2 tiles, and pair + triplets + runs of every listed split
    add up to exactly that shape (runs stay inside one block)."""
    import gen_agari_table as g

    for key, divs in agari_table.items():
        blocks = _decode_shape(key)
        assert g.shape_key(blocks) == key
        counts = [c for b in blocks for c in b]
        block_of = [i for i, b in enumerate(blocks) for _ in b]
        assert sum(counts) in (2, 5, 8, 11, 14) and max(counts) <= 4 and len(counts) <= 14
        assert len(set(divs)) == len(divs)
        for d in divs:
            if d & g.F_CHITOI:
                assert counts == [2] * 7 and d == g.F_CHITOI
                continue
            nk, ns, pair = d & 7, (d >> 3) & 7, (d >> 6) & 15
            idx = [(d >> (10 + 4 * j)) & 15 for j in range(nk + ns)]
            rebuilt = [0] * len(counts)
            rebuilt[pair] += 2
            for i in idx[:nk]:
                rebuilt[i] += 3
            for i in idx[nk:]:
                assert block_of[i] == block_of[i + 2]
                for j in range(3):
                    rebuilt[i + j] += 1
            assert rebuilt == counts, (hex(key), hex(d))
            assert 3 * (nk + ns) + 2 == sum(counts)


def _hand_blocks(counts34):
    """the shape of a concrete hand: runs of adjacent kinds inside a suit, every honour its own block (agari.rs:767-838)"""
    blocks = []
    for lo, hi in ((0, 9), (9, 18), (18, 27)):
        run = []
        for c in list(counts34[lo:hi]) + [0]:
            if c:
                run.append(c)
            elif run:
                blocks.append(run)
                run = []
    blocks += [[c] for c in counts34[27:] if c]
    return blocks


def _splits_into_melds(counts34, need_pair):
    c = list(counts34)

    def rec(i, pair_left):
        while i < 34 and c[i] == 0:
            i += 1
        if i == 34:
            return not pair_left
        ok = False
        if c[i] >= 3:
            c[i] -= 3
            ok = rec(i, pair_left)
            c[i] += 3
        if not ok and pair_left and c[i] >= 2:
            c[i] -= 2
            ok = rec(i, False)
            c[i] += 2
        if not ok and i < 27 and i % 9 <= 6 and c[i + 1] and c[i + 2]:
            for j in range(3):
                c[i + j] -= 1
            ok = rec(i, pair_left)
            for j in range(3):
                c[i + j] += 1
        return ok

    return rec(0, need_pair)


def test_agari_table_membership_equals_brute_force_on_random_hands(agari_table):
    """Completeness, reference-independent: a concrete hand's key is in the table iff the hand splits into melds + pair or is
    seven distinct pairs (10,000 hands built from random melds and then perturbed, sizes 2..14)."""
    import gen_agari_table as g

    rng = np.random.default_rng(7)
    n_win = n_lose = 0
    for _ in range(10_000):
        n_melds = int(rng.integers(0, 5))
        c = [0] * 34
        for _m in range(n_melds):
            if rng.random() < 0.4:
                c[int(rng.integers(0, 34))] += 3
            else:
                s0 = int(rng.integers(0, 3)) * 9 + int(rng.integers(0, 7))
                for j in range(3):
                    c[s0 + j] += 1
        c[int(rng.integers(0, 34))] += 2
        if rng.random() < 0.15 and n_melds == 4:  # some seven-pairs shapes
            c = [0] * 34
            for t in rng.choice(34, 7, replace=False):
                c[int(t)] = 2
        if rng.random() < 0.5:  # move one tile: usually breaks the hand, sometimes not
            held = [t for t in range(34) if c[t]]
            c[held[int(rng.integers(0, len(held)))]] -= 1
            c[int(rng.integers(0, 34))] += 1
        if max(c) > 4:
            continue
        wins = _splits_into_melds(c, True) or (sum(c) == 14 and sorted(x for x in c if x) == [2] * 7)
        in_table = g.shape_key(_hand_blocks(c)) in agari_table
        assert wins == in_table, c
        n_win += wins
        n_lose += not wins
    assert n_win > 2000 and n_lose > 2000
