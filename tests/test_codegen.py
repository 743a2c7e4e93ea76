"""The problem compiler (codegen/gen_eval.py): its schedule must contain every non-zero term of the reference's index tables
exactly once, in table order, and the committed header must be what the generator produces."""
import os

import numpy as np

from trifocal_pose_estimation_using_improved_gpuhc_b200.codegen import gen_eval

PKG = os.path.dirname(os.path.dirname(os.path.abspath(gen_eval.__file__)))


def test_generated_header_is_current(tmp_path):
    g = gen_eval.build()
    text = gen_eval.emit(g, str(tmp_path / "gen.h"))
    assert text == open(os.path.join(PKG, "csrc", "hc_problem_gen.h")).read()


def test_table_statistics_match_survey():
    g = gen_eval.build()
    assert len(g["hx_terms"]) == 170                                   # SURVEY.md App. F: 170 of 900 entries
    assert sum(len(v) for v in g["hx_terms"].values()) == 558          # 558 of 7200 padded terms
    assert sum(len(v) for v in g["h_terms"].values()) == 360
    ht = sum(1 for v in g["h_terms"].values() for (c, a, b, xs) in v if not (a == 33 and b == 33))
    assert ht == 300                                                   # 60 parameter-free terms vanish in d/dt
    assert len(g["hx_slots"]) == 25 and len(g["h_slots"]) == 16 and len(g["ht_slots"]) == 16


def _unpack(word):
    return word & 0xffff, word >> 16


def _xs_of(g, xp_off):
    """invert the x-product offset: entry of x itself, of the pair table, or of the triple table"""
    i = xp_off // 8
    if i < 32:
        return [] if i == 30 else [i]
    if i < g["XP_TRI0"]:
        return list(g["pairs"][i - g["XP_PAIR0"]])
    return list(g["triples"][i - g["XP_TRI0"]])


def test_schedule_covers_every_term_once_in_table_order():
    g = gen_eval.build()
    rol = g["row_of_lane"]
    assert sorted(r for r in rol if r >= 0) == list(range(30)) and rol[30] == rol[31] == -1
    # Hx: per (lane, class) the slot sequence must equal the entry of the lane's ROW in that class
    for lane in range(30):
        row = rol[lane]
        for ci, cols in enumerate(g["classes"]):
            mine = [c for c in cols if (row, c) in g["hx_terms"]]
            assert len(mine) <= 1
            want = g["hx_terms"][(row, mine[0])] if mine else []
            got = []
            for cls, slot_row in g["hx_slots"]:
                if cls != ci:
                    continue
                off, xp = _unpack(gen_eval.pack_word(slot_row[lane]))
                if off == 0:
                    assert xp == 30 * 8          # empty slot: zero coefficient times x[30] == 1
                    continue
                c, a, b = g["cq_list"][off // 8]
                got.append((c, a, b, _xs_of(g, xp)))
            assert got == want
    for name, lst, drop in (("h_slots", g["cq_list"], False), ("ht_slots", g["dq_list"], True)):
        for lane in range(30):
            want = [(c, a, b, xs) for (c, a, b, xs) in g["h_terms"][rol[lane]] if not (drop and a == 33 and b == 33)]
            got = []
            for slot_row in g[name]:
                off, xp = _unpack(gen_eval.pack_word(slot_row[lane]))
                if off == 0:
                    continue
                c, a, b = lst[off // 8]
                got.append((c, a, b, _xs_of(g, xp)))
            assert got == want
    # lanes 30, 31 never hold a term
    for _, slot_row in g["hx_slots"]:
        assert slot_row[30] is None and slot_row[31] is None


def test_block_structure_is_what_the_kernel_assumes():
    """analyze_blocks + level_schedule: 18 sparse pivot columns in five independent 6-row groups, scheduled on 4 levels (columns of a
    group whose rows are disjoint share a level), 12 shared columns, 16 register slots."""
    g = gen_eval.build()
    assert g["K1"] == 18 and g["nsp"] == 4 and g["nd"] == 12 and g["nslot"] == 16
    assert g["segments"] == [[3, 4, 5, 12, 13, 14], [6, 7, 8, 15, 16, 17], [0, 1, 2, 9, 10, 11], [18, 19, 20, 24, 25, 26], [21, 22, 23, 27, 28, 29]]
    assert g["seg_cols"] == [[0, 3, 6], [1, 4, 7], [2, 5], [8, 9, 12, 13, 14], [10, 11, 15, 16, 17]]
    assert [sorted(c for (_, c, _) in lv) for lv in g["levels"]] == [[0, 1, 2, 5, 8, 9, 10, 11], [3, 4, 12, 15], [6, 7, 13, 16], [14, 17]]
    assert g["sp_first_shared"] == [18, 18, 18, 24] and g["max_sub"] == 2
    # every structural non-zero of a row is in one of the row's slots, and rows are ascending inside a segment
    for lane, row in enumerate(g["row_of_lane"]):
        if row < 0:
            continue
        seg = lane // 6
        for c in range(30):
            if (row, c) in g["hx_terms"]:
                assert c >= g["K1"] or (c in g["seg_cols"][seg] and g["col_at"][lane][g["level_of_col"][c]] == c)
    for seg in g["segments"]:
        assert seg == sorted(seg)
    # independence that makes the block-parallel schedule exact: a sparse column is non-zero only inside its own segment
    for (row, c) in g["hx_terms"]:
        if c < g["K1"]:
            owner = [i for i, cols in enumerate(g["seg_cols"]) if c in cols][0]
            assert row in g["segments"][owner]


def test_level_schedule_is_exact():
    """Replays a symbolic natural-order elimination with worst-case fill-in and checks what the levels rely on: the groups of one
    level have pairwise disjoint rows, a column's level is above the level of every earlier column that shares a row with it, and a
    row's entry in a column it does not 'meet' stays structurally zero (so leaving it out of that column's pivot search and update
    changes nothing)."""
    g = gen_eval.build()
    P = np.zeros((30, 30), bool)
    for (r, c) in g["hx_terms"]:
        P[r, c] = True
    part_of = {}
    for lv in g["levels"]:
        rows = [r for (_, _, part) in lv for r in part]
        assert len(rows) == len(set(rows))
        for (_, c, part) in lv:
            part_of[c] = part
    assert sorted(part_of) == list(range(g["K1"]))
    last_level = {}
    for c in range(g["K1"]):                                  # natural order, as the oracle eliminates
        touched = [r for r in range(30) if P[r, c]]
        assert sorted(touched) == sorted(part_of[c])          # exactly the rows of the group: everything else is structurally zero
        u = np.zeros(30, bool)
        for r in touched:
            u |= P[r]
        for r in touched:
            P[r] |= u
            assert last_level.get(r, -1) < g["level_of_col"][c]
            last_level[r] = g["level_of_col"][c]
    # rows taking part in the last level never touch shared columns 18..23
    for (_, c, part) in g["levels"][-1]:
        for r in part:
            assert not P[r, 18:24].any()


def test_column_classes_partition_the_nonzero_columns():
    g = gen_eval.build()
    cols = sorted(c for cl in g["classes"] for c in cl)
    assert cols == list(range(30))
    for cl in g["classes"]:
        for lane in range(30):
            assert sum((lane, c) in g["hx_terms"] for c in cl) <= 1
