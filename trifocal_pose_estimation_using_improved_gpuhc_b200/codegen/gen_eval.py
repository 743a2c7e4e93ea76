#!/usr/bin/env python3
"""Problem compiler: turns the reference's padded evaluation-index tables into a compact SIMT schedule.

Input  : the two index tables of a minimal problem (reference format, SURVEY.md App. A.3;
         `problems/trifocal_2op1p_30x30/dHdx_indx.txt`, `dHdt_indx.txt`), taken from the packaged fixture.
Output : `csrc/hc_problem_gen.h` — tables + X-macros consumed by the CUDA tracker (`csrc/hc_tracker.cu`).

What the reference does (gpu-idx-evals/dev-eval-indxing-trifocal_2op1p_30x30_LimUnroll_L2Cache.cuh:57-148):
every lane (= matrix row) walks 30 columns x 8 padded term slots for Hx (7200 slots, 558 non-zero) and
16 padded slots for H / Ht, reading 5-6 int32 indices per slot from a 152 KB table in global memory.

What we emit instead (same arithmetic per term, see "evaluation spec" in DESIGN.md):
  * coefficient tables: every distinct (coef, p_a, p_b) triple becomes one entry  cq = coef * p_a(t) * p_b(t)
    (and  dq = coef * (dp_a p_b + dp_b p_a)  for Ht); the warp builds them cooperatively once per change of t;
  * column classes: columns that never share a row (e.g. 24|27, 0|1, 2..11) are evaluated in ONE accumulator
    per lane and scattered to the register row afterwards, so Hx needs ~32 term slots per lane instead of 240;
  * every slot multiplies ALL factor positions, padded ones included (x[30] == 1), exactly like the reference's
    `coef * p[a] * p[b] * x[d] * x[e]`; a lane without a term in a slot reads the zero coefficient and x[30];
  * x-products: every distinct product x_d*x_e (Hx) or x_d*x_e*x_f (H, Ht) of non-padded factors is computed once per
    stage by the warp (36 pairs + 84 triples) into shared memory next to x itself, so a term is ONE complex multiply
    cq * xprod and its per-lane operand word is just two 16-bit byte offsets:  cq offset | xprod offset << 16.
Term order inside every matrix entry is the table order, so sums are bit-identical to the oracle's
table-driven evaluation (`oracle/hc_oracle.c`).

Block structure of the Jacobian (`analyze_blocks`).  A symbolic partial-pivoting elimination in natural column order shows
that the first K1 = 18 pivot steps never couple more than six rows: the rows fall into independent groups (here four 6-row
blocks and two 3-row blocks) whose "sparse" columns are private to the group, and only columns 18..29 are shared.  Steps
of different groups commute exactly, so the kernel runs them side by side ("super-steps": 5 instead of 18 sequential
steps) and keeps, per row, only the group's <= 5 sparse columns plus the 12 dense ones (17 register slots instead of 30).
The generator assigns every group a 6-lane segment (two 3-row groups share one), rows ascending inside a segment, and emits
the lane permutation, the per-lane slot maps and the scatter of the evaluated entries into slots.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
sys.path.insert(0, os.path.dirname(PKG))

N = 30          # variables / equations                        } of the problem being compiled: set by configure()
P_PAD = 33      # parameter index that holds the constant 1    } (defaults: trifocal_2op1p_30x30)
X_PAD = 30      # variable index that holds the constant 1     }
WARP = 32
SPEC = dict(name="trifocal_2op1p_30x30", n_vars=30, n_params=33, n_tracks=312, hx_terms=8, hx_parts=5, ht_terms=16, ht_parts=6,
            n_depths=8, trifocal=1, branch_free_update=1)


def configure(spec):
    """Select the minimal problem to compile (sizes as in gpuhc_settings.yaml: Num_Of_Vars, Num_Of_Params, Num_Of_Tracks,
    dHdx_Max_Terms, dHdx_Max_Parts, dHdt_Max_Terms, dHdt_Max_Parts).  The lane-per-row mapping needs Num_Of_Vars <= 31."""
    global N, P_PAD, X_PAD, SPEC
    SPEC = dict(spec)
    N, P_PAD, X_PAD = SPEC["n_vars"], SPEC["n_params"], SPEC["n_vars"]
    assert 1 <= N <= 31 and SPEC["hx_parts"] == 5 and SPEC["ht_parts"] == 6


def read_problem_dir(path):
    """A problem folder in the reference's layout (problems/<name>/: gpuhc_settings.yaml, dHdx_indx.txt, dHdt_indx.txt;
    reference Data_Reader.cpp:123-189, gpuhc_settings.yaml:5-34) -> (spec, dHdx index array, dHdt index array)."""
    cfg = {}
    for line in open(os.path.join(path, "gpuhc_settings.yaml")):
        line = line.split("#")[0]
        if ":" in line:
            k, v = line.split(":", 1)
            cfg[k.strip()] = v.strip().strip('"')
    spec = dict(name=cfg["problem_name"], n_vars=int(cfg["Num_Of_Vars"]), n_params=int(cfg["Num_Of_Params"]), n_tracks=int(cfg["Num_Of_Tracks"]),
                hx_terms=int(cfg["dHdx_Max_Terms"]), hx_parts=int(cfg["dHdx_Max_Parts"]), ht_terms=int(cfg["dHdt_Max_Terms"]),
                ht_parts=int(cfg["dHdt_Max_Parts"]), n_depths=int(cfg.get("Num_Of_Depth_Vars", 0)), trifocal=int(cfg["problem_name"] == "trifocal_2op1p_30x30"),
                branch_free_update=int(cfg.get("HC_Branch_Free_Update", 1)))
    if spec["trifocal"]:
        spec["n_depths"] = 8
    hx = np.array(open(os.path.join(path, "dHdx_indx.txt")).read().split(), dtype=np.int64)
    ht = np.array(open(os.path.join(path, "dHdt_indx.txt")).read().split(), dtype=np.int64)
    return spec, hx, ht


_TABLES = None      # (dHdx, dHdt) flat index arrays of the configured problem; None = the packaged trifocal fixture


def load_tables():
    if _TABLES is None:
        from trifocal_pose_estimation_using_improved_gpuhc_b200 import fixtures
        prob = fixtures.load_problem()
        hx_flat, ht_flat = prob["dHdx_indx"], prob["dHdt_indx"]
    else:
        hx_flat, ht_flat = _TABLES
    hx = np.asarray(hx_flat).reshape(N, SPEC["hx_terms"], SPEC["hx_parts"], N)    # [col][term][part][row]   (Data_Reader.cpp:123-165 token order)
    ht = np.asarray(ht_flat).reshape(SPEC["ht_terms"], SPEC["ht_parts"], N)       # [term][part][row]
    return hx, ht


def parse_terms(hx, ht):
    """Return hx_terms[(row, col)] = [(coef,a,b,[x...])...], h_terms[row] = [...], in table order, zero coefs dropped."""
    hx_terms = {}
    for col in range(N):
        for row in range(N):
            lst = []
            for t in range(hx.shape[1]):
                c, a, b, d, e = (int(v) for v in hx[col, t, :, row])
                if c == 0:
                    continue
                xs = [v for v in (d, e) if v != X_PAD]
                assert not (a == P_PAD and b != P_PAD)
                lst.append((c, a, b, xs))
            if lst:
                hx_terms[(row, col)] = lst
    h_terms = {}
    for row in range(N):
        lst = []
        for t in range(ht.shape[0]):
            c, a, b, d, e, f = (int(v) for v in ht[t, :, row])
            if c == 0:
                continue
            xs = [v for v in (d, e, f) if v != X_PAD]
            assert not (a == P_PAD and b != P_PAD)
            lst.append((c, a, b, xs))
        h_terms[row] = lst
    return hx_terms, h_terms


def level_schedule(hx_terms, K1, segments, seg_cols):
    """Schedule of the sparse phase.  Inside a segment, two private pivot columns commute exactly when no row takes part in both
    (a row takes part in a column's step when its entry there can be non-zero, fill-in included, every pivot choice allowed), so
    columns are put on LEVELS: level(c) = 1 + the last level any of c's rows was busy in, walking the columns in natural order.
    One level of all segments is one super-step of the kernel; within a segment a level holds one or more GROUPS = (column,
    rows) with disjoint row sets, each with its own pivot search and pivot row.
    Returns (levels, level_of_col, first_shared): levels[T] = list of (segment, column, rows); first_shared[T] = the lowest
    shared column that can be non-zero in any row taking part in level T (shared columns below it are exact zeros in all of
    them, so that super-step neither ships nor updates them)."""
    P = np.zeros((N, N), bool)
    for (r, c) in hx_terms:
        P[r, c] = True
    level_of_col = {}
    groups = []                                   # (level, segment, column, rows, union pattern)
    for g, (seg, cols) in enumerate(zip(segments, seg_cols)):
        busy = {r: -1 for r in seg}
        for c in cols:
            part = [r for r in seg if P[r, c]]
            lvl = 1 + max(busy[r] for r in part)
            u = np.zeros(N, bool)
            for r in part:
                u |= P[r]
            for r in part:
                P[r] |= u
                busy[r] = lvl
            level_of_col[c] = lvl
            groups.append((lvl, g, c, part, u.copy()))
    n_levels = 1 + max([l for l, *_ in groups] or [-1])
    levels, first_shared = [], []
    for T in range(n_levels):
        here = [(g, c, part) for (l, g, c, part, u) in groups if l == T]
        for g in range(len(segments)):            # groups of one segment on one level never share a row
            rows = [r for (gg, c, part) in here if gg == g for r in part]
            assert len(rows) == len(set(rows))
        need = np.zeros(N, bool)
        for (l, g, c, part, u) in groups:
            if l == T:
                need |= u
        shared = [c for c in range(K1, N) if need[c]]
        levels.append(here)
        first_shared.append(min(shared) if shared else N)
    return levels, level_of_col, first_shared


def column_classes(hx_terms):
    """Greedy colouring: two columns may share a class iff no row has a non-zero in both."""
    rows_of = {c: {r for (r, cc) in hx_terms if cc == c} for c in range(N)}
    order = sorted(range(N), key=lambda c: (-max((len(hx_terms[(r, c)]) for r in rows_of[c]), default=0), c))
    classes = []
    for c in order:
        if not rows_of[c]:
            continue
        for cl in classes:
            if all(not (rows_of[c] & rows_of[o]) for o in cl):
                cl.append(c)
                break
        else:
            classes.append([c])
    return [sorted(cl) for cl in classes]


def schedule(seqs):
    """seqs[lane] = list of payloads in table order.  Slot k holds every lane's k-th term (None = no term)."""
    n = max(len(q) for q in seqs)
    return [[q[k] if k < len(q) else None for q in seqs] for k in range(n)]


def analyze_blocks(hx_terms):
    """Block structure of the Jacobian, or (0, [], []) — no block-parallel phase, every pivot step warp-wide — when the rows do not
    fall into independent groups of at most six (e.g. a small fully coupled system)."""
    try:
        return _analyze_blocks(hx_terms)
    except AssertionError:
        return 0, [], []


def _analyze_blocks(hx_terms):
    """Symbolic elimination -> (K1, segments, seg_cols).  segments[g] = sorted rows (<= 6), seg_cols[g] = the segment's
    private pivot columns in natural order; columns K1..N-1 are dense (shared by all rows)."""
    P = np.zeros((N, N), bool)
    for (r, c) in hx_terms:
        P[r, c] = True
    parent = list(range(N))

    def find(a):
        while parent[a] != a:
            parent[a] = parent[parent[a]]
            a = parent[a]
        return a

    cand_of = []
    K1 = N
    for k in range(N):
        cand = [r for r in range(N) if P[r, k]]
        if len(cand) > 6:
            K1 = k
            break
        cand_of.append(cand)
        u = np.zeros(N, bool)
        for r in cand:
            u |= P[r]
        u[:k + 1] = False
        for r in cand:
            P[r] |= u
        for r in cand[1:]:
            parent[find(r)] = find(cand[0])
    comps = {}
    for r in range(N):
        comps.setdefault(find(r), []).append(r)
    assert K1 > 0 and all(len(rows) <= 6 for rows in comps.values())
    comps = sorted(comps.values(), key=lambda rows: min([k for k in range(K1) if set(cand_of[k]) & set(rows)] or [N]))
    # pack components into 6-row segments (first-fit in order of their first pivot column)
    segments = []
    for rows in comps:
        for seg in segments:
            if len(seg) + len(rows) <= 6 and len(seg) < 6 and len(rows) < 6:
                seg.extend(rows)
                break
        else:
            segments.append(list(rows))
    segments = [sorted(seg) for seg in segments]
    assert all(len(seg) <= 6 for seg in segments) and len(segments) * 6 <= WARP and sum(len(x) for x in segments) == N
    seg_cols = []
    for seg in segments:
        cols = [k for k in range(K1) if set(cand_of[k]) <= set(seg) and cand_of[k]]
        seg_cols.append(cols)
    assert sorted(c for cols in seg_cols for c in cols) == list(range(K1))
    # every structurally possible non-zero of a row lies in its segment's private columns or in the dense columns
    for g, seg in enumerate(segments):
        for r in seg:
            for c in range(K1):
                assert (not P[r, c]) or c in seg_cols[g], (r, c)
    return K1, segments, seg_cols


def optimise_layout(n_pos, movable_sets, groups, seed=1):
    """Table layout against shared-memory bank conflicts.  A 64-bit gather by a half-warp needs as many wavefronts as the
    largest number of DISTINCT entries that fall into one of the 16 bank pairs (position mod 16).  `groups` lists, for every
    (term slot, half-warp), the set of table entries gathered together; entries inside one of `movable_sets` may exchange
    positions.  Deterministic pairwise-swap local search; returns pos[entry]."""
    import random
    rnd = random.Random(seed)
    pos = list(range(n_pos))
    member = {}
    for gi, grp in enumerate(groups):
        for e in grp:
            member.setdefault(e, []).append(gi)

    def gcost(gi):
        cnt = {}
        for e in groups[gi]:
            k = pos[e] % 16
            cnt[k] = cnt.get(k, 0) + 1
        return max(cnt.values())

    cost = [gcost(gi) for gi in range(len(groups))]
    for mv in movable_sets:
        mv = list(mv)
        for sweep in range(8):
            improved = False
            rnd.shuffle(mv)
            for i in range(len(mv)):
                for j in range(i + 1, len(mv)):
                    e, f = mv[i], mv[j]
                    affected = set(member.get(e, [])) | set(member.get(f, []))
                    if not affected:
                        continue
                    before = sum(cost[gi] for gi in affected)
                    pos[e], pos[f] = pos[f], pos[e]
                    after = {gi: gcost(gi) for gi in affected}
                    if sum(after.values()) < before:
                        for gi, c in after.items():
                            cost[gi] = c
                        improved = True
                    else:
                        pos[e], pos[f] = pos[f], pos[e]
            if not improved:
                break
    return pos, sum(cost)


def _groups(slot_rows, field, pad_entry):
    out = []
    for row in slot_rows:
        for half in (range(0, 16), range(16, 32)):
            out.append({pad_entry if row[l] is None else row[l][field] for l in half})
    return out


def build():
    hx, ht = load_tables()
    hx_terms, h_terms = parse_terms(hx, ht)

    # ---- coefficient tables -------------------------------------------------------------------------------
    cq_keys = set()
    for lst in hx_terms.values():
        cq_keys.update((c, a, b) for c, a, b, _ in lst)
    for lst in h_terms.values():
        cq_keys.update((c, a, b) for c, a, b, _ in lst)
    # index 0 is the zero coefficient used by empty slots
    cq_list = [(0, P_PAD, P_PAD)] + sorted(cq_keys, key=lambda k: (k[2] == P_PAD, k[1], k[2], k[0]))
    cq_index = {k: i for i, k in enumerate(cq_list)}
    dq_keys = set()
    for lst in h_terms.values():
        dq_keys.update((c, a, b) for c, a, b, _ in lst if not (a == P_PAD and b == P_PAD))
    dq_list = [(0, P_PAD, P_PAD)] + sorted(dq_keys, key=lambda k: (k[2] == P_PAD, k[1], k[2], k[0]))
    dq_index = {k: i for i, k in enumerate(dq_list)}

    # ---- block structure -> lane permutation and register slots -------------------------------------------
    K1, segments, seg_cols = analyze_blocks(hx_terms)
    levels, level_of_col, sp_first_shared = level_schedule(hx_terms, K1, segments, seg_cols)
    if len(levels) > 4 or (len(levels) + N - K1) % 2:      # the kernel packs at most four levels per lane word and moves slots in pairs
        K1, segments, seg_cols = 0, [], []
        levels, level_of_col, sp_first_shared = level_schedule(hx_terms, K1, segments, seg_cols)
    SEG = 6
    row_of_lane = [-1] * WARP
    for g, seg in enumerate(segments):
        for i, r in enumerate(seg):
            row_of_lane[g * SEG + i] = r
    if not segments:                               # no block structure: row r on lane r
        for r in range(N):
            row_of_lane[r] = r
    lane_of_row = [row_of_lane.index(r) for r in range(N)]
    nsp = len(levels)
    nd = N - K1
    # per lane and level: the private column the lane's row meets there (or None), the lanes of its group (6-bit mask relative
    # to the segment's first lane) and the group's index within the segment (selects the pivot-row buffer)
    col_at = [[None] * nsp for _ in range(WARP)]
    grp_mask = [[0] * nsp for _ in range(WARP)]
    grp_sub = [[0] * nsp for _ in range(WARP)]
    max_sub = 1
    for T, here in enumerate(levels):
        n_in_seg = {}
        for (g, c, part) in here:
            sub = n_in_seg.get(g, 0)
            n_in_seg[g] = sub + 1
            max_sub = max(max_sub, sub + 1)
            mask = 0
            for r in part:
                mask |= 1 << (lane_of_row[r] - g * SEG)
            for r in part:
                ln = lane_of_row[r]
                col_at[ln][T], grp_mask[ln][T], grp_sub[ln][T] = c, mask, sub
    assert max_sub <= 2

    def slot_of(lane, col):
        if col >= K1:
            return nsp + (col - K1)
        assert col_at[lane][level_of_col[col]] == col
        return level_of_col[col]

    # ---- x-product table: [x(32 entries, x[30] = 1) | pairs (padded to a multiple of 32) | triples] -------------------
    pairs, triples = set(), set()
    for lst in list(hx_terms.values()) + list(h_terms.values()):
        for c, a, b, xs in lst:
            if len(xs) == 2:
                pairs.add(tuple(xs))
            elif len(xs) == 3:
                triples.add(tuple(xs))
    pairs, triples = sorted(pairs), sorted(triples)
    XP_PAIR0 = 32
    XP_TRI0 = XP_PAIR0 + ((len(pairs) + WARP - 1) // WARP) * WARP
    XP_TOTAL = XP_TRI0 + ((len(triples) + 7) // 8) * 8

    def xp_index(xs):
        if len(xs) == 0:
            return X_PAD
        if len(xs) == 1:
            return xs[0]
        if len(xs) == 2:
            return XP_PAIR0 + pairs.index(tuple(xs))
        return XP_TRI0 + triples.index(tuple(xs))

    # ---- Hx: classes + slots ------------------------------------------------------------------------------
    classes = column_classes(hx_terms)
    col_class = {c: ci for ci, cl in enumerate(classes) for c in cl}
    hx_slots = []      # (class, [payload]*32)
    for ci, cl in enumerate(classes):
        seqs = []
        for lane in range(WARP):
            seq = []
            row = row_of_lane[lane]
            if row >= 0:
                cols = [c for c in cl if (row, c) in hx_terms]
                assert len(cols) <= 1
                if cols:
                    for c, a, b, xs in hx_terms[(row, cols[0])]:
                        seq.append((cq_index[(c, a, b)], xp_index(xs)))
            seqs.append(seq)
        for row in schedule(seqs):
            hx_slots.append((ci, row))

    def sched_rows(terms_of_row, index, drop_const):
        seqs = []
        for lane in range(WARP):
            seq = []
            if row_of_lane[lane] >= 0:
                for c, a, b, xs in terms_of_row[row_of_lane[lane]]:
                    if drop_const and a == P_PAD and b == P_PAD:
                        continue      # d/dt of a parameter-free term vanishes (…L2Cache.cuh:107-118 adds an exact 0)
                    seq.append((index[(c, a, b)], xp_index(xs)))
            seqs.append(seq)
        return schedule(seqs)

    h_slots = sched_rows(h_terms, cq_index, False)
    ht_slots = sched_rows(h_terms, dq_index, True)
    while len(ht_slots) < len(h_slots):            # H and Ht share one slot loop in the kernel: pad with empty slots (cq[0] == 0 times x[N] == 1)
        ht_slots.append([None] * WARP)
    assert (nsp + nd) % 2 == 0, "the kernel moves register slots in pairs: levels + dense columns must be even"
    assert all(row_of_lane[l] >= 0 for l in range(N)) and all(row_of_lane[l] < 0 for l in range(N, WARP)), "rows must occupy lanes 0..N-1"
    assert all(-2 <= c <= 5 for lst in list(hx_terms.values()) + list(h_terms.values()) for c, _, _, _ in lst), "coefficients are packed into 3 bits"

    # ---- bank-conflict-aware table layouts --------------------------------------------------------------------------
    hx_rows = [row for _, row in hx_slots]
    cost0 = [sum(max(sum(1 for e in grp if e % 16 == k) for k in range(16)) for grp in _groups(r, f, pe))
             for r, f, pe in ((hx_rows + h_slots, 0, 0), (ht_slots, 0, 0), (hx_rows + h_slots + ht_slots, 1, X_PAD))]
    cq_pos, c_cq = optimise_layout(len(cq_list), [range(1, len(cq_list))], _groups(hx_rows + h_slots, 0, 0))
    dq_pos, c_dq = optimise_layout(len(dq_list), [range(1, len(dq_list))], _groups(ht_slots, 0, 0))
    xp_pos, c_xp = optimise_layout(XP_TOTAL, [range(XP_PAIR0, XP_TRI0), range(XP_TRI0, XP_TOTAL)],
                                   _groups(hx_rows + h_slots + ht_slots, 1, X_PAD))
    layout_cost = dict(before=cost0, after=[c_cq, c_dq, c_xp])

    def remap(rows, cpos):
        return [[None if p is None else (cpos[p[0]], xp_pos[p[1]]) for p in row] for row in rows]

    hx_slots = [(ci, r) for (ci, _), r in zip(hx_slots, remap(hx_rows, cq_pos))]
    h_slots = remap(h_slots, cq_pos)
    ht_slots = remap(ht_slots, dq_pos)
    # tables in POSITION order (the build rounds walk positions, so their stores stay conflict-free)
    cq_by_pos = [(0, P_PAD, P_PAD)] * len(cq_list)
    for e, q in enumerate(cq_pos):
        cq_by_pos[q] = cq_list[e]
    dq_by_pos = [(0, P_PAD, P_PAD)] * len(dq_list)
    for e, q in enumerate(dq_pos):
        dq_by_pos[q] = dq_list[e]
    cq_list, dq_list = cq_by_pos, dq_by_pos
    pair_by_pos = [None] * (XP_TRI0 - XP_PAIR0)
    for i, pr in enumerate(pairs):
        pair_by_pos[xp_pos[XP_PAIR0 + i] - XP_PAIR0] = pr
    tri_by_pos = [None] * (XP_TOTAL - XP_TRI0)
    for i, tr in enumerate(triples):
        tri_by_pos[xp_pos[XP_TRI0 + i] - XP_TRI0] = tr

    # ---- scatter of the class accumulators into register slots --------------------------------------------------
    # slot t of a lane holds the private column its row meets on level t (t < nsp) or K1 + (t - nsp); the class feeding it may
    # depend on the lane -> at most two candidates per slot, chosen by one per-lane selector bit
    nslot = nsp + nd
    scatter = []           # per slot: (classA, classB or -1, selector bit index or -1)
    sel_of_lane = [0] * WARP
    nz_of_lane = [0] * WARP
    n_sel = 0
    for t in range(nslot):
        cls_per_lane = []
        for lane in range(WARP):
            col = col_at[lane][t] if t < nsp else (K1 + (t - nsp) if row_of_lane[lane] >= 0 else None)
            cls_per_lane.append(col_class.get(col) if col is not None else None)
        used = sorted({c for c in cls_per_lane if c is not None})
        assert 1 <= len(used) <= 2
        if len(used) == 1:
            scatter.append((used[0], -1, -1))
        else:
            scatter.append((used[0], used[1], n_sel))
            for lane in range(WARP):
                if cls_per_lane[lane] == used[1]:
                    sel_of_lane[lane] |= 1 << n_sel
            n_sel += 1
    for lane in range(WARP):
        row = row_of_lane[lane]
        if row < 0:
            continue
        for c in range(N):
            if (row, c) in hx_terms:
                nz_of_lane[lane] |= 1 << slot_of(lane, c)
    return dict(hx_terms=hx_terms, h_terms=h_terms, cq_list=cq_list, dq_list=dq_list, classes=classes,
                col_class=col_class, hx_slots=hx_slots, h_slots=h_slots, ht_slots=ht_slots,
                K1=K1, segments=segments, seg_cols=seg_cols, row_of_lane=row_of_lane, lane_of_row=lane_of_row,
                nsp=nsp, nd=nd, nslot=nslot, sp_first_shared=sp_first_shared, levels=levels, level_of_col=level_of_col,
                col_at=col_at, grp_mask=grp_mask, grp_sub=grp_sub, max_sub=max_sub, scatter=scatter, sel_of_lane=sel_of_lane, nz_of_lane=nz_of_lane, n_sel=n_sel,
                pairs=pair_by_pos, triples=tri_by_pos, XP_PAIR0=XP_PAIR0, XP_TRI0=XP_TRI0, XP_TOTAL=XP_TOTAL,
                layout_cost=layout_cost)


def pack_word(payload):
    """cq byte offset (16 bits) | x-product byte offset << 16; an empty slot reads cq[0] == 0 and x[30] == 1."""
    idx, xp = (0, X_PAD) if payload is None else payload
    return (idx * 8) | ((xp * 8) << 16)


def pack_xp_word(xs):
    """x byte offsets of up to three factors, 8 bits each (x[i] is entry i of the x-product array)."""
    xs = list(xs) + [X_PAD] * (3 - len(xs))
    return (xs[0] * 8) | ((xs[1] * 8) << 8) | ((xs[2] * 8) << 16)


def pack_build_word(key):
    c, a, b = key
    # a_off (9 bits) | b_off (9 bits) << 9 | (coef + 2) << 18
    return (a * 8) | ((b * 8) << 9) | ((c + 2) << 18)


def emit(g, path):
    ncq, ndq = len(g["cq_list"]), len(g["dq_list"])
    rounds = lambda n: (n + WARP - 1) // WARP
    L = []
    w = L.append
    w("// GENERATED by codegen/gen_eval.py from the problem's evaluation-index tables — do not edit.")
    w("// Problem: %s (%d equations, %d unknowns, %d parameters, %d paths)." % (SPEC["name"], N, N, SPEC["n_params"], SPEC["n_tracks"]))
    w("#ifndef HC_PROBLEM_GEN_H")
    w("#define HC_PROBLEM_GEN_H")
    w("#define HCG_N %d" % N)
    w("#define HCG_NUM_PARAMS %d" % SPEC["n_params"])
    w("#define HCG_NUM_CQ %d   /* coef*p_a*p_b table (entry 0 == 0) */" % ncq)
    w("#define HCG_NUM_DQ %d   /* coef*(dp_a*p_b + dp_b*p_a) table (entry 0 == 0) */" % ndq)
    w("#define HCG_CQ_ROUNDS %d" % rounds(ncq))
    w("#define HCG_DQ_ROUNDS %d" % rounds(ndq))
    w("#define HCG_NUM_CLASSES %d" % len(g["classes"]))
    w("#define HCG_HX_SLOTS %d" % len(g["hx_slots"]))
    w("#define HCG_H_SLOTS %d" % len(g["h_slots"]))
    w("#define HCG_HT_SLOTS %d" % len(g["ht_slots"]))
    nnz = len(g["hx_terms"])
    nterms = sum(len(v) for v in g["hx_terms"].values())
    w("#define HCG_HX_NNZ %d" % nnz)
    w("#define HCG_HX_TERMS %d" % nterms)
    w("#define HCG_H_TERMS %d" % sum(len(v) for v in g["h_terms"].values()))
    # word table layout: [cq build rounds][dq build rounds][pair rounds][triple rounds][hx slots][h slots][ht slots], 32 words each
    off_cq = 0
    off_dq = off_cq + rounds(ncq)
    off_pair = off_dq + rounds(ndq)
    off_tri = off_pair + rounds(len(g["pairs"]))
    off_hx = off_tri + rounds(len(g["triples"]))
    w("#define HCG_XP_PAIR0 %d   /* x-product array: [0,32) x itself, then %d pairs, then %d triples */" % (g["XP_PAIR0"], len(g["pairs"]), len(g["triples"])))
    w("#define HCG_XP_TRI0 %d" % g["XP_TRI0"])
    w("#define HCG_XP_TOTAL %d" % g["XP_TOTAL"])
    w("#define HCG_NUM_PAIRS %d" % len(g["pairs"]))
    w("#define HCG_NUM_TRIPLES %d" % len(g["triples"]))
    w("#define HCG_PAIR_ROUNDS %d" % rounds(len(g["pairs"])))
    w("#define HCG_TRI_ROUNDS %d" % rounds(len(g["triples"])))
    w("#define HCG_TBL_PAIR %d" % off_pair)
    w("#define HCG_TBL_TRI %d" % off_tri)
    off_h = off_hx + len(g["hx_slots"])
    off_ht = off_h + len(g["h_slots"])
    total = off_ht + len(g["ht_slots"])
    w("#define HCG_TBL_CQ %d" % off_cq)
    w("#define HCG_TBL_DQ %d" % off_dq)
    w("#define HCG_TBL_HX %d" % off_hx)
    w("#define HCG_TBL_H %d" % off_h)
    w("#define HCG_TBL_HT %d" % off_ht)
    w("#define HCG_TBL_ROWS %d" % total)
    rows = []
    for lst, n in ((g["cq_list"], ncq), (g["dq_list"], ndq)):
        for r in range(rounds(n)):
            rows.append([pack_build_word(lst[r * WARP + l]) if r * WARP + l < n else pack_build_word((0, P_PAD, P_PAD))
                         for l in range(WARP)])
    for lst in (g["pairs"], g["triples"]):
        for r in range(rounds(len(lst))):
            rows.append([pack_xp_word(lst[r * WARP + l]) if r * WARP + l < len(lst) and lst[r * WARP + l] is not None else pack_xp_word([])
                         for l in range(WARP)])
    for _, row in g["hx_slots"]:
        rows.append([pack_word(p) for p in row])
    for row in g["h_slots"]:
        rows.append([pack_word(p) for p in row])
    for row in g["ht_slots"]:
        rows.append([pack_word(p) for p in row])
    assert len(rows) == total
    w("// packed per-lane operand words, [row][lane]")
    w("#define HCG_TBL_INIT { \\")
    for r in rows:
        w("  " + ",".join("0x%08xu" % v for v in r) + ", \\")
    w("}")
    # ---- block structure ----------------------------------------------------------------------------------------
    w("// block structure: %d segments of 6 lanes; sparse pivot columns per segment %s; dense columns %d..%d"
      % (len(g["segments"]), g["seg_cols"], g["K1"], N - 1))
    for T, here in enumerate(g["levels"]):
        w("//   level %d: %s" % (T, "  ".join("col %d rows %s" % (c, part) for (_, c, part) in here)))
    w("#define HCG_K1 %d        /* first dense pivot column */" % g["K1"])
    w("#define HCG_NSP %d        /* sparse slots == levels (super-steps) */" % g["nsp"])
    w("#define HCG_ND %d        /* dense slots */" % g["nd"])
    w("#define HCG_NSLOT %d     /* register slots per row */" % g["nslot"])
    w("#define HCG_SEG 6")
    w("#define HCG_NSEG %d" % max(1, len(g["segments"])))
    w("// per super-step: first register slot of the shared columns that can be non-zero in a participating row")
    w("#define HCG_SP_FIRST_SHARED_SLOT_INIT { " + ",".join([str(g["nsp"] + c - g["K1"]) for c in g["sp_first_shared"]] or ["0"]) + " }")
    w("#define HCG_ROW_OF_LANE_INIT { " + ",".join(str(r) for r in g["row_of_lane"]) + " }")
    w("#define HCG_LANE_OF_ROW_INIT { " + ",".join(str(r) for r in g["lane_of_row"]) + " }")
    # per-lane info word: nz mask over slots (bits 0..nslot-1) | selector bits << 20
    info, cols, grps = [], [], []
    for lane in range(WARP):
        assert g["nslot"] <= 20 and g["n_sel"] <= 4 and g["nsp"] <= 4
        info.append(g["nz_of_lane"][lane] | (g["sel_of_lane"][lane] << 20))
        packed, gp = 0, 0
        for t in range(g["nsp"]):
            if g["col_at"][lane][t] is not None:
                packed |= g["col_at"][lane][t] << (5 * t)
                gp |= (g["grp_mask"][lane][t] | (g["grp_sub"][lane][t] << 6)) << (7 * t)
        cols.append(packed)
        grps.append(gp)
    w("#define HCG_LANEINFO_INIT { " + ",".join("0x%08xu" % v for v in info) + " }")
    w("#define HCG_LANECOLS_INIT { " + ",".join("0x%08xu" % v for v in cols) + " }   /* 5 bits per level: the private column the lane's row meets there */")
    w("#define HCG_LANEGRP_INIT { " + ",".join("0x%08xu" % v for v in grps) + " }   /* 7 bits per level: lanes of my pivot group (6, relative to the segment) | group index << 6; 0 = idle */")
    w("#define HCG_MAX_GROUPS_PER_SEG %d" % g["max_sub"])
    w("// X(slot, class): one Hx term slot; acc[class] += cq * xprod")
    # slots are ordered by class: first slot of every class (+ end), for the rolled per-class loops of the evaluator
    begs, prev = [], None
    for i, (ci, _) in enumerate(g["hx_slots"]):
        if ci != prev:
            assert prev is None or ci == prev + 1
            begs.append(i)
            prev = ci
    begs.append(len(g["hx_slots"]))
    assert len(begs) == len(g["classes"]) + 1
    w("#define HCG_HX_CLASS_BEGIN_INIT { " + ",".join(str(b) for b in begs) + " }   /* first Hx slot of every class, then the end */")
    w("#define HCG_HX_SLOT_LIST(X) \\")
    for s, (ci, _) in enumerate(g["hx_slots"]):
        w("  X(%d, %d) \\" % (s, ci))
    w("")
    w("// X(slot, classA, classB, selbit): A[slot] = lane has a non-zero there ? acc[selbit set ? classB : classA] : 0")
    w("#define HCG_HX_SCATTER_LIST(X) \\")
    for t, (ca, cb, sb) in enumerate(g["scatter"]):
        w("  X(%d, %d, %d, %d) \\" % (t, ca, cb, sb))
    w("")
    w("// problem identity: the kernel takes every size from this header (codegen/gen_eval.py --problem-dir compiles another problem)")
    w("#define HCG_PROBLEM_NAME \"%s\"" % SPEC["name"])
    w("#define HCG_TRACKS %d        /* homotopy paths per hypothesis (Num_Of_Tracks) */" % SPEC["n_tracks"])
    w("#define HCG_NUM_DEPTHS %d      /* leading variables that are depths: positive-depth pruning tests them (0: no pruning) */" % SPEC["n_depths"])
    w("#define HCG_TRIFOCAL %d        /* 1: the trifocal relative-pose problem (in-kernel scoring, pose records, target-parameter gather) */" % SPEC["trifocal"])
    w("#define HCG_BRANCH_FREE_UPDATE %d   /* elimination-step update predicate: 1 with & (no divergent region), 0 with && (settings key HC_Branch_Free_Update) */"
      % SPEC["branch_free_update"])
    w("")
    w("#endif")
    text = "\n".join(L) + "\n"
    with open(path, "w") as f:
        f.write(text)
    return text


def compile_problem(problem_dir, out):
    """Problem folder in the reference's layout -> generated header for csrc/hc_tracker.cu (-DHC_PROBLEM_HEADER)."""
    global _TABLES
    spec, hx, ht = read_problem_dir(problem_dir)
    configure(spec)
    _TABLES = (hx, ht)
    g = build()
    emit(g, out)
    return g


def main():
    import argparse
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--problem-dir", default=None, help="problems/<name>/ in the reference's layout (default: the packaged trifocal_2op1p_30x30 tables)")
    ap.add_argument("--out", default=None, help="header to write (default: csrc/hc_problem_gen.h, or csrc/hc_problem_gen_<name>.h with --problem-dir)")
    a = ap.parse_args()
    if a.problem_dir:
        spec = read_problem_dir(a.problem_dir)[0]
        out = a.out or os.path.join(PKG, "csrc", "hc_problem_gen_%s.h" % spec["name"])
        g = compile_problem(a.problem_dir, out)
        print("problem %s: N %d, parameters %d, paths %d | K1 %d segments %s | classes %s | Hx slots %d, H slots %d, Ht slots %d | cq %d dq %d | pairs %d triples %d"
              % (SPEC["name"], N, SPEC["n_params"], SPEC["n_tracks"], g["K1"], g["segments"], g["classes"], len(g["hx_slots"]), len(g["h_slots"]),
                 len(g["ht_slots"]), len(g["cq_list"]), len(g["dq_list"]), sum(p is not None for p in g["pairs"]), sum(t is not None for t in g["triples"])))
        print("wrote", out)
        return
    g = build()
    out = a.out or os.path.join(PKG, "csrc", "hc_problem_gen.h")
    emit(g, out)
    print("classes:", g["classes"])
    print("K1 %d segments %s seg_cols %s" % (g["K1"], g["segments"], g["seg_cols"]))
    print("row_of_lane", g["row_of_lane"])
    print("scatter", g["scatter"])
    print("cq entries %d, dq entries %d" % (len(g["cq_list"]), len(g["dq_list"])))
    print("Hx slots %d (ref 240), H slots %d (ref 16), Ht slots %d (ref 16)" %
          (len(g["hx_slots"]), len(g["h_slots"]), len(g["ht_slots"])))
    print("gather wavefront model (cq, dq, xp) before/after layout optimisation:", g["layout_cost"])
    print("hx_slots", [(ci, sum(p is not None for p in row)) for ci, row in g["hx_slots"]])
    print("h_slots", [sum(p is not None for p in row) for row in g["h_slots"]])
    print("ht_slots", [sum(p is not None for p in row) for row in g["ht_slots"]])
    print("wrote", out)


if __name__ == "__main__":
    main()
