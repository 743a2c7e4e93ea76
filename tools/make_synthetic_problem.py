#!/usr/bin/env python3
"""Writes problems/coupled_quadrics_8x8/ and problems/dense_quadrics_6x6/ — two more minimal problems in the reference's problem-folder
format (SURVEY.md App. A.3; reference problems/trifocal_2op1p_30x30/*, Data_Reader.cpp:37-189), used to show that the problem compiler
(codegen/gen_eval.py), the tracker kernel, the oracle and the reference's own generic CPU-HC solver all take a problem as DATA.

coupled_quadrics_8x8 (8 equations, 8 unknowns x0..x7, 10 parameters p0..p9; i+k taken modulo 8) — its Jacobian has a block structure the
compiler finds (two private pivot columns, six shared ones):

    f_i = x_i^2 - p_i^2 + p_8 x_{i+1} x_{i+3} + p_9 x_{i+2}  [+ p_8 p_9 x_{i+5} x_{i+6} x_{i+7}  for i = 0, 4]

dense_quadrics_6x6 (6 unknowns, 7 parameters) — every equation couples every unknown, so there is NO block structure and the kernel runs
all six pivot steps warp-wide (the compiler's fallback):

    f_i = x_i^2 - p_i^2 + p_6 x_i (sum over j != i of x_j)

mixed_12x12 (12 unknowns, 14 parameters, 64 paths) — six quadrics and six equations that are linear in their own unknown, two 6-row blocks:

    f_i = x_i^2 - p_i^2 + p_12 x_{i+1} x_{i+6}   (i < 6)        f_i = x_i - p_i + p_13 x_{i-6} x_{i+1}   (i >= 6)

Start parameters: p_0..p_7 = a_i (random complex, fixed seed), p_8 = p_9 = 0  ->  the start system decouples into x_i^2 = a_i^2 and has the
2^8 = 256 regular solutions x_i = +-a_i: those are the start solutions (Num_Of_Tracks = 256).  Target parameters are real, like the
reference's (they come from image measurements there): every hypothesis draws p_0..p_7 in [0.6, 1.4] and the couplings p_8, p_9 in
[-0.45, 0.45].  The tables use every feature of the format: parameter-free terms, one- and two-parameter coefficients, products of one,
two and three unknowns, coefficients 1, -1 and 2, and the Jacobian table is the exact derivative of the H table.

    python tools/make_synthetic_problem.py            # (re)writes the folder; deterministic
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAME = "coupled_quadrics_8x8"
NAMES = ("coupled_quadrics_8x8", "dense_quadrics_6x6", "mixed_12x12")
SIZES = {"coupled_quadrics_8x8": (8, 10, 2), "dense_quadrics_6x6": (6, 7, 0), "mixed_12x12": (12, 14, 3)}      # unknowns, parameters, depth unknowns
# ptxas's register outcome of the two update-predicate forms, per problem (lib/ptxas_hc_tracker_<name>.log): mixed_12x12 spills with &
BRANCH_FREE_UPDATE = {"coupled_quadrics_8x8": 1, "dense_quadrics_6x6": 1, "mixed_12x12": 0}
N_SQUARES = {"coupled_quadrics_8x8": 8, "dense_quadrics_6x6": 6, "mixed_12x12": 6}      # equations that are quadratic in their own unknown: 2^k start solutions
N, NP = 8, 10
X_PAD, P_PAD = N, NP


def select(name):
    global NAME, N, NP, X_PAD, P_PAD
    NAME = name
    N, NP = SIZES[name][:2]
    X_PAD, P_PAD = N, NP


def system():
    """terms[i] = list of (coef, a, b, [x factors]) of equation i, in table order."""
    eqs = []
    for i in range(N):
        if NAME == "coupled_quadrics_8x8":
            t = [(1, P_PAD, P_PAD, [i, i]),
                 (-1, i, i, []),
                 (1, 8, P_PAD, [(i + 1) % N, (i + 3) % N]),
                 (1, 9, P_PAD, [(i + 2) % N])]
            if i in (0, 4):
                t.append((1, 8, 9, [(i + 5) % N, (i + 6) % N, (i + 7) % N]))
        elif NAME == "dense_quadrics_6x6":
            t = [(1, P_PAD, P_PAD, [i, i]), (-1, i, i, [])] + [(1, N, P_PAD, sorted([i, j])) for j in range(N) if j != i]
        elif i < 6:
            t = [(1, P_PAD, P_PAD, [i, i]), (-1, i, i, []), (1, 12, P_PAD, sorted([(i + 1) % N, (i + 6) % N]))]
        else:
            t = [(1, P_PAD, P_PAD, [i]), (-1, i, P_PAD, []), (1, 13, P_PAD, sorted([i - 6, (i + 1) % N]))]
        eqs.append(t)
    return eqs


def jacobian(eqs):
    """jac[(row, col)] = list of (coef, a, b, [x factors]): d/dx_col of every term of equation `row`, table order kept."""
    jac = {}
    for i, terms in enumerate(eqs):
        for c, a, b, xs in terms:
            for j in sorted(set(xs)):
                m = xs.count(j)
                rest = list(xs)
                rest.remove(j)
                jac.setdefault((i, j), []).append((c * m, a, b, rest))
    return jac


def tables(eqs, jac):
    hx_terms = max(len(v) for v in jac.values())
    ht_terms = max(len(t) for t in eqs)
    hx = np.zeros((N, hx_terms, 5, N), np.int64)            # [col][term][part][row]: coef, p_a, p_b, x_d, x_e
    hx[:, :, 1:3, :] = P_PAD
    hx[:, :, 3:5, :] = X_PAD
    for (i, j), lst in jac.items():
        for t, (c, a, b, xs) in enumerate(lst):
            xs = list(xs) + [X_PAD] * (2 - len(xs))
            hx[j, t, :, i] = [c, a, b, xs[0], xs[1]]
    ht = np.zeros((ht_terms, 6, N), np.int64)                # [term][part][row]: coef, p_a, p_b, x_d, x_e, x_f
    ht[:, 1:3, :] = P_PAD
    ht[:, 3:6, :] = X_PAD
    for i, terms in enumerate(eqs):
        for t, (c, a, b, xs) in enumerate(terms):
            xs = list(xs) + [X_PAD] * (3 - len(xs))
            ht[t, :, i] = [c, a, b, xs[0], xs[1], xs[2]]
    return hx, ht


def start_data(seed=20241):
    rng = np.random.RandomState(seed + N)
    a = (rng.uniform(0.7, 1.3, N) * np.exp(1j * rng.uniform(-np.pi, np.pi, N))).astype(np.complex64)
    sp = np.zeros(NP, np.complex64)
    sp[:N] = a
    k2 = N_SQUARES[NAME]
    sols = np.empty((1 << k2, N), np.complex64)
    for k in range(1 << k2):
        for i in range(N):
            sols[k, i] = -a[i] if (i < k2 and (k >> i) & 1) else a[i]
    return sp, sols


def target_params(n_hyp, seed=1):
    """[n_hyp][NP + 1] complex64 real-valued target parameters (index NP is the constant-one pad), deterministic."""
    rng = np.random.RandomState(seed)
    t = np.zeros((n_hyp, NP + 1), np.complex64)
    t[:, :N] = rng.uniform(0.6, 1.4, (n_hyp, N)).astype(np.float32)
    lim = {"coupled_quadrics_8x8": 0.45, "dense_quadrics_6x6": 0.3, "mixed_12x12": 0.4}[NAME]
    for k in range(N, NP):                                   # the coupling parameters (0 in the start system)
        t[:, k] = rng.uniform(-lim, lim, n_hyp).astype(np.float32)
    t[:, NP] = 1.0
    return t


def write_folder(path):
    eqs = system()
    jac = jacobian(eqs)
    hx, ht = tables(eqs, jac)
    sp, sols = start_data()
    os.makedirs(path, exist_ok=True)
    fmt = lambda v: "%.9g" % float(v)
    with open(os.path.join(path, "start_params.txt"), "w") as f:
        for v in sp:
            f.write("%s\t%s\n" % (fmt(v.real), fmt(v.imag)))
    with open(os.path.join(path, "start_sols.txt"), "w") as f:
        for v in sols.reshape(-1):
            f.write("%s\t%s\n" % (fmt(v.real), fmt(v.imag)))
    with open(os.path.join(path, "target_params.txt"), "w") as f:
        for v in target_params(1)[0, :NP]:
            f.write("%s\t%s\n" % (fmt(v.real), fmt(v.imag)))
    for name, arr in (("dHdx_indx.txt", hx), ("dHdt_indx.txt", ht)):
        with open(os.path.join(path, name), "w") as f:
            for row in arr.reshape(-1, N):
                f.write("\t".join(str(int(v)) for v in row) + "\t\n")
    with open(os.path.join(path, "gpuhc_settings.yaml"), "w") as f:
        f.write("""# Settings of the synthetic minimal problem "%s" (written by tools/make_synthetic_problem.py).
# Key names are the ones the reference's readers look up (CPU_HC_Solver.cpp:34-60, GPU_HC_Solver.cpp:36-70); values describe THIS system.

# sizes of the polynomial system and of its evaluation-index tables
Num_Of_Vars: %d
Num_Of_Params: %d
Num_Of_Tracks: %d
dHdx_Max_Terms: %d
dHdx_Max_Parts: 5
dHdt_Max_Terms: %d
dHdt_Max_Parts: 6
# leading unknowns that must become positive for a path to be kept (an extension of this repository: the reference's GPU kernels hard-code
# 8 depths for the trifocal problem, TrunPaths.cu:148-154); 0 switches pruning off
Num_Of_Depth_Vars: %d
# elimination-step update predicate of the compiled tracker (an extension of this repository, codegen/gen_eval.py): 1 forms it with & and
# without a divergent region, 0 with && and a branch; which one ptxas allocates better depends on the problem (DESIGN.md §3)
HC_Branch_Free_Update: %d

# identity
problem_name: %s
problem_print_out_name: %s (synthetic problem for the problem compiler)

# path tracker: step cap, Newton iterations per step, successes before the step doubles
GPUHC_Max_Steps: 80
GPUHC_Max_Correction_Steps: 3
GPUHC_Num_Of_Steps_to_Increase_Delta_t: 4

# keys the reference's solver objects insist on although a synthetic problem has no RANSAC data
Num_Of_GPUs: 1
Num_Of_Cores: 4
RANSAC_Dataset: Synthetic
Abort_RANSAC_by_Good_Sol: false
""" % (NAME, N, NP, 1 << N_SQUARES[NAME], hx.shape[1], ht.shape[0], SIZES[NAME][2], BRANCH_FREE_UPDATE[NAME], NAME, NAME.replace("_", " ")))
    return hx, ht, sp, sols


def load_folder(path):
    """numpy view of a problem folder: dict(start_sols[T,N] c64, start_params[NP] c64, dHdx_indx, dHdt_indx (flat int32), spec)."""
    sys.path.insert(0, ROOT)
    from trifocal_pose_estimation_using_improved_gpuhc_b200.codegen import gen_eval
    spec, hx, ht = gen_eval.read_problem_dir(path)
    sp = np.loadtxt(os.path.join(path, "start_params.txt"), dtype=np.float32).reshape(-1, 2)
    ss = np.loadtxt(os.path.join(path, "start_sols.txt"), dtype=np.float32).reshape(spec["n_tracks"], spec["n_vars"], 2)
    return dict(spec=spec, start_params=(sp[:, 0] + 1j * sp[:, 1]).astype(np.complex64), start_sols=(ss[..., 0] + 1j * ss[..., 1]).astype(np.complex64),
                dHdx_indx=hx.astype(np.int32), dHdt_indx=ht.astype(np.int32))


if __name__ == "__main__":
    for name in NAMES:
        select(name)
        out = os.path.join(ROOT, "problems", name)
        hx, ht, sp, sols = write_folder(out)
        print("wrote", out, "| dHdx", hx.shape, "dHdt", ht.shape, "| start solutions", sols.shape)
