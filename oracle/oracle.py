"""ctypes binding of the CPU oracle (oracle/_build/liblfold_oracle.so).  TEST INFRASTRUCTURE:
only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_build", "liblfold_oracle.so")
CLI = os.path.join(HERE, "_build", "lfold_oracle")
RLF = os.path.join(HERE, "_ref", "RNALfold")
_lib = None

# Tie-break mutants of the traceback (lfold_oracle.c, TB_*): each bit flips one "first match wins" rule.  Tests only:
# a corpus whose output changes under a bit contains ties that rule must break.
TIEBREAK = {
    "F3_LAST": 1 << 0,          # exterior scan: last k instead of first
    "F3_ORDER": 1 << 1,         # exterior scan, one k: (i+1,k) wins over (i,k)
    "HAIRPIN_LAST": 1 << 2,     # pair: two-loop tried before hairpin
    "LOOP_LAST": 1 << 3,        # two-loop scan: last (p,q) instead of first
    "ML_BEFORE_LOOP": 1 << 4,   # pair: multiloop closing tried before two-loop
    "MLC_LAST": 1 << 5,         # multiloop closing: last split k
    "MLC_VARIANT": 1 << 6,      # multiloop closing, one k: dangle variants in reverse order
    "FML_PEEL_5": 1 << 7,       # fML segment: peel the 5' base before the 3' base
    "FML_PAIR_ORDER": 1 << 8,   # fML segment: cij > ci1j1 > cij1 > ci1j
    "FML_SPLIT_LAST": 1 << 9,   # fML segment: last split k
}

# Energy perturbations (lfold_oracle_fold_pert, PERT_*): kind -> (code, index length).  fold(..., perturb=(kind, *index),
# delta=d) raises that term class by d dcal.  Tests only: a class whose raise changes the c matrix is the unique minimiser
# of some cell, where a kernel that computes it wrongly must differ from the oracle.
PERTURB = {
    "shape": (1, 3),            # (n1, n2, parity of j-i): every two-loop of that shape (stacks and bulges included)
    "ring": (2, 2),             # (s, d): every two-loop of n1+n2 = s closed by a pair on diagonal j-i = d
    "hairpin_size": (3, 1),     # (s,): every hairpin of s unpaired bases, after the log extrapolation of s > 30
    "stack": (4, 2),            # table entries: stack[t][t2], bulge[s], internal_loop[s], int11[t][t2][x][y], ...
    "bulge": (5, 1),
    "internal_loop": (6, 1),
    "int11": (7, 4),
    "int21": (8, 6),            # (n1, t, t2, x, y, z): int21[t][t2][x][y][z] as read by 1x2 loops with that n1 only
    "int22": (9, 6),
    "mismatchI": (10, 3),
    "mismatchH": (11, 3),
    "hairpin": (12, 1),
    "tetra": (13, 1),           # (k,): the k-th entry of the tetraloop list
}


def build():
    subprocess.run(["make", "-C", HERE, "all"], check=True, stdout=subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO):
            build()
        L = C.CDLL(SO)
        L.lfold_oracle_fold.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int]
        L.lfold_oracle_fold.restype = C.c_void_p
        L.lfold_oracle_fold_mut.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.lfold_oracle_fold_mut.restype = C.c_void_p
        L.lfold_oracle_fold_pert.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int]
        L.lfold_oracle_fold_pert.restype = C.c_void_p
        L.lfold_oracle_hairpin_energy.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int]
        L.lfold_oracle_hairpin_energy.restype = C.c_int
        L.lfold_oracle_free.argtypes = [C.c_void_p]
        for name in ("nhits", "total", "failed", "W"):
            getattr(L, "lfold_oracle_" + name).argtypes = [C.c_void_p]
            getattr(L, "lfold_oracle_" + name).restype = C.c_int
        for name in ("hit_start", "hit_energy"):
            getattr(L, "lfold_oracle_" + name).argtypes = [C.c_void_p, C.c_int]
            getattr(L, "lfold_oracle_" + name).restype = C.c_int
        L.lfold_oracle_hit_ss.argtypes = [C.c_void_p, C.c_int]
        L.lfold_oracle_hit_ss.restype = C.c_char_p
        L.lfold_oracle_conv.argtypes = [C.c_void_p]
        L.lfold_oracle_conv.restype = C.c_char_p
        for name in ("c", "m", "f3"):
            getattr(L, "lfold_oracle_" + name).argtypes = [C.c_void_p]
            getattr(L, "lfold_oracle_" + name).restype = C.POINTER(C.c_int)
        _lib = L
    return _lib


def fold(seq, span, matrices=False, tiebreak=0, perturb=None, delta=1):
    """-> dict(hits=[(ss, energy_dcal, start)], total=int[, c, m, f3]).  tiebreak: OR of TIEBREAK bits (0 = RNALfold);
    perturb: (kind, *index) of PERTURB, whose term class costs `delta` dcal more in this fold (None = RNALfold)."""
    L = lib()
    b = seq.encode() if isinstance(seq, str) else seq
    if perturb is None:
        r = L.lfold_oracle_fold_mut(b, len(b), span, 1 if matrices else 0, int(tiebreak))
    else:
        code, nidx = PERTURB[perturb[0]]
        if len(perturb) != 1 + nidx:
            raise ValueError("perturb %r: %s takes %d indices" % (perturb, perturb[0], nidx))
        idx = (C.c_int * 6)(*[int(v) for v in perturb[1:]])
        r = L.lfold_oracle_fold_pert(b, len(b), span, 1 if matrices else 0, int(tiebreak), code, idx, int(delta))
        if not r:
            raise ValueError("perturb %r: index out of range" % (perturb,))
    try:
        if L.lfold_oracle_failed(r):
            raise RuntimeError("oracle: backtrack failed")
        hits = [(L.lfold_oracle_hit_ss(r, k).decode(), L.lfold_oracle_hit_energy(r, k), L.lfold_oracle_hit_start(r, k))
                for k in range(L.lfold_oracle_nhits(r))]
        out = {"hits": hits, "total": L.lfold_oracle_total(r)}
        if matrices:
            n, W = len(b), L.lfold_oracle_W(r)
            out["c"] = np.ctypeslib.as_array(L.lfold_oracle_c(r), shape=(n + 2, W)).copy()
            out["m"] = np.ctypeslib.as_array(L.lfold_oracle_m(r), shape=(n + 2, W)).copy()
            out["f3"] = np.ctypeslib.as_array(L.lfold_oracle_f3(r), shape=(n + 4,)).copy()
        return out
    finally:
        L.lfold_oracle_free(r)


def hairpin_energy(seq, i, j):
    """Energy (dcal) of the hairpin closed by (i, j), 1-based, with the unmodified tables; 1000000 if (i, j) cannot pair."""
    b = seq.encode() if isinstance(seq, str) else seq
    return lib().lfold_oracle_hairpin_energy(b, len(b), int(i), int(j))


def fold_text(text, span, binary=None):
    """stdout of the oracle CLI (or of the reference's RNALfold when binary=RLF)."""
    if binary is None:
        if not os.path.exists(CLI):
            build()
        binary = CLI
    return subprocess.run([binary, "-L", str(span)], input=text.encode(), stdout=subprocess.PIPE, check=True).stdout.decode()


def have_rlf():
    return os.path.exists(RLF) and os.access(RLF, os.X_OK)
