"""An independent float64 statement of the hmmsearch pipeline that ITSxpress runs (SURVEY.md Appendix A.1-A.5).

TEST INFRASTRUCTURE ONLY.  Written from the appendix, not from oracle/ora_hmm.c or search.cu: it shares no code and
no operation order with either, so it catches a formulation mistake the oracle and the kernels would share (an entry
or exit term, a length model set up for the wrong L, a null2 that is not HMMER's, a score bookkeeping rule).

Numerics: Forward and Backward run in float64 scaled odds (every row divided by its largest value, the logs of the
factors kept per row); MSV runs in the same integer (byte) arithmetic that defines it; everything else is float64.
Each DP is vectorised over a batch of targets of one profile (rows beyond a target's length are frozen), and the
serial D->D chain of a row is one product with a precomputed transfer matrix, i.e. (I - T_DD)^-1 restricted to the
chain.

Every threshold decision records its margin (distance of the float64 value from the threshold), so that a test can
tell a near-tie, where fp32 rounding may legitimately decide the other way, from a real disagreement.
"""
import math

import numpy as np

LN2 = math.log(2.0)
OMEGA = 1.0 / 256.0
RT1, RT2, RT3 = 0.25, 0.10, 0.20
MM, MI, MD, IM, II, DM, DD = range(7)

# residue codes: A C G T, then the IUPAC codes R Y M K S W H B V D N (X = N, U = T)
_SYM = "ACGTRYMKSWHBVDN"
MEMBERS = [(0,), (1,), (2,), (3,), (0, 2), (1, 3), (0, 1), (2, 3), (1, 2), (0, 3), (0, 1, 3), (1, 2, 3),
           (0, 1, 2), (0, 2, 3), (0, 1, 2, 3)]
NCODE = len(MEMBERS)
_MAP = np.full(256, 255, np.uint8)
for _i, _c in enumerate(_SYM):
    _MAP[ord(_c)] = _MAP[ord(_c.lower())] = _i
for _c, _v in (("U", 3), ("X", 14)):
    _MAP[ord(_c)] = _MAP[ord(_c.lower())] = _v


def digitize(ascii_bytes):
    a = _MAP[np.frombuffer(bytes(ascii_bytes), np.uint8)]
    if (a == 255).any():
        raise ValueError("illegal residue character")
    return a


def _member_mean(v4):
    """v4: [..., 4] values of the canonical residues -> [..., NCODE] means over each code's members."""
    return np.stack([v4[..., list(m)].mean(axis=-1) for m in MEMBERS], axis=-1)


# ---------------------------------------------------------------------------------------------------------------
# HMMER3/f text parser (A.1)
class Profile:
    pass


def _prob(tok):
    return 0.0 if tok == "*" else math.exp(-float(tok))


def parse_hmm(path, prefixes=None):
    """Profiles whose NAME starts with one of `prefixes` (all if None), in file order."""
    out = []
    with open(path) as f:
        lines = f.read().split("\n")
    i = 0
    while i < len(lines):
        if not lines[i].startswith("HMMER3"):
            i += 1
            continue
        p = Profile()
        while not lines[i].startswith("HMM "):
            t = lines[i].split()
            if t[0] == "NAME":
                p.name = t[1]
            elif t[0] == "LENG":
                p.M = int(t[1])
            elif t[:3] == ["STATS", "LOCAL", "MSV"]:
                p.msv_mu, p.msv_lambda = float(t[3]), float(t[4])
            elif t[:3] == ["STATS", "LOCAL", "VITERBI"]:
                p.vit_mu, p.vit_lambda = float(t[3]), float(t[4])
            elif t[:3] == ["STATS", "LOCAL", "FORWARD"]:
                p.tau, p.lam = float(t[3]), float(t[4])
            i += 1
        i += 2                                           # "HMM A C G T" + the transition-name line
        t = lines[i].split()
        p.compo = np.array([_prob(x) for x in t[1:5]]) if t[0] == "COMPO" else np.full(4, 0.25)
        if t[0] == "COMPO":
            i += 1
        i += 1                                           # node-0 insert emissions
        M = p.M
        p.t = np.zeros((M + 1, 7))
        p.t[0] = [_prob(x) for x in lines[i].split()]
        i += 1
        p.mat = np.zeros((M + 1, 4))
        for k in range(1, M + 1):
            t = lines[i].split()
            assert int(t[0]) == k
            p.mat[k] = [_prob(x) for x in t[1:5]]
            p.t[k] = [_prob(x) for x in lines[i + 2].split()]
            i += 3
        assert lines[i].strip() == "//"
        if prefixes is None or any(p.name.startswith(q) for q in prefixes):
            out.append(_configure(p))
        i += 1
    return out


# ---------------------------------------------------------------------------------------------------------------
# local profile configuration (A.3) and the MSV byte profile (A.4 step 1)
def _configure(p):
    M, t = p.M, p.t
    occ = np.zeros(M + 1)
    occ[1] = t[0, MI] + t[0, MM]
    for k in range(2, M + 1):
        occ[k] = occ[k - 1] * (t[k - 1, MM] + t[k - 1, MI]) + (1.0 - occ[k - 1]) * t[k - 1, DM]
    Z = sum(occ[k] * (M - k + 1) for k in range(1, M + 1))
    p.tBM = occ[1:] / Z                                   # [M], node k at index k-1
    tr = t[1:].copy()                                     # node k's transitions at index k-1; node M exits only
    tr[M - 1] = 0.0
    p.tMM, p.tMI, p.tMD, p.tIM, p.tII, p.tDM, p.tDD = (tr[:, c].copy() for c in range(7))
    odds4 = p.mat[1:] / 0.25                              # [M, 4]
    p.odds4 = odds4
    with np.errstate(divide="ignore"):
        msc4 = np.log(odds4)
    p.msc = _member_mean(msc4).T                          # [NCODE, M]: degenerate code = mean of members' scores
    p.emit = np.exp(p.msc)                                # Forward / Backward match odds
    p.n2odds = _member_mean(odds4).T                      # null2: plain mean of member odds
    # D->D chain as one product.  Forward: D[:, k] = sum_{j<k} Mn[:, j] * tMD[j] * prod_{j<l<k} tDD[l]
    G = np.zeros((M, M))
    for j in range(M):
        acc = p.tMD[j]
        for k in range(j + 1, M):
            G[j, k] = acc
            acc *= p.tDD[k]
    p.Gf = G
    # Backward: D[:, k] = sum_{j>=k} a[:, j] * prod_{k<=l<j} tDD[l]
    H = np.zeros((M, M))
    for k in range(M):
        acc = 1.0
        for j in range(k, M):
            H[j, k] = acc
            acc *= p.tDD[j]
    p.Hb = H
    # MSV byte profile, third-bits
    p.scale_b = 3.0 / LN2
    maxsc = max(0.0, float(np.max(msc4)))
    p.bias_b = _byteify(-maxsc)
    p.base_b = 190
    p.tbm_b = _byteify(math.log(2.0 / (M * (M + 1.0))))
    p.tec_b = _byteify(math.log(0.5))
    cost = np.empty((NCODE, M), np.int64)
    for x in range(NCODE):
        for k in range(M):
            v = -_roundf(p.scale_b * p.msc[x, k])
            cost[x, k] = 255 if v > 255 - p.bias_b else int(v) + p.bias_b
    p.msv_cost = cost
    # bias-filter composition model: emission odds, degenerate codes = mean of members
    p.bias_odds1 = _member_mean(p.compo / 0.25)
    return p


def _roundf(x):
    return math.floor(x + 0.5) if x >= 0 else -math.floor(-x + 0.5)


def _byteify(sc):
    v = -_roundf(3.0 / LN2 * sc)
    return 255 if v > 255 else int(v)


# ---------------------------------------------------------------------------------------------------------------
# statistics
def nullsc(L):
    if L == 0:
        return 0.0
    p1 = L / (L + 1.0)
    return L * math.log(p1) + math.log(1.0 - p1)


def gumbel_surv(x, mu, lam):
    y = lam * (x - mu)
    return -math.expm1(-math.exp(-y)) if y > -700 else 1.0


def exp_surv(x, tau, lam):
    return 1.0 if x < tau else math.exp(-lam * (x - tau))


def exp_logsurv(x, tau, lam):
    return 0.0 if x < tau else -lam * (x - tau)


def logsum(a, b):
    m = max(a, b)
    return m + math.log(math.exp(a - m) + math.exp(b - m))


# ---------------------------------------------------------------------------------------------------------------
# batches: a list of code arrays -> left-aligned [n, Lmax] matrix (padding code 0) and lengths
def _pad(seqs):
    L = np.array([len(s) for s in seqs], np.int64)
    X = np.zeros((len(seqs), max(1, int(L.max(initial=0)))), np.int64)
    for r, s in enumerate(seqs):
        X[r, :len(s)] = s
    return X, L


def msv_batch(p, seqs):
    """A.4 step 1 in byte arithmetic.  Returns (usc nats, overflow bool) per target."""
    X, L = _pad(seqs)
    n, M = len(seqs), p.M
    bias, base, tec, tbm = p.bias_b, p.base_b, p.tec_b, p.tbm_b
    tjb = np.array([_byteify(math.log(3.0 / (l + 3.0))) for l in L], np.int64)
    xJ = np.zeros(n, np.int64)
    xB = np.maximum(base - (tjb + tbm), 0)
    Mv = np.zeros((n, M), np.int64)
    ovf = np.zeros(n, bool)
    for i in range(int(L.max(initial=0))):
        live = (i < L) & ~ovf
        prev = np.concatenate([np.zeros((n, 1), np.int64), Mv[:, :-1]], axis=1)
        sv = np.minimum(np.maximum(prev, xB[:, None]) + bias, 255)
        sv = np.maximum(sv - p.msv_cost[X[:, i]], 0)
        xE = sv.max(axis=1)
        ovf |= live & (xE >= 255 - bias)
        xJn = np.maximum(xJ, np.maximum(xE - tec, 0))
        xBn = np.maximum(np.maximum(base, xJn) - (tjb + tbm), 0)
        Mv = np.where(live[:, None], sv, Mv)
        xJ = np.where(live, xJn, xJ)
        xB = np.where(live, xBn, xB)
    usc = ((xJ - tjb) - base) / p.scale_b - 3.0
    return np.where(ovf, np.inf, usc), ovf


def bias_batch(p, seqs):
    """A.4 step 2: the two-state composition HMM, scaled Forward in float64.  Returns filtersc (nats)."""
    X, L = _pad(seqs)
    n = len(seqs)
    L1 = p.M / 8.0
    t00, t01 = 400.0 / 401.0, 1.0 / 401.0
    t11, t10 = L1 / (L1 + 1.0), 1.0 / (L1 + 1.0)
    f0, f1 = np.full(n, 0.999), np.full(n, 0.001)
    logs = np.zeros(n)
    for i in range(int(L.max(initial=0))):
        live = i < L
        e1 = p.bias_odds1[X[:, i]]
        if i == 0:
            g0, g1 = f0, f1 * e1
        else:
            g0 = f0 * t00 + f1 * t10
            g1 = (f0 * t01 + f1 * t11) * e1
        s = g0 + g1
        f0 = np.where(live, g0 / s, f0)
        f1 = np.where(live, g1 / s, f1)
        logs += np.where(live, np.log(s), 0.0)
    return np.array([logs[r] + nullsc(int(L[r])) if L[r] > 0 else 0.0 for r in range(n)])


# ---------------------------------------------------------------------------------------------------------------
# Forward / Backward (A.3, A.4 steps 4-5), float64 scaled odds
def _lengthmodel(Lmodel, nj):
    Lm = np.asarray(Lmodel, np.float64)
    move = (2.0 + nj) / (Lm + 2.0 + nj)
    return move, 1.0 - move


def forward_batch(p, seqs, Lmodel, multihit, keep_cells=False):
    """Returns dict: sc [n] (nats), specials F[n, Lmax+1, 5] (E N J B C, scaled), cum[n, Lmax+1] (log of the row
    scale factors up to and including row i), and if keep_cells the scaled match / insert cells [n, Lmax+1, M]."""
    X, L = _pad(seqs)
    n, M, Lmax = len(seqs), p.M, int(L.max(initial=0))
    move, loop = _lengthmodel(Lmodel, 1 if multihit else 0)
    tEC, tEJ = (0.5, 0.5) if multihit else (1.0, 0.0)
    Mx, Ix, Dx = np.zeros((n, M)), np.zeros((n, M)), np.zeros((n, M))
    xN, xJ, xC, xE = np.ones(n), np.zeros(n), np.zeros(n), np.zeros(n)
    xB = move.copy()
    F = np.zeros((n, Lmax + 1, 5))
    cum = np.zeros((n, Lmax + 1))
    F[:, 0] = np.stack([xE, xN, xJ, xB, xC], 1)
    cells = (np.zeros((n, Lmax + 1, M)), np.zeros((n, Lmax + 1, M))) if keep_cells else None
    for i in range(1, Lmax + 1):
        live = i <= L
        e = p.emit[X[:, i - 1]]
        Mn = xB[:, None] * p.tBM[None, :]
        Mn[:, 1:] += Mx[:, :-1] * p.tMM[:-1] + Ix[:, :-1] * p.tIM[:-1] + Dx[:, :-1] * p.tDM[:-1]
        Mn *= e
        In = Mx * p.tMI + Ix * p.tII
        Dn = Mn @ p.Gf
        En = Mn.sum(1) + Dn.sum(1)
        Nn = xN * loop
        Jn = xJ * loop + En * tEJ
        Cn = xC * loop + En * tEC
        Bn = (Nn + Jn) * move
        s = np.maximum.reduce([En, Nn, Jn, Cn, Mn.max(1), In.max(1)])
        s = np.where(live & (s > 0), s, 1.0)
        w = live[:, None]
        Mx, Ix, Dx = np.where(w, Mn / s[:, None], Mx), np.where(w, In / s[:, None], Ix), np.where(w, Dn / s[:, None], Dx)
        xE, xN, xJ, xB, xC = (np.where(live, v / s, o) for v, o in ((En, xE), (Nn, xN), (Jn, xJ), (Bn, xB), (Cn, xC)))
        F[:, i] = np.stack([xE, xN, xJ, xB, xC], 1)
        cum[:, i] = cum[:, i - 1] + np.log(s)
        if keep_cells:
            cells[0][:, i], cells[1][:, i] = Mx, Ix
    last = cum[np.arange(n), L]
    with np.errstate(divide="ignore"):
        sc = last + np.log(F[np.arange(n), L, 4] * move)
    return dict(sc=sc, F=F, cum=cum, L=L, X=X, move=move, loop=loop, cells=cells)


def backward_batch(p, fw, multihit, keep_cells=False):
    """Backward over the same batch; returns specials Bk[n, Lmax+1, 5], cum[n, Lmax+1] (log of the row scale factors
    from row i to L) and sc = ln N(0).  With keep_cells, the scaled match / insert cells."""
    X, L, move, loop = fw["X"], fw["L"], fw["move"], fw["loop"]
    n, M, Lmax = len(L), p.M, int(L.max(initial=0))
    tEC, tEJ = (0.5, 0.5) if multihit else (1.0, 0.0)
    Mb, Ib, Db = np.zeros((n, M)), np.zeros((n, M)), np.zeros((n, M))
    bN, bJ, bC, bB, bE = (np.zeros(n) for _ in range(5))
    Bk = np.zeros((n, Lmax + 1, 5))
    cum = np.zeros((n, Lmax + 1))
    cells = (np.zeros((n, Lmax + 1, M)), np.zeros((n, Lmax + 1, M))) if keep_cells else None
    cum_next = np.zeros(n)
    hsum = p.Hb.sum(0)
    for i in range(Lmax, -1, -1):
        start, rec = (i == L), (i < L)
        # the last row: C -> T, E -> C; every M_k / D_k exits to E, M_k also through D_{k+1} ... D_M -> E
        Cs = move
        Es = Cs * tEC
        Ds = Es[:, None] * hsum[None, :]
        Ms = Es[:, None] + np.concatenate([Ds[:, 1:] * p.tMD[None, :-1], np.zeros((n, 1))], axis=1)
        # rows i < L
        xn = X[:, i] if i < X.shape[1] else np.zeros(n, np.int64)
        mp = p.emit[xn] * Mb                              # e_k(x_{i+1}) M_k(i+1)
        Br = mp @ p.tBM
        Jr = bJ * loop + Br * move
        Cr = bC * loop
        Er = Jr * tEJ + Cr * tEC
        Nr = bN * loop + Br * move
        mplus = np.concatenate([mp[:, 1:], np.zeros((n, 1))], axis=1)
        Dr = (mplus * p.tDM + Er[:, None]) @ p.Hb
        Ir = mplus * p.tIM + Ib * p.tII
        Dnext = np.concatenate([Dr[:, 1:], np.zeros((n, 1))], axis=1)
        Mr = mplus * p.tMM + Ib * p.tMI + Dnext * p.tMD + Er[:, None]
        z = np.zeros(n)
        vals = []
        for sv, rv, old in ((Es, Er, bE), (z, Nr, bN), (z, Jr, bJ), (z, Br, bB), (Cs, Cr, bC)):
            vals.append(np.where(start, sv, np.where(rec, rv, old)))
        w1, w2 = start[:, None], rec[:, None]
        Mn = np.where(w1, Ms, np.where(w2, Mr, Mb))
        In = np.where(w1, 0.0, np.where(w2, Ir, Ib))
        Dn = np.where(w1, Ds, np.where(w2, Dr, Db))
        act = start | rec
        s = np.maximum.reduce(vals + [Mn.max(1), In.max(1), Dn.max(1)])
        s = np.where(act & (s > 0), s, 1.0)
        Mb, Ib, Db = Mn / s[:, None], In / s[:, None], Dn / s[:, None]
        bE, bN, bJ, bB, bC = (v / s for v in vals)
        cum_next = np.where(start, np.log(s), np.where(rec, cum_next + np.log(s), cum_next))
        Bk[:, i] = np.stack([bE, bN, bJ, bB, bC], 1)
        cum[:, i] = cum_next
        if keep_cells:
            cells[0][:, i], cells[1][:, i] = Mb, Ib
    with np.errstate(divide="ignore"):
        sc = cum[:, 0] + np.log(Bk[:, 0, 1])
    return dict(sc=sc, Bk=Bk, cum=cum, cells=cells)


def decode_specials(fw, bw, r):
    """A.5 inputs for target r: btot, etot, mocc over rows 0..L (index 0 unused for mocc)."""
    L = int(fw["L"][r])
    F, cf, Bk, cb = fw["F"][r, :L + 1], fw["cum"][r, :L + 1], bw["Bk"][r, :L + 1], bw["cum"][r, :L + 1]
    tot = fw["sc"][r]
    w = np.exp(cf + cb - tot)                              # posterior weight of a (state, row) pair
    pB = F[:, 3] * Bk[:, 3] * w
    pE = F[:, 0] * Bk[:, 0] * w
    loop = fw["loop"][r]
    w1 = np.exp(cf[:-1] + cb[1:] - tot)
    emit = (F[:-1, 1] * Bk[1:, 1] + F[:-1, 2] * Bk[1:, 2] + F[:-1, 4] * Bk[1:, 4]) * loop * w1
    btot = np.zeros(L + 1)
    etot = np.zeros(L + 1)
    mocc = np.zeros(L + 1)
    btot[1:] = np.cumsum(pB[:-1])
    etot[1:] = np.cumsum(pE[1:])
    mocc[1:] = 1.0 - emit
    return btot, etot, mocc


def find_regions(btot, etot, mocc):
    """A.5 region scan.  Returns ([(i, j, multidomain)], min margin over every threshold comparison evaluated)."""
    L = len(mocc) - 1
    regs = []
    margin = math.inf
    i, triggered = -1, False
    for j in range(1, L + 1):
        if not triggered:
            v = mocc[j] - (btot[j] - btot[j - 1])
            margin = min(margin, abs(v - RT2))
            if v < RT2:
                i = j
            elif i == -1:
                i = j
            margin = min(margin, abs(mocc[j] - RT1))
            if mocc[j] >= RT1:
                triggered = True
        else:
            v = mocc[j] - (etot[j] - etot[j - 1])
            margin = min(margin, abs(v - RT2))
            if v < RT2:
                z = np.arange(i, j + 1)
                m3 = float(np.max(np.minimum(etot[z] - etot[i - 1], btot[j] - btot[z - 1])))
                margin = min(margin, abs(m3 - RT3))
                regs.append((i, j, m3 >= RT3))
                i, triggered = -1, False
    return regs, margin


def rescore_envelopes(p, items, chunk_cells=4_000_000):
    """Unihit rescoring (A.5) of envelopes given as (codes of the target, ienv, jenv) with 1-based inclusive
    coordinates.  Returns per item: envsc (nats), domcorrection (nats, not clamped), null2 odds by HMMER's direct
    formula and by the shortcut, and the largest row deviation of the decoded posteriors from 1."""
    out = [None] * len(items)
    order = sorted(range(len(items)), key=lambda r: items[r][2] - items[r][1])
    b0 = 0
    while b0 < len(order):
        b1 = b0 + 1
        while b1 < len(order) and (b1 + 1 - b0) * (items[order[b1]][2] - items[order[b1]][1] + 2) * p.M <= chunk_cells:
            b1 += 1
        idx = order[b0:b1]
        b0 = b1
        subs = [items[r][0][items[r][1] - 1:items[r][2]] for r in idx]
        Lfull = [len(items[r][0]) for r in idx]
        fw = forward_batch(p, subs, Lfull, multihit=False, keep_cells=True)
        bw = backward_batch(p, fw, multihit=False, keep_cells=True)
        for q, r in enumerate(idx):
            Ld = len(subs[q])
            tot = fw["sc"][q]
            cf, cb = fw["cum"][q, :Ld + 1], bw["cum"][q, :Ld + 1]
            w = np.exp(cf[1:] + cb[1:] - tot)
            pM = fw["cells"][0][q, 1:Ld + 1] * bw["cells"][0][q, 1:Ld + 1] * w[:, None]
            pI = fw["cells"][1][q, 1:Ld + 1] * bw["cells"][1][q, 1:Ld + 1] * w[:, None]
            F, Bk = fw["F"][q, :Ld + 1], bw["Bk"][q, :Ld + 1]
            w1 = np.exp(cf[:-1] + cb[1:] - tot) * fw["loop"][q]
            pN, pJ, pC = (F[:-1, c] * Bk[1:, c] * w1 for c in (1, 2, 4))
            rowsum = pM.sum(1) + pI.sum(1) + pN + pJ + pC
            mbar, ibar = pM.sum(0) / Ld, pI.sum(0) / Ld
            sbar = (pN.sum() + pJ.sum() + pC.sum()) / Ld
            direct4 = mbar @ p.odds4 + ibar.sum() + sbar                       # HMMER's p7_Null2_ByExpectation
            short4 = 1.0 + mbar @ (p.odds4 - 1.0)                             # the shortcut DESIGN.md section 2 uses
            direct, short = _member_mean(direct4), _member_mean(short4)
            dc = float(np.log(direct[subs[q]]).sum())
            out[r] = dict(envsc=float(tot), domcorrection=dc, null2=direct, null2_short=short,
                          rowdev=float(np.max(np.abs(rowsum - 1.0))), bwd_minus_fwd=float(bw["sc"][q] - tot))
    return out


# ---------------------------------------------------------------------------------------------------------------
# the whole pipeline for one profile over a set of targets
def search_profile(p, seqs, T=10.0, F1=1e-6, F3=1e-6, md_envelopes=None):
    """Every (target, profile) pair through A.4-A.5.  `md_envelopes(r, i, j)` returns the cluster envelopes
    (list of (ienv, jenv)) another implementation reported for a multidomain region, or None to rescore the region
    as one envelope (resolve_multidomain = 0).  Returns one dict per target."""
    n = len(seqs)
    res = [dict(L=len(s)) for s in seqs]
    usc, ovf = msv_batch(p, seqs)
    fsc = bias_batch(p, seqs)
    cand = []
    for r in range(n):
        L = len(seqs[r])
        d = res[r]
        d["usc"], d["overflow"] = float(usc[r]), bool(ovf[r])
        d["nullsc"] = nullsc(L)
        d["filtersc"] = float(fsc[r])
        if L == 0:
            d.update(pass_msv=False, pass_bias=False, pass_fwd=False, margin_msv=math.inf, margin_bias=math.inf)
            continue
        if ovf[r]:
            d["P_msv"], d["pass_msv"], d["margin_msv"] = 0.0, True, math.inf
            d["P_bias"], d["pass_bias"], d["margin_bias"] = 0.0, True, math.inf
        else:
            d["P_msv"] = gumbel_surv((usc[r] - d["nullsc"]) / LN2, p.msv_mu, p.msv_lambda)
            d["pass_msv"] = d["P_msv"] <= F1
            d["margin_msv"] = abs(math.log(max(d["P_msv"], 1e-300)) - math.log(F1))
            d["P_bias"] = gumbel_surv((usc[r] - fsc[r]) / LN2, p.msv_mu, p.msv_lambda)
            d["pass_bias"] = d["pass_msv"] and d["P_bias"] <= F1
            d["margin_bias"] = abs(math.log(max(d["P_bias"], 1e-300)) - math.log(F1))
        d["pass_fwd"] = False
        if d["pass_bias"]:
            cand.append(r)
    if not cand:
        return res
    fw = forward_batch(p, [seqs[r] for r in cand], [len(seqs[r]) for r in cand], multihit=True)
    keep = []
    for q, r in enumerate(cand):
        d = res[r]
        d["fwdsc"] = float(fw["sc"][q])
        d["P_fwd"] = exp_surv((d["fwdsc"] - d["filtersc"]) / LN2, p.tau, p.lam)
        d["pass_fwd"] = d["P_fwd"] <= F3
        d["margin_fwd"] = abs(math.log(d["P_fwd"]) - math.log(F3))
        if d["pass_fwd"]:
            keep.append(q)
    if not keep:
        return res
    fw2 = forward_batch(p, [seqs[cand[q]] for q in keep], [len(seqs[cand[q]]) for q in keep], multihit=True)
    bw2 = backward_batch(p, fw2, multihit=True)
    env_items, env_of = [], []
    for q2, q in enumerate(keep):
        r = cand[q]
        d = res[r]
        d["bcksc"] = float(bw2["sc"][q2])
        regs, d["margin_rt"] = find_regions(*decode_specials(fw2, bw2, q2))
        d["regions"] = regs
        d["doms"] = []
        for (i, j, multi) in regs:
            envs = md_envelopes(r, i, j) if (multi and md_envelopes is not None) else None
            resolved = envs is not None
            for (a, b) in (envs if resolved else [(i, j)]):
                d["doms"].append(dict(ienv=a, jenv=b, is_multidomain=bool(multi), resolved=resolved))
                env_items.append((seqs[r], a, b))
                env_of.append((r, len(d["doms"]) - 1))
    for (r, k), e in zip(env_of, rescore_envelopes(p, env_items)):
        res[r]["doms"][k].update(e)
    for q in keep:
        _scores(p, res[cand[q]], T)
    return res


def _scores(p, d, T):
    """A.4 steps 6-7 for one target that passed Forward."""
    L = d["L"]
    doms = d["doms"]
    for x in doms:
        Ld = x["jenv"] - x["ienv"] + 1
        x["dombias"] = logsum(0.0, math.log(OMEGA) + x["domcorrection"])
        x["bits"] = (x["envsc"] + (L - Ld) * math.log(L / (L + 3.0)) - (d["nullsc"] + x["dombias"])) / LN2
        x["lnP"] = exp_logsurv(x["bits"], p.tau, p.lam)
    if not doms:
        d["seq_score"], d["reported"], d["margin_T"] = -math.inf, False, math.inf
        return
    # the per-sequence null2 sum covers every envelope position once (simple-region envelopes do not overlap)
    seqbias = logsum(0.0, math.log(OMEGA) + sum(x["domcorrection"] for x in doms))
    seq_score = (d["fwdsc"] - (d["nullsc"] + seqbias)) / LN2
    used = [x for x in doms if x["envsc"] - x["domcorrection"] > 0.0]
    Ld = sum(x["jenv"] - x["ienv"] + 1 for x in used)
    ssum = sum(x["envsc"] for x in used) + (L - Ld) * math.log(L / (L + 3.0))
    sbias = logsum(0.0, math.log(OMEGA) + sum(x["domcorrection"] for x in used))
    sum_score = (ssum - (d["nullsc"] + sbias)) / LN2
    d["seq_score_fwd"], d["sum_score"] = seq_score, sum_score
    if Ld > 0 and sum_score > seq_score:
        seq_score = sum_score
    d["seq_score"] = seq_score
    d["lnP"] = exp_logsurv(seq_score, p.tau, p.lam)
    d["reported"] = seq_score >= T
    d["margin_T"] = abs(seq_score - T)
