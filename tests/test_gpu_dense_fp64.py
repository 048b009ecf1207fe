"""The dense-path kernels element by element against a float64 reference written from include/pcgnn_b200.h.

`pcg_tile_fwd` / `pcg_tile_train` (k_tile + k_wgrad), `pcg_dense_fwd` / `pcg_dense_bwd`, `pcg_center_*`,
`pcg_head_loss_*` and `pcg_encoder_*` are called through the C ABI with caller-chosen strides, offsets and pointers.

Two regimes:
* exact: every input (features, aggregates, weights, given gradients) is a small integer times a power of two. If
  every partial sum is a multiple of the grid g and sum |a*b| < 2^24 g, fp32 gives the exact result in any summation
  order. `_exact_mm` checks that condition on the reference itself, so a case cannot quietly stop being exact. Forward
  outputs and the gradients of pcg_dense_bwd / pcg_center_bwd / pcg_encoder_bwd must then equal the reference bit for
  bit (compared as values, so -0 == +0).
* bounded: where a softmax comes in (pcg_tile_train's gradients and loss, pcg_head_loss_*), every ReLU mask still
  matches the reference exactly, and each element is compared with a running absolute error bound propagated through
  the graph with Higham's gamma_k = k u / (1 - k u), u = 2^-24 (`train_bounds`). The CPU tests below show the bound
  is neither unsound (a float32 torch evaluation in another order passes it) nor toothless (dropping one batch row or
  chunk, counting a batch slice twice, reading agg row w instead of rep[w], or dropping the last real feature column
  fails at least one element of every bounded case).

The case matrix is chosen by launch-plan branch. `_tile_plan`, `_wgrad_plan`, `_pick_tm` / `_dense_splits` and the
k_tile phase task counts mirror the C functions of csrc/pcg_tile.cu / csrc/pcg_dense.cu at 148 SMs (B200), and
`test_case_matrix_reaches_every_branch` asserts the cases reach every branch; the parametrisation ids name them.
"""
import ctypes as C
import warnings

import numpy as np
import pytest

U = 2.0 ** -24
SMS = 148                      # the B200 the plan mirror assumes
POISON = 2.0 ** 20             # finite: rows that must not be read (NaN would vanish in fmaxf(x, 0))
SENT = -12345.0                # pre-fill of every output: shows each element is written
# |fp32 - exact| of dl = (softmax - onehot) / B is at most C_SOFTMAX * u / B: one of the two expf is exp(0) = 1, the
# other has <= 2 ulp error; the sum, the quotient, the subtraction of the label and the product with fl(1 / B) add
# one rounding each, and logit differences that need a 25th bit add < 0.25 u; 7.3 u + 2 u < 12 u.
C_SOFTMAX = 12
# per-target cross-entropy m + log(e0 + e1) - l_y: the log's argument carries <= 5 u, the log 1 ulp of a value
# below log 2, the two additions one rounding each of values below |l0| + |l1| + 1: below 16 u (|l0| + |l1| + 1).
C_LOSS = 16


def gamma(k):
    return k * U / (1.0 - k * U)


# ------------------------------------------------------------------------------------------------ plan mirrors
TILE_KC, TILE_NWC, TILE_MAX_STAGE, TILE_MAX_E, TILE_SMEM_MAX = 32, 8, 32, 256, 227 * 1024
WG_KC, WG_BUF_BYTES = 32, 48 * 1024


def _ld_pad(x):                                  # ld_pad()
    return x + ((4 - (x & 15)) & 15)


def _tile_smem_bytes(TM, F, R, E, mode, ns):    # tile_smem()
    Fp = (F + 3) & ~3
    K2p = Fp + R * E
    LDC, LDA, LDO = _ld_pad(K2p), _ld_pad(Fp), E + 4
    tpg = (TM // 8) * (E // 64)
    o = TM * LDC + R * TM * LDA + TM * LDO + (TM * LDO if mode == 2 else 0) + ns * TILE_KC * E
    o += 0 if tpg >= TILE_NWC else 2 * TILE_NWC * 16 * 32
    o += 2 * E + 2 * Fp + 4 + TM * 8 + 4 * TILE_MAX_STAGE
    return o * 4


def _tile_chunks(F, R, E, mode):                # tile_chunks()
    Fp = (F + 3) & ~3
    K2p = Fp + R * E
    return R * -(-2 * Fp // TILE_KC) + -(-K2p // TILE_KC) + (R * (E // TILE_KC) if mode == 2 else 0)


def _tile_plan(B, F, R, E, mode, sms=SMS):      # tile_plan(): (TM, ring depth) or None
    chunks = _tile_chunks(F, R, E, mode)
    for tm in (32, 16, 8):
        if tm > 8 and -(-B // tm) < sms - sms // 5:
            continue
        if (tm // 8) * (E // 64) > TILE_NWC or R * (tm // 8) * (E // 64) > 4 * TILE_NWC:
            continue
        ns = min(chunks, TILE_MAX_STAGE)
        while ns >= 3 and _tile_smem_bytes(tm, F, R, E, mode, ns) > TILE_SMEM_MAX:
            ns -= 1
        if _tile_smem_bytes(tm, F, R, E, mode, ns) > TILE_SMEM_MAX:
            continue
        return tm, ns
    return None


def _tile_supported(B, R, F, E, sms=SMS):       # pcg_tile_supported()
    if B <= 0 or R < 1 or R > 8 or F < 1 or E < 64 or E > TILE_MAX_E or E % 64:
        return False
    return _tile_plan(B, F, R, E, 2, sms) is not None


def _ksplit(ntask):                             # phase_k(): spare warps split K
    k = 1
    while k * 2 * ntask <= TILE_NWC:
        k *= 2
    return k


def _wgrad_plan(B, F, R, E, sms=SMS):           # wgrad_plan() + k_wgrad's choice of the single wait
    S = 8
    while S > 1 and -(-B // S) < 64:
        S >>= 1
    Fp = (F + 3) & ~3
    K2p = Fp + R * E

    def blocks(W):
        return (-(-K2p // W) + R * -(-2 * Fp // W)) * -(-E // W)

    W = 64 if blocks(64) * S >= sms else 32
    nbuf = WG_BUF_BYTES // (2 * WG_KC * (W + 4) * 4)
    nt = -(-(-(-B // S)) // WG_KC)               # chunks of the first (longest) slice
    return S, W, ("single" if nbuf > 2 and nt <= nbuf else "ring")


def _tile_branches(B, F, R, E, sms=SMS):
    """Every launch-plan branch pcg_tile_train takes for this shape."""
    tm, ns = _tile_plan(B, F, R, E, 2, sms)
    tpg = (tm // 8) * (E // 64)
    S, W, load = _wgrad_plan(B, F, R, E, sms)
    br = {f"TM{tm}", "resident" if _tile_chunks(F, R, E, 2) <= ns else "ring", f"S{S}", f"W{W}", f"wgrad-{load}"}
    for ntask in (R * tpg, tpg):                 # phase A (R relations side by side), phase B (combine)
        br.add(f"ksplit{_ksplit(ntask)}")
        br.add(f"tpw{-(-ntask // TILE_NWC)}")
    return br


def _pick_tm(M):                                # pick_tm()
    return 16 if M <= 2048 else 64


def _dense_splits(B, R, F, E):                  # dense_splits()
    Mw = max(F + R * E, 2 * F)
    tiles = -(-Mw // 64) * -(-E // 64) * (R + 1)
    s = -(-2 * 148 // tiles)
    s = min(s, -(-B // 64))
    return min(max(s, 1), 32)


def _dense_branches(B, F, R, E, ldf):
    """pcg_dense_fwd / pcg_dense_bwd kernels for this shape (all pointers 16-byte aligned)."""
    tm = _pick_tm(B)
    vec = tm == 16 and F % 4 == 0 and E % 4 == 0 and ldf % 4 == 0
    br = {"fwd-gemm_pv" if vec else ("fwd-gemm_p" if tm == 16 else "fwd-gemm64")}
    if F > E:
        br.add("copy_self")
    if B > 0:
        br.add("bwd-dH-gemm_p" if tm == 16 else "bwd-dH-gemm64")
    else:
        br.add("bwd-B0")
    br.add("bwd-wg-gemm_v" if F % 4 == 0 and E % 4 == 0 and ldf % 4 == 0 else "bwd-wg-gemm64")
    if 2 * F > F + R * E:
        br.add("bwd-Mw2F")
    return br


# ------------------------------------------------------------------------------------------------ case matrix
def _largest_tile_F(B, R, E):
    lo, hi = 1, 1
    while _tile_supported(B, R, hi * 2, E):
        hi *= 2
    lo, hi = hi, hi * 2
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if _tile_supported(B, R, mid, E) else (lo, mid)
    return lo


F_MAX_TILE = _largest_tile_F(64, 1, 64)

# (F, E, R, B, lambda, labels): labels "mix" | "zeros" | "ones"
TILE_CASES = [
    (1, 64, 1, 1, 2.0, "ones"), (3, 64, 2, 2, 2.0, "mix"), (4, 128, 1, 7, 0.0, "mix"), (5, 192, 3, 8, 2.0, "zeros"),
    (25, 64, 3, 9, 2.0, "mix"), (32, 256, 8, 126, 2.0, "mix"), (33, 128, 5, 127, 2.0, "mix"),
    (100, 192, 8, 252, 2.0, "mix"), (12, 64, 6, 253, 0.0, "mix"), (25, 128, 7, 504, 2.0, "mix"),
    (100, 256, 4, 505, 2.0, "mix"), (32, 64, 1, 1280, 2.0, "mix"), (32, 64, 1, 1281, 2.0, "mix"),
    (25, 64, 3, 1888, 2.0, "mix"), (25, 64, 3, 1889, 2.0, "mix"), (100, 128, 3, 3776, 2.0, "mix"),
    (100, 128, 3, 3777, 2.0, "mix"), (16, 64, 8, 3777, 2.0, "mix"), (100, 128, 3, 4096, 2.0, "mix"),
    (100, 256, 8, 4096, 2.0, "mix"), (F_MAX_TILE, 64, 1, 64, 2.0, "mix"),
]
# pcg_dense_fwd / pcg_dense_bwd: (F, E, R, B)
DENSE_CASES = [
    (3, 1, 1, 5), (12, 16, 3, 60), (5, 50, 2, 33), (100, 100, 1, 40), (32, 256, 8, 300), (33, 64, 3, 2049),
    (64, 16, 1, 100), (100, 50, 1, 3000), (25, 64, 3, 0), (F_MAX_TILE + 1, 64, 1, 64),
]


def _ldf(F):
    return ((F + 3) & ~3) + 8                    # wider than Fp: the padding the header asks for is zero


def _tile_id(c):
    F, E, R, B, lam, lab = c
    return f"F{F}-E{E}-R{R}-B{B}-lam{lam:g}-{lab}-" + "-".join(sorted(_tile_branches(B, F, R, E)))


def _dense_id(c):
    F, E, R, B = c
    return f"F{F}-E{E}-R{R}-B{B}-" + "-".join(sorted(_dense_branches(B, F, R, E, _ldf(F))))


REQUIRED_TILE = ({"TM8", "TM16", "TM32", "ksplit1", "ksplit2", "ksplit4", "ksplit8", "tpw1", "tpw2", "tpw3", "tpw4",
                  "resident", "ring", "S1", "S2", "S4", "S8", "W32", "W64", "wgrad-single", "wgrad-ring"})
REQUIRED_DENSE = {"fwd-gemm_pv", "fwd-gemm_p", "fwd-gemm64", "copy_self", "bwd-dH-gemm_p", "bwd-dH-gemm64", "bwd-B0",
                  "bwd-wg-gemm_v", "bwd-wg-gemm64", "bwd-Mw2F"}


# ------------------------------------------------------------------------------------------------ inputs
def _grid(x):
    """Largest power of two that divides every element of x (exact dyadic values)."""
    x = np.asarray(x, np.float64)
    nz = x[x != 0]
    if nz.size == 0:
        return np.inf
    m, e = np.frexp(nz)
    ints = np.abs(m * 2.0 ** 53).astype(np.int64)
    low = (ints & -ints).astype(np.float64)
    return float(np.min(np.ldexp(low, e - 53)))


def _exact_mm(a, b):
    """a @ b in float64, after checking that fp32 computes it exactly in any order."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    g = _grid(a) * _grid(b)
    if np.isfinite(g) and a.size and b.size:
        mag = np.abs(a) @ np.abs(b)
        assert mag.max(initial=0.0) < 2.0 ** 24 * g, f"inputs too large to stay exact: {mag.max()} vs {2**24 * g}"
    return a @ b


def _q(rng, shape, scale, lo=-2, hi=2):
    return (rng.integers(lo, hi + 1, size=shape) * scale).astype(np.float32)


class Case:
    """Inputs of one dense-path call in the exact regime, poison and padding included."""

    def __init__(self, F, E, R, B, lam=2.0, labels="mix", seed=0, dups=True):
        rng = np.random.default_rng(seed * 7919 + F * 131 + E * 17 + R * 3 + B)
        self.F, self.E, self.R, self.B, self.lam = F, E, R, B, float(lam)
        self.Fp = (F + 3) & ~3
        self.ldf, self.lda = _ldf(F), self.Fp + 4
        pool = max(1, (3 * B) // 4) if dups else max(B, 1)
        N = pool + 37
        perm = rng.permutation(N)
        nodes = perm[:pool]
        self.targets = (rng.choice(nodes, B) if dups else rng.permutation(nodes)[:B]).astype(np.int32)
        # features: sparse small integers / 4; rows of nodes outside the batch are poison
        feat = np.zeros((N, self.ldf), np.float32)
        feat[:, :F] = _q(rng, (N, F), 0.25) * (rng.random((N, F)) < 0.35)
        outside = np.setdiff1d(np.arange(N), self.targets)
        feat[outside, :F] = POISON
        self.feat = feat
        # aggregates: representatives (first occurrence of a target) carry rows, repeated targets are poison
        first = {}
        rep_i = np.array([first.setdefault(int(t), i) for i, t in enumerate(self.targets)], np.int32)
        self.rep = np.concatenate([r * B + rep_i for r in range(R)]).astype(np.int32)
        agg = np.zeros((R * B, self.lda), np.float32)
        agg[:, :F] = _q(rng, (R * B, F), 0.25) * (rng.random((R * B, F)) < 0.35)
        agg[self.rep != np.arange(R * B), :F] = POISON
        self.agg = agg
        self.w_intra = [_q(rng, (2 * F, E), 1 / 16) for _ in range(R)]
        self.w_inter = _q(rng, (F + R * E, E), 1 / 16)
        self.w_clf = _q(rng, (2, F), 1 / 16)
        self.b_clf = _q(rng, (2,), 1 / 64)
        self.w_head = _q(rng, (2, E), 1 / 16)
        y = {"mix": rng.integers(0, 2, B), "zeros": np.zeros(B), "ones": np.ones(B)}[labels]
        self.labels = y.astype(np.int64)
        self.d_out = _q(rng, (E, B), 1 / 8, -3, 3)          # given gradient of `out` for pcg_dense_bwd

    def agg_ldf(self):
        """agg with row stride ldf (pcg_dense_fwd / pcg_dense_bwd read agg with the feature stride)."""
        a = np.zeros((self.R * self.B, self.ldf), np.float32)
        a[:, :self.lda] = self.agg
        return a


def reference(c: Case):
    """float64 forward of the header's formulas; every product is checked to be exact in fp32."""
    F, R, B = c.F, c.R, c.B
    self_ = c.feat[c.targets, :F].astype(np.float64)
    X = [np.hstack([self_, c.agg[c.rep[r * B:(r + 1) * B], :F].astype(np.float64)]) for r in range(R)]
    h = [np.maximum(_exact_mm(X[r], c.w_intra[r]), 0.0) for r in range(R)]
    cat = np.hstack([self_] + h)
    Z = np.maximum(_exact_mm(cat, c.w_inter), 0.0)
    center = _exact_mm(np.hstack([self_, np.ones((B, 1))]), np.vstack([c.w_clf.T, c.b_clf[None, :]]))
    logits = _exact_mm(Z, c.w_head.T.astype(np.float64))
    return dict(self=self_, X=X, h=h, cat=cat, Z=Z, center=center, logits=logits)


def _softmax1(l):
    m = l.max(axis=1, keepdims=True)
    e = np.exp(l - m)
    return e[:, 1] / e.sum(axis=1), (m[:, 0] + np.log(e.sum(axis=1)))


def train_reference(c: Case, f=None, omega=None, agg_rows=None, drop_col=False):
    """float64 loss and every gradient of pcg_tile_train. omega: per-row multiplicity of the batch sums (1 = as the
    header says; the sensitivity test drops or repeats rows), agg_rows / drop_col: what the weight-gradient sums read."""
    B, R, E, F, lam = c.B, c.R, c.E, c.F, c.lam
    f = f or reference(c)
    y = c.labels
    p, lse_g = _softmax1(f["logits"])
    q, lse_c = _softmax1(f["center"])
    lg = lse_g - f["logits"][np.arange(B), y]
    ll = lse_c - f["center"][np.arange(B), y]
    dl1 = (p - y) / B
    dc1 = lam * (q - y) / B
    dl = np.stack([-dl1, dl1], 1)
    dc = np.stack([-dc1, dc1], 1)
    wh = c.w_head.astype(np.float64)
    W = c.w_inter.astype(np.float64)
    dZ = (dl @ wh) * (f["Z"] > 0)
    dH = [(dZ @ W[F + r * E:F + (r + 1) * E].T) * (f["h"][r] > 0) for r in range(R)]
    om = np.ones(B) if omega is None else omega
    X = f["X"]
    cat = f["cat"]
    if agg_rows is not None:
        X = [np.hstack([f["self"], c.agg[agg_rows[r * B:(r + 1) * B], :F].astype(np.float64)]) for r in range(R)]
    if drop_col:
        X = [x.copy() for x in X]
        for x in X:
            x[:, [F - 1, 2 * F - 1]] = 0.0
        cat = f["cat"].copy()
        cat[:, F - 1] = 0.0
    g = dict(loss=np.array([(lg.sum() + lam * ll.sum()) / B]),
             d_w_inter=cat.T @ (om[:, None] * dZ),
             d_w_head=dl.T @ (om[:, None] * f["Z"]),
             d_w_clf=dc.T @ (om[:, None] * f["self"]),
             d_b_clf=(om[:, None] * dc).sum(0))
    for r in range(R):
        g[f"d_w_intra{r}"] = X[r].T @ (om[:, None] * dH[r])
    g.update(dl1=dl1, dc1=dc1, dZ=dZ, dH=dH, lg=lg, ll=ll, p=p, q=q)
    return g


def train_bounds(c: Case, f, g):
    """Absolute error bound of every bounded output of pcg_tile_train, propagated from err(dl) = C_SOFTMAX u / B."""
    B, R, E, F, lam = c.B, c.R, c.E, c.F, c.lam
    e_dl = C_SOFTMAX * U / B
    e_dc = lam * C_SOFTMAX * U / B
    wh = np.abs(c.w_head.astype(np.float64)).sum(0)                      # |W_head|^T (1, 1)
    dl1, dc1 = np.abs(g["dl1"]), np.abs(g["dc1"])
    eZ = (f["Z"] > 0) * (wh[None, :] * (e_dl + gamma(2) * dl1[:, None]))
    W = np.abs(c.w_inter.astype(np.float64))
    gB = gamma(B + 1)
    b = dict(d_w_inter=np.abs(f["cat"]).T @ (eZ + gB * np.abs(g["dZ"])),
             d_w_head=np.abs(f["Z"]).sum(0)[None, :] * e_dl + gB * (np.stack([dl1, dl1], 1).T @ np.abs(f["Z"])),
             d_w_clf=np.abs(f["self"]).sum(0)[None, :] * e_dc + gB * (np.stack([dc1, dc1], 1).T @ np.abs(f["self"])),
             d_b_clf=np.full(2, B * e_dc + gB * dc1.sum()))
    for r in range(R):
        Wr = W[F + r * E:F + (r + 1) * E]
        eH = (f["h"][r] > 0) * (eZ @ Wr.T + gamma(E + 1) * (np.abs(g["dZ"]) @ Wr.T))
        b[f"d_w_intra{r}"] = np.abs(f["X"][r]).T @ (eH + gB * np.abs(g["dH"][r]))
    lg_err = C_LOSS * U * (np.abs(f["logits"]).sum(1) + 1)
    ll_err = C_LOSS * U * (np.abs(f["center"]).sum(1) + 1)
    b["loss"] = np.array([(lg_err.sum() + lam * ll_err.sum()) / B + gamma(B + 4) * (g["lg"].sum() + lam * g["ll"].sum()) / B])
    return b


BOUNDED = ("loss", "d_w_inter", "d_w_head", "d_w_clf", "d_b_clf")


def _bounded_keys(R):
    return BOUNDED + tuple(f"d_w_intra{r}" for r in range(R))


def _violations(got, ref, bound, keys):
    """{key: number of elements outside the bound} (NaN counts as outside)."""
    out = {}
    for k in keys:
        a = np.asarray(got[k], np.float64).reshape(np.shape(ref[k]))
        ok = np.abs(a - ref[k]) <= bound[k]
        if not ok.all():
            out[k] = int((~ok).sum())
    return out


def _mutations(c: Case):
    """The wrong answers a bounded case must reject: (name, train_reference kwargs)."""
    B = c.B
    S = _wgrad_plan(B, c.F, c.R, c.E)[0]
    per = -(-B // S)
    last = (B - 1) // per * per                  # first row of the last batch slice
    muts = []
    om = np.ones(B)
    om[B - 1] = 0
    muts.append(("drop the last row", dict(omega=om)))
    om = np.ones(B)
    om[0] = 0
    muts.append(("drop the first row", dict(omega=om)))
    om = np.ones(B)
    om[last + ((B - 1 - last) // WG_KC) * WG_KC:] = 0
    muts.append(("drop the last 32-row chunk", dict(omega=om)))
    om = np.ones(B)
    om[last:] = 2
    muts.append(("count the last batch slice twice", dict(omega=om)))
    if (c.rep != np.arange(c.R * B)).any():
        muts.append(("read agg row w instead of rep[w]", dict(agg_rows=np.arange(c.R * B))))
    muts.append(("drop the last real feature column", dict(drop_col=True)))
    return muts


# ------------------------------------------------------------------------------------------------ CPU tests
def test_case_matrix_reaches_every_branch():
    """At 148 SMs the tile cases reach every k_tile / k_wgrad plan branch and the dense cases every pcg_dense kernel."""
    got_t = set().union(*(_tile_branches(B, F, R, E) for F, E, R, B, _, _ in TILE_CASES))
    got_d = set().union(*(_dense_branches(B, F, R, E, _ldf(F)) for F, E, R, B in DENSE_CASES))
    missing = sorted((REQUIRED_TILE - got_t) | (REQUIRED_DENSE - got_d))
    assert not missing, f"branches no case reaches: {missing}"
    for F, E, R, B, _, _ in TILE_CASES:
        assert _tile_supported(B, R, F, E), (F, E, R, B)
    assert not _tile_supported(64, 1, F_MAX_TILE + 1, 64)
    # the B boundaries of tile_plan / wgrad_plan sit where the mirror says
    assert _tile_plan(1888, 25, 3, 64, 2)[0] == 8 and _tile_plan(1889, 25, 3, 64, 2)[0] == 16
    assert _tile_plan(3776, 100, 3, 128, 2)[0] == 16 and _tile_plan(3777, 100, 3, 128, 2)[0] == 32
    assert [_wgrad_plan(b, 32, 1, 64)[0] for b in (126, 127, 252, 253, 504, 505)] == [1, 2, 2, 4, 4, 8]
    assert [_wgrad_plan(b, 32, 1, 64)[2] for b in (1280, 1281)] == ["single", "ring"]


@pytest.mark.parametrize("case", TILE_CASES, ids=_tile_id)
def test_bounds_admit_fp32_in_another_order_and_reject_wrong_sums(case):
    """A float32 torch CPU evaluation of the same math passes every bound; each mutation of the reference fails at
    least one element."""
    import torch

    F, E, R, B, lam, lab = case
    c = Case(F, E, R, B, lam, lab)
    f = reference(c)
    g = train_reference(c, f)
    bnd = train_bounds(c, f, g)
    keys = _bounded_keys(R)
    # float32 torch: matmuls in BLAS order, torch softmax / log_softmax
    t = {k: torch.from_numpy(np.asarray(v, np.float32)) for k, v in
         dict(cat=f["cat"], Z=f["Z"], logits=f["logits"], center=f["center"], self=f["self"]).items()}
    y = torch.from_numpy(c.labels)
    sm = torch.softmax(t["logits"], 1)
    sc = torch.softmax(t["center"], 1)
    oh = torch.nn.functional.one_hot(y, 2).float()
    dl = (sm - oh) / B
    dc = lam * (sc - oh) / B
    wh = torch.from_numpy(c.w_head)
    W = torch.from_numpy(c.w_inter)
    dZ = (dl @ wh) * (t["Z"] > 0)
    got = dict(loss=(torch.nn.functional.cross_entropy(t["logits"], y) +
                     lam * torch.nn.functional.cross_entropy(t["center"], y)).numpy().reshape(1),
               d_w_inter=(t["cat"].T @ dZ).numpy(), d_w_head=(dl.T @ t["Z"]).numpy(),
               d_w_clf=(dc.T @ t["self"]).numpy(), d_b_clf=dc.sum(0).numpy())
    for r in range(R):
        dH = (dZ @ W[F + r * E:F + (r + 1) * E].T) * torch.from_numpy((f["h"][r] > 0))
        got[f"d_w_intra{r}"] = (torch.from_numpy(np.asarray(f["X"][r], np.float32)).T @ dH).numpy()
    assert not _violations(got, g, bnd, keys)
    weak = []
    for name, kw in _mutations(c):
        bad = train_reference(c, f, **kw)
        if not _violations(bad, g, bnd, keys):
            weak.append(name)
    assert not weak, f"the bound of this case is too weak to catch: {weak}"


def test_exact_inputs_stay_exact_at_the_largest_shapes():
    """Inputs in {-2..2}/4 and weights in {-2..2}/16 stay exact at F = 100, R = 8, E = 256 and at C3's shape; the
    sparse features leave headroom of more than 70x below the fp32 limit in the combine."""
    for F, E, R, B in ((100, 256, 8, 512), (100, 128, 3, 512)):
        c = Case(F, E, R, B)
        f = reference(c)
        mag = np.abs(f["cat"]) @ np.abs(c.w_inter.astype(np.float64))
        assert mag.max() * 70 < 2.0 ** 24 * _grid(f["cat"]) * _grid(c.w_inter)


# ------------------------------------------------------------------------------------------------ GPU helpers
def _torch():
    import torch

    return torch


def _lib():
    from pcgnn_b200 import _lib as L

    return L


def _dev(a):
    torch = _torch()
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _buf(shape, offset=0, dtype=None):
    """Sentinel-filled device tensor of `shape` starting `offset` floats into its allocation."""
    torch = _torch()
    n = int(np.prod(shape))
    return torch.full((n + offset,), SENT, dtype=dtype or torch.float32, device="cuda")[offset:].view(*shape)


def _ptrs(ts):
    return (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def _np(t):
    return t.detach().cpu().numpy().astype(np.float64)


def _assert_equal(name, got, ref):
    got = np.asarray(got, np.float64).reshape(np.shape(ref))
    bad = got != ref
    assert not bad.any(), f"{name}: {int(bad.sum())} of {bad.size} elements differ, first at " \
                          f"{np.argwhere(bad)[0].tolist()}: {got[bad][0]} vs {np.asarray(ref)[bad][0]}"


def _assert_bounded(got, ref, bound, keys):
    v = _violations(got, ref, bound, keys)
    if v:
        k = next(iter(v))
        a = np.asarray(got[k], np.float64).reshape(np.shape(ref[k]))
        i = np.argmax(np.abs(a - ref[k]) - bound[k])
        raise AssertionError(f"outside the bound: {v}; {k} flat {i}: got {a.flat[i]} ref {ref[k].flat[i]} "
                             f"bound {bound[k].flat[i]}")


def _check_sms():
    sms = _lib().lib().pcg_device_sms()
    if sms != SMS:
        warnings.warn(f"device has {sms} SMs, the plan mirror assumes {SMS}: which branch a case reaches is not checked")
        return False
    return True


class Dev:
    """Device copies of a Case."""

    def __init__(self, c: Case):
        self.c = c
        self.feat = _dev(c.feat)
        self.targets = _dev(c.targets)
        self.agg = _dev(c.agg)
        self.agg_ldf = _dev(c.agg_ldf())
        self.rep = _dev(c.rep)
        self.w_intra = [_dev(w) for w in c.w_intra]
        self.w_inter = _dev(c.w_inter)
        self.w_clf = _dev(c.w_clf)
        self.b_clf = _dev(c.b_clf)
        self.w_head = _dev(c.w_head)
        self.labels = _dev(c.labels)

    def tile_fwd(self, keep_cat=True, center=True, w_clf=True, rep=True):
        L, c = _lib(), self.c
        out = _buf((c.E, c.B))
        cen = _buf((c.B, 2)) if center else None
        cat = _buf((c.B, c.F + c.R * c.E)) if keep_cat else None
        rc = L.lib().pcg_tile_fwd(self.feat.data_ptr(), c.ldf, c.F, self.targets.data_ptr(), c.B, c.R, c.E,
                                  self.agg.data_ptr(), c.lda, L.ptr(self.rep if rep else None), _ptrs(self.w_intra),
                                  self.w_inter.data_ptr(), L.ptr(self.w_clf) if w_clf else None,
                                  L.ptr(self.b_clf) if w_clf else None, int(keep_cat), out.data_ptr(), L.ptr(cen),
                                  L.ptr(cat), L.stream_ptr())
        L.check(rc, "pcg_tile_fwd")
        return out, cen, cat

    def dense_fwd(self):
        L, c = _lib(), self.c
        out = _buf((c.E, c.B))
        cat = _buf((c.B, c.F + c.R * c.E))
        rc = L.lib().pcg_dense_fwd(self.feat.data_ptr(), c.ldf, c.F, self.targets.data_ptr(), c.B, c.R, c.E,
                                   self.agg_ldf.data_ptr(), self.rep.data_ptr(), _ptrs(self.w_intra),
                                   self.w_inter.data_ptr(), cat.data_ptr(), out.data_ptr(), L.stream_ptr())
        L.check(rc, "pcg_dense_fwd")
        return out, cat

    def dense_bwd(self, cat, out, d_out):
        L, c = _lib(), self.c
        d_intra = [_buf((2 * c.F, c.E), 1 + r % 3) for r in range(c.R)]
        d_inter = _buf((c.F + c.R * c.E, c.E), 2)
        n = int(L.lib().pcg_dense_bwd_scratch_floats(c.B, c.R, c.F, c.E))
        scratch = _buf((n,))
        rc = L.lib().pcg_dense_bwd(c.ldf, c.F, c.B, c.R, c.E, self.agg_ldf.data_ptr(), self.rep.data_ptr(),
                                   self.w_inter.data_ptr(), cat.data_ptr(), out.data_ptr(), d_out.data_ptr(),
                                   _ptrs(d_intra), d_inter.data_ptr(), scratch.data_ptr(), L.stream_ptr())
        L.check(rc, "pcg_dense_bwd")
        return d_intra, d_inter

    def tile_train(self, logits=True, center=True):
        L, c = _lib(), self.c
        out = _buf((c.E, c.B))
        cen = _buf((c.B, 2)) if center else None
        lg = _buf((c.B, 2)) if logits else None
        loss = _buf((1,), 3)
        d_intra = [_buf((2 * c.F, c.E), 1 + r % 3) for r in range(c.R)]
        d_inter = _buf((c.F + c.R * c.E, c.E), 1)
        d_clf = _buf((2, c.F), 2)
        d_bclf = _buf((2,), 3)
        d_head = _buf((2, c.E), 1)
        n = int(L.lib().pcg_tile_scratch_floats(c.B, c.R, c.F, c.E))
        scratch = _buf((n,))
        rc = L.lib().pcg_tile_train(self.feat.data_ptr(), c.ldf, c.F, self.targets.data_ptr(), c.B, c.R, c.E,
                                    self.agg.data_ptr(), c.lda, self.rep.data_ptr(), _ptrs(self.w_intra),
                                    self.w_inter.data_ptr(), self.w_clf.data_ptr(), self.b_clf.data_ptr(),
                                    self.w_head.data_ptr(), self.labels.data_ptr(), c.lam, out.data_ptr(), L.ptr(cen),
                                    L.ptr(lg), loss.data_ptr(), _ptrs(d_intra), d_inter.data_ptr(), d_clf.data_ptr(),
                                    d_bclf.data_ptr(), d_head.data_ptr(), scratch.data_ptr(), 0, L.stream_ptr())
        L.check(rc, "pcg_tile_train")
        g = dict(loss=loss, d_w_inter=d_inter, d_w_head=d_head, d_w_clf=d_clf, d_b_clf=d_bclf)
        g.update({f"d_w_intra{r}": d for r, d in enumerate(d_intra)})
        return out, cen, lg, g


# ------------------------------------------------------------------------------------------------ GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("case", TILE_CASES, ids=_tile_id)
def test_tile_kernels_match_float64(case):
    """pcg_tile_fwd (both cat modes, with and without center / w_clf), pcg_dense_fwd on the same inputs, pcg_dense_bwd
    from the exact cat, and pcg_tile_train: forward outputs bit-exact, cross-path bit-identical, gradients bounded."""
    torch = _torch()
    F, E, R, B, lam, lab = case
    c = Case(F, E, R, B, lam, lab)
    L = _lib().lib()
    if _check_sms():
        assert L.pcg_tile_supported(B, R, F, E) == 1
        assert L.pcg_tile_supported(B, R, F + 1, E) == int(_tile_supported(B, R, F + 1, E))
    f = reference(c)
    d = Dev(c)
    out, cen, cat = d.tile_fwd(keep_cat=True)
    _assert_equal("tile_fwd out", _np(out), f["Z"].T)
    _assert_equal("tile_fwd center", _np(cen), f["center"])
    _assert_equal("tile_fwd cat", _np(cat), f["cat"])
    out0, cen0, cat0 = d.tile_fwd(keep_cat=False, center=False, w_clf=False)
    assert cen0 is None and cat0 is None
    assert torch.equal(out0, out)
    out1, cen1, _ = d.tile_fwd(keep_cat=False, center=True)
    assert torch.equal(out1, out) and torch.equal(cen1, cen)
    # the fallback GEMMs give the same bits
    dout, dcat = d.dense_fwd()
    assert torch.equal(dout, out) and torch.equal(dcat, cat)
    # pcg_dense_bwd, the autograd backward of pcg_tile_fwd, on exact inputs
    d_out = _dev(c.d_out)
    d_intra, d_inter = d.dense_bwd(cat, out, d_out)
    dZ = c.d_out.T.astype(np.float64) * (f["Z"] > 0)
    W = c.w_inter.astype(np.float64)
    _assert_equal("dense_bwd d_w_inter", _np(d_inter), _exact_mm(f["cat"].T, dZ))
    for r in range(R):
        dH = _exact_mm(dZ, W[F + r * E:F + (r + 1) * E].T) * (f["h"][r] > 0)
        _assert_equal(f"dense_bwd d_w_intra{r}", _np(d_intra[r]), _exact_mm(f["X"][r].T, dH))
    # the training form
    tout, tcen, tlog, g = d.tile_train()
    assert torch.equal(tout, out) and torch.equal(tcen, cen)
    _assert_equal("tile_train logits", _np(tlog), f["logits"])
    ref = train_reference(c, f)
    _assert_bounded({k: _np(v) for k, v in g.items()}, ref, train_bounds(c, f, ref), _bounded_keys(R))
    # logits / center NULL, same gradients
    tout2, _, _, g2 = d.tile_train(logits=False, center=False)
    assert torch.equal(tout2, out)
    for k in g:
        assert torch.equal(g[k], g2[k]), k


@pytest.mark.gpu
def test_tile_fwd_without_agg_rep_reads_row_w():
    """agg_rep = NULL: item w reads agg row w (no repeated targets)."""
    c = Case(25, 128, 3, 300, dups=False)
    f = reference(c)
    out, cen, cat = Dev(c).tile_fwd(rep=False)
    _assert_equal("out", _np(out), f["Z"].T)
    _assert_equal("cat", _np(cat), f["cat"])


@pytest.mark.gpu
def test_largest_tile_F_and_the_next_one_falls_back():
    L = _lib().lib()
    assert L.pcg_tile_supported(64, 1, F_MAX_TILE, 64) == 1
    assert L.pcg_tile_supported(64, 1, F_MAX_TILE + 1, 64) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("case", DENSE_CASES, ids=_dense_id)
def test_dense_gemms_match_float64(case):
    """pcg_dense_fwd (cat, out) and pcg_dense_bwd (every weight gradient) bit-exact; at B = 0 the gradients are
    overwritten with zeros."""
    F, E, R, B = case
    c = Case(F, E, R, B)
    d = Dev(c)
    W = c.w_inter.astype(np.float64)
    torch = _torch()
    if B == 0:
        cat, out, d_out = _buf((1, F + R * E)), _buf((E, 1)), _buf((E, 1))
        d.agg_ldf = _buf((1, c.ldf))                 # R * B = 0 rows; the pointers must still be real
        d_intra, d_inter = d.dense_bwd(cat, out, d_out)
        assert not torch.count_nonzero(d_inter) and all(not torch.count_nonzero(x) for x in d_intra)
        return
    f = reference(c)
    out, cat = d.dense_fwd()
    _assert_equal("dense_fwd out", _np(out), f["Z"].T)
    _assert_equal("dense_fwd cat", _np(cat), f["cat"])
    d_intra, d_inter = d.dense_bwd(cat, out, _dev(c.d_out))
    dZ = c.d_out.T.astype(np.float64) * (f["Z"] > 0)
    _assert_equal("d_w_inter", _np(d_inter), _exact_mm(f["cat"].T, dZ))
    for r in range(R):
        dH = _exact_mm(dZ, W[F + r * E:F + (r + 1) * E].T) * (f["h"][r] > 0)
        _assert_equal(f"d_w_intra{r}", _np(d_intra[r]), _exact_mm(f["X"][r].T, dH))
    if _check_sms():
        assert int(_lib().lib().pcg_dense_bwd_scratch_floats(B, R, F, E)) == \
            B * E + B * R * E + _dense_splits(B, R, F, E) * ((F + R * E) * E + R * 2 * F * E) + 64


@pytest.mark.gpu
@pytest.mark.parametrize("F,B", [(1, 1), (5, 9), (25, 33), (100, 1000), (257, 4097)])
def test_center_head_matches_float64(F, B):
    """pcg_center_fwd / pcg_center_bwd bit-exact; the backward runs twice on one ticket and scratch."""
    L = _lib()
    c = Case(F, 64, 1, B)
    d = Dev(c)
    f = reference(c)
    cen = _buf((B, 2))
    L.check(L.lib().pcg_center_fwd(d.feat.data_ptr(), c.ldf, F, d.targets.data_ptr(), B, d.w_clf.data_ptr(),
                                   d.b_clf.data_ptr(), cen.data_ptr(), L.stream_ptr()), "pcg_center_fwd")
    _assert_equal("center", _np(cen), f["center"])
    rng = np.random.default_rng(F + B)
    g = _q(rng, (B, 2), 1 / 8, -3, 3)
    dg = _dev(g)                                    # device buffers stay referenced until the kernels have run
    scratch = _buf((int(L.lib().pcg_head_scratch_floats(B, F, 64)),))
    ticket = _torch().zeros(1, dtype=_torch().int32, device="cuda")
    for _ in range(2):
        dw, db = _buf((2, F), 1), _buf((2,), 3)
        L.check(L.lib().pcg_center_bwd(d.feat.data_ptr(), c.ldf, F, d.targets.data_ptr(), B, dg.data_ptr(),
                                       dw.data_ptr(), db.data_ptr(), scratch.data_ptr(), ticket.data_ptr(),
                                       L.stream_ptr()), "pcg_center_bwd")
        _assert_equal("d_w", _np(dw), _exact_mm(g.T, f["self"]))
        _assert_equal("d_b", _np(db), g.astype(np.float64).sum(0))
    assert int(ticket.item()) == 0


def _head_inputs(E, B, scale, labels, seed):
    rng = np.random.default_rng(seed)
    if scale is None:
        emb = np.maximum(_q(rng, (E, B), 1 / 4), 0)
        w = _q(rng, (2, E), 1 / 16)
        center = _q(rng, (B, 2), 1 / 16, -8, 8)
    else:                                          # logits and center scores of exactly +-scale
        emb = np.zeros((E, B), np.float32)
        emb[0] = scale * rng.choice([-1, 1], B)
        emb[1] = scale * rng.choice([-1, 1], B)
        emb[2:] = _q(rng, (E - 2, B), 1 / 4)
        w = np.zeros((2, E), np.float32)
        w[0, 0] = w[1, 1] = 1
        center = (scale * rng.choice([-1, 1], (B, 2))).astype(np.float32)
    y = {"mix": rng.integers(0, 2, B), "zeros": np.zeros(B), "ones": np.ones(B)}[labels].astype(np.int64)
    return emb, w, center, y


@pytest.mark.gpu
@pytest.mark.parametrize("E,B,lam,labels,scale", [
    (64, 1, 2.0, "ones", None), (64, 33, 0.0, "mix", None), (128, 1000, 2.0, "zeros", None),
    (256, 4097, 2.0, "mix", None), (64, 300, 2.0, "mix", 100.0), (16, 300, 2.0, "mix", 1e4), (5, 65, 2.0, "ones", 1e4)])
def test_head_loss_matches_float64(E, B, lam, labels, scale):
    """pcg_head_loss_fwd / _bwd: logits bit-exact; probabilities, loss and gradients within the bound; logits of
    +-100 and +-1e4 give a finite loss. Both calls run twice on one ticket and scratch."""
    torch = _torch()
    L = _lib()
    emb, w, center, y = _head_inputs(E, B, scale, labels, E + B)
    logits = _exact_mm(emb.T, w.T)
    p, lse_g = _softmax1(logits)
    q, lse_c = _softmax1(center.astype(np.float64))
    lg = lse_g - logits[np.arange(B), y]
    ll = lse_c - center[np.arange(B), y]
    loss = (lg.sum() + lam * ll.sum()) / B
    e_loss = (C_LOSS * U * ((np.abs(logits).sum(1) + 1).sum() + lam * (np.abs(center).sum(1) + 1).sum())) / B \
        + gamma(B + 4) * (lg.sum() + lam * ll.sum()) / B
    demb, dw_, dcen, dy = _dev(emb), _dev(w), _dev(center), _dev(y)
    scratch = _buf((int(L.lib().pcg_head_scratch_floats(B, 1, E)),))
    ticket = torch.zeros(1, dtype=torch.int32, device="cuda")
    d_loss = _dev(np.ones(1, np.float32))
    dl1 = (p - y) / B
    dc1 = lam * (q - y) / B
    e_dl = C_SOFTMAX * U / B
    aw = np.abs(w.astype(np.float64)).sum(0)
    ref_demb = np.outer(w[1].astype(np.float64) - w[0], dl1)
    ref_dw = np.stack([-dl1, dl1]) @ emb.T.astype(np.float64)
    b_demb = aw[:, None] * (e_dl + gamma(2) * np.abs(dl1)[None, :])
    b_dw = np.abs(emb).sum(1)[None, :] * e_dl + gamma(B + 1) * (np.stack([np.abs(dl1)] * 2) @ np.abs(emb.T))
    for _ in range(2):
        lo, p1, q1, ls = _buf((B, 2)), _buf((B,)), _buf((B,)), _buf((1,), 1)
        L.check(L.lib().pcg_head_loss_fwd(demb.data_ptr(), E, B, dw_.data_ptr(), dcen.data_ptr(),
                                          dy.data_ptr(), lam, lo.data_ptr(), p1.data_ptr(), q1.data_ptr(),
                                          ls.data_ptr(), scratch.data_ptr(), ticket.data_ptr(), L.stream_ptr()),
                "pcg_head_loss_fwd")
        _assert_equal("logits", _np(lo), logits)
        assert np.isfinite(_np(ls)).all()
        _assert_bounded(dict(loss=_np(ls), p=_np(p1), q=_np(q1)), dict(loss=np.array([loss]), p=p, q=q),
                        dict(loss=np.array([e_loss]), p=np.full(B, C_SOFTMAX * U), q=np.full(B, C_SOFTMAX * U)),
                        ("loss", "p", "q"))
        d_emb, d_cen, d_w = _buf((E, B)), _buf((B, 2), 1), _buf((2, E), 3)
        L.check(L.lib().pcg_head_loss_bwd(demb.data_ptr(), E, B, dw_.data_ptr(), dy.data_ptr(), p1.data_ptr(),
                                          q1.data_ptr(), lam, d_loss.data_ptr(), d_emb.data_ptr(), d_cen.data_ptr(),
                                          d_w.data_ptr(), scratch.data_ptr(), ticket.data_ptr(), L.stream_ptr()),
                "pcg_head_loss_bwd")
        _assert_bounded(dict(d_emb=_np(d_emb), d_cen=_np(d_cen), d_w=_np(d_w)),
                        dict(d_emb=ref_demb, d_cen=np.stack([-dc1, dc1], 1), d_w=ref_dw),
                        dict(d_emb=b_demb, d_cen=np.full((B, 2), lam * e_dl), d_w=b_dw), ("d_emb", "d_cen", "d_w"))
    assert int(ticket.item()) == 0


def _enc_max_F(E, self_cat):
    """Largest F whose pcg_encoder_fwd / _bwd tiles fit the 200 KB the encoder asks for."""
    F = 1
    while True:
        Fin = 2 * (F + 1) if self_cat else F + 1
        if max(E * Fin + 32 * (Fin + 1), E * 33 + 32 * (Fin + 1)) * 4 > 200 * 1024:
            return F
        F += 1


@pytest.mark.gpu
@pytest.mark.parametrize("F,E,B,self_cat", [(3, 64, 1, False), (25, 64, 100, True), (25, 64, 1025, False),
                                            (7, 16, 33, True), (_enc_max_F(64, True), 64, 70, True),
                                            (_enc_max_F(64, False), 64, 40, False)])
def test_encoder_matches_float64(F, E, B, self_cat):
    """pcg_encoder_fwd / _bwd bit-exact with and without the self concat, with F_in not a multiple of 4 and at the
    shared-memory limit; the backward runs twice on one ticket and scratch."""
    torch = _torch()
    L = _lib()
    c = Case(F, E, 1, B, dups=False)
    d = Dev(c)
    self_ = c.feat[c.targets, :F].astype(np.float64)
    X = np.hstack([self_, c.agg[:B, :F]]) if self_cat else c.agg[:B, :F].astype(np.float64)
    rng = np.random.default_rng(F * E + B)
    w = _q(rng, (E, X.shape[1]), 1 / 16)
    ref = np.maximum(_exact_mm(w, X.T), 0.0)
    dwt = _dev(w)
    out = _buf((E, B))
    featp = d.feat.data_ptr() if self_cat else None
    tgtp = d.targets.data_ptr() if self_cat else None
    L.check(L.lib().pcg_encoder_fwd(d.agg.data_ptr(), c.lda, featp, c.ldf, tgtp, F, dwt.data_ptr(), B, E,
                                    out.data_ptr(), L.stream_ptr()), "pcg_encoder_fwd")
    _assert_equal("encoder out", _np(out), ref)
    d_out = _q(rng, (E, B), 1 / 8, -3, 3)
    ddo = _dev(d_out)
    scratch = _buf((int(L.lib().pcg_encoder_scratch_floats(B, X.shape[1], E)),))
    ticket = torch.zeros(1, dtype=torch.int32, device="cuda")
    for _ in range(2):
        dw = _buf((E, X.shape[1]), 1)
        L.check(L.lib().pcg_encoder_bwd(d.agg.data_ptr(), c.lda, featp, c.ldf, tgtp, F, B, E, out.data_ptr(),
                                        ddo.data_ptr(), dw.data_ptr(), scratch.data_ptr(), ticket.data_ptr(),
                                        L.stream_ptr()), "pcg_encoder_bwd")
        _assert_equal("encoder d_w", _np(dw), _exact_mm(d_out * (ref > 0), X))
    assert int(ticket.item()) == 0
