"""Count-by-count replay of `pst_draw_counts` in fp64.  TEST INFRASTRUCTURE ONLY.

Every count of both samplers is a pure function of (seed, global cell, gene) and the count's fp32
parameters, through named Philox4x32-10 blocks (pst_counts.cu, pst_common.cuh).  This module replays
that function with the documented algorithm evaluated in fp64 and, for every count, returns the
interval [lo, hi] of the values the kernel can produce within its fp32 error model.  A count is
*determined* when lo == hi: whatever the rounding of the fp32 chain, the algorithm fixes it, so the
kernel must produce exactly that value.  Counts next to a decision (a cdf step, an acceptance test, the
floor in PTRS) are undetermined and only have to lie in [lo, hi].

Inputs are the fp32 parameters exactly as the kernel forms them (mu, theta, q, a, log2p0 and route from
the hook `pst_nb_params_f32`, which runs the kernel's own __device__ functions).  The uniforms the kernel
forms from Philox words with exact IEEE operations (u01, the stretched inversion uniform, the 64-bit
far-tail uniform) are reproduced bit for bit in NumPy; everything that goes through a MUFU instruction or
an fp32 chain is given an error bound (constants below, from the PTX ISA accuracy tables, times a safety
factor of two).

Plain NumPy, vectorised over counts.  Nothing under prosstt_b200/ imports it.
"""
import numpy as np

from oracle.prosstt_oracle import philox4x32_10

TAG_COUNT, TAG_QUAD = 0x200, 0x201
FLAG_DOMAIN, FLAG_CLAMPED = 1, 4
INT_MAX = 2147483647
CLAMP_AT = 2147483520.0

# paths a count can take (for per-regime statistics)
P_DOMAIN, P_HEAD, P_SEARCH, P_TAIL, P_MIX_SMALL, P_MIX_FAR, P_PTRS, P_NORMAL = range(8)
PATH_NAMES = ["domain", "inv_head", "inv_search", "inv_far_tail", "mix_lambda<10", "mix_lambda<10_far",
              "mix_ptrs", "mix_normal"]

E24 = 2.0 ** -24
SAFETY = 2.0
# PTX ISA accuracy of the approximate instructions the kernels use (relative unless noted)
EX2_REL = 2.0 ** -22              # ex2.approx.ftz.f32: 2 ulp
RCP_REL = 2.0 ** -23              # rcp.approx.ftz.f32: 1 ulp
RSQRT_REL = 2.0 ** -22            # rsqrt.approx.ftz.f32: 2 ulp
LG2_ABS = 2.0 ** -22              # lg2.approx.ftz.f32: absolute for x in [0.5, 2], relative beyond
COS_ABS = 2.0 ** -21.4            # __cosf on [-pi, pi]
# first k at which the hybrid search leaves the t_k = P(k) k! form for the P(k) form with a + q k
# advanced by additions: HY_KFIX_N - 1 + HY_STAGE2 = 33 by default; 24 covers every kept variant
K_SWITCH = 24

_TOP = np.float32(0.99999994)


# ---------------------------------------------------------------------------------------- Philox
def philox_block(seed, c0, cell, tag, block):
    """Block `block` of Philox4x32-10 keyed by the seed, counter (c0, cell lo, tag << 16 | cell hi,
    block): the counter layout of every stream of pst_draw_counts.  -> (n, 4) uint32."""
    c0, cell, block = np.broadcast_arrays(np.asarray(c0, np.uint64), np.asarray(cell, np.uint64),
                                          np.asarray(block, np.uint64))
    ctr = np.stack([c0 & 0xFFFFFFFF, cell & 0xFFFFFFFF, (np.uint64(tag) << np.uint64(16)) | (cell >> np.uint64(32)),
                    block & 0xFFFFFFFF], axis=-1).astype(np.uint32)
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    return philox4x32_10(ctr, np.broadcast_to(key, ctr.shape[:-1] + (2,)))


def u01(w):
    """pst::u01 bit for bit: fminf(fmaf((float)w, 2^-32, 2^-33), 1 - 2^-24).  (float)w rounds to
    nearest, the product by 2^-32 is exact and so the FFMA is one rounding of an fp64-exact sum."""
    fw = np.asarray(w, np.uint32).astype(np.float32).astype(np.float64)
    return np.minimum((fw * 2.0 ** -32 + 2.0 ** -33).astype(np.float32), _TOP)


# ----------------------------------------------------------------------- inversion of a cdf
def _first_crossings(U, p0, ratio, rho, eta_scale, stop_tail=None, kmax=1 << 16, cdf_form=False):
    """For each row: the computed cdf C(k) = sum_{j<=k} P(j), P(0) = p0, P(k+1) = P(k) ratio(k) in fp64,
    and its error band err(k) = sum_j P(j) rho(j) + eta_scale sum_j |C(j) - U| (the fp32 accumulation of
    d = cdf - u; with `cdf_form` the cdf itself is accumulated and C(j) replaces |C(j) - U|).  Returns
    (point, lo, hi, top_above): point = #{k : C(k) < U}, lo = first k with C + err >= U, hi = first k with
    C - err >= U.  `stop_tail` (mu) enables the far tail's redraw test: rows whose cdf never reaches U
    get top_above = +1 when U is above the top beyond the band, 0 when undecidable."""
    n = U.shape[0]
    point = np.full(n, -1, np.int64); lo = np.full(n, -1, np.int64); hi = np.full(n, -1, np.int64)
    top = np.full(n, -1, np.int64)            # -1: crossing found, +1: redraw, 0: undetermined
    idx = np.arange(n)
    P = p0.astype(np.float64).copy(); C = P.copy()
    serr = P * rho(0, idx); sabs = eta_scale * (C if cdf_form else np.abs(C - U) + U)
    k = 0
    while idx.size:
        err = serr + sabs
        newp = (point[idx] < 0) & (C >= U)
        point[idx[newp]] = k
        newl = (lo[idx] < 0) & (C + err >= U)
        lo[idx[newl]] = k
        done = C - err >= U
        hi[idx[done]] = k
        if stop_tail is not None:
            dead = ~done & (P < 1e-30) & (k > stop_tail[idx]) | (k >= kmax)
            if dead.any():
                d = idx[dead]
                top[d] = np.where(lo[d] < 0, 1, 0)         # even C + err stays below U: redraw
                done = done | dead
        elif k >= kmax:                                    # the band swallows the top of the cdf
            hi[idx[~done]] = INT_MAX
            done = done | True
        keep = ~done
        idx, P, C, serr, sabs = idx[keep], P[keep], C[keep], serr[keep], sabs[keep]
        U = U[keep]
        P = P * ratio(k, idx)
        C = C + P
        k += 1
        serr = serr + P * rho(k, idx)
        # a rounding of d + P(k) is at most half an ulp of the result and never more than P(k) itself
        sabs = sabs + np.minimum(eta_scale * (C if cdf_form else np.abs(C - U)), 2.0 * P)
    return point, lo, hi, top


def nb_inversion(U, q, a, log2p0, far, mu):
    """The hybrid sampler's inversion of the NB cdf for uniforms U (fp64, exact): the cdf of the NB with
    the kernel's fp32 q and a (r = a/q) times the common factor 2^(log2p0 - log2 P(0)) the kernel's fp32
    log2 P(0) carries (both known exactly from the hook).  The remaining error per pmf term j:
      ex2 of P(0), 2 roundings per t_{k+1} = t_k (a + q k) and the rounding of 1/k! (3 per term);
      beyond K_SWITCH the P(k) form: rounding of a q k + a, 1/(k+1) (1 ulp of an MUFU rcp in developer
      builds), the product and P(k) itself (5 per term) and the drift of a + q k advanced by additions,
      at most m (m+1)/2 roundings after m terms.
    `far`: the far-tail path accumulates the cdf in fp64 (no eta); the head and drains accumulate
    d = cdf - u in fp32, one rounding of |d| per term plus the first FFMA.  Returns point, lo, hi, top."""
    q = q.astype(np.float64); a = a.astype(np.float64)
    log2p0_exact = (a / q) * np.log1p(-q) / np.log(2.0)          # log2 (1-q)^r, r = a/q
    cfac = np.exp2(log2p0.astype(np.float64) - log2p0_exact)
    p0 = np.exp2(log2p0.astype(np.float64))                         # = cfac * P(0)

    def ratio(k, idx):
        return (a[idx] + q[idx] * k) / (k + 1.0)

    def rho(k, idx):
        m = max(k - K_SWITCH, 0)
        return SAFETY * (EX2_REL + (3 * min(k, K_SWITCH) + 2 + 5 * m + m * (m + 1) / 2) * E24)

    eta = 0.0 if far else SAFETY * E24
    return _first_crossings(U, p0, ratio, rho, eta, stop_tail=mu.astype(np.float64) if far else None,
                            kmax=(1 << 16) if far else 4096)


def poisson_inversion(U, lam_lo, lam_hi, fp64):
    """Poisson(lambda) by inversion (both mixture kernels, lambda < 10) for lambda in [lam_lo, lam_hi]:
    the Poisson cdf falls with lambda, so lo comes from lam_lo and hi from lam_hi.  fp32 path: exp_fast(-lam)
    (ex2 plus the rounding of -lam log2 e), per term a MUFU rcp or an fp32 power and 2-3 roundings, fp32
    accumulation of the cdf.  fp64 path (the far tail): exp and products in fp64."""
    def run(lam):
        lam = lam.astype(np.float64)

        def ratio(k, idx):
            return lam[idx] / (k + 1.0)

        if fp64:
            def rho(k, idx):
                return 1e-14 * (k + 1)
            eta = 1e-16
        else:
            def rho(k, idx):
                return SAFETY * (EX2_REL + lam[idx] * 2 * E24 + (4 * k + 2) * E24 + k * RCP_REL)
            eta = SAFETY * E24
        return _first_crossings(U, np.exp(-lam), ratio, rho, eta, kmax=4096, cdf_form=True)
    pt_lo, lo, _, _ = run(lam_lo)
    _, _, hi, _ = run(lam_hi)
    return pt_lo, lo, hi


# --------------------------------------------------------------------------- gamma (Marsaglia-Tsang)
def _gamma_attempt(mu, th, w):
    """One Marsaglia-Tsang attempt from block w (x, y Box-Muller, z acceptance, w boost).  Returns
    (accept, certain, lam_lo, lam_hi): `certain` is False when a decision lies inside its error margin."""
    mu = mu.astype(np.float64); th = th.astype(np.float64)
    r = mu / th
    lt1 = r < 1.0
    certain = np.abs(r - 1.0) > 4 * E24 + RCP_REL
    shape = np.where(lt1, r + 1.0, r)
    d = shape - 1.0 / 3.0
    c = 1.0 / np.sqrt(9.0 * d)
    u1 = u01(w[:, 0]).astype(np.float64)
    lg = np.log2(u1)
    rad2 = -2.0 * np.log(u1)
    drad2 = 2 * np.log(2.0) * LG2_ABS * np.maximum(1.0, np.abs(lg)) + rad2 * 4 * E24
    sr = np.sqrt(rad2)
    arg = 2 * np.pi * u01(w[:, 1]).astype(np.float64) - np.pi
    cs = np.cos(arg)
    xn = sr * cs
    dxn = SAFETY * (np.abs(cs) * (drad2 / (2 * sr) + sr * (RSQRT_REL + 3 * E24)) + sr * (COS_ABS + 8 * E24 * 4))
    e = c * xn
    de = np.abs(c) * dxn + np.abs(e) * (RSQRT_REL + E24)
    t = 1.0 + e
    v = t ** 3
    u = u01(w[:, 2]).astype(np.float64)
    x2 = xn * xn
    ok_t = t > 0
    certain &= np.abs(t) > de + 2 * E24
    sq = 1.0 - 0.0331 * x2 * x2
    dsq = 0.0331 * 4 * np.abs(xn) ** 3 * dxn + 4 * E24 * (1 + 0.0331 * x2 * x2)
    squeeze = u < sq
    sq_certain = np.abs(u - sq) > dsq
    # h = 0.5 x^2 + d (1 - v + log v), by series in e where that cancels
    with np.errstate(invalid="ignore", divide="ignore"):
        hs = d * e ** 4 * (-0.75 + e * (0.6 + e * (-0.5 + e * (3 / 7 + e * (-0.375 + e * (1 / 3 + e * (-0.3 + e * (
            3 / 11 + e * (-0.25 + e * 3 / 13)))))))))
        hl = 0.5 * x2 + d * (1.0 - v + np.log(np.where(v > 0, v, 1.0)))
        h = np.where(np.abs(e) < 0.05, hs, hl)
        dh = (np.abs(xn) * dxn + 3 * d * np.abs(t * t - 1.0 / np.where(t != 0, t, 1.0)) * de
              + SAFETY * 8 * E24 * (0.5 * x2 + d * (np.abs(v) + 1.0 + np.abs(np.log(np.where(v > 0, v, 1.0)))))
              + SAFETY * 2 * RSQRT_REL * 0.5 * x2)
        lu = np.log(u)
        dlu = SAFETY * (np.log(2.0) * LG2_ABS * np.maximum(1.0, np.abs(np.log2(u))) + np.abs(lu) * E24)
        logt = lu < h
        log_certain = np.abs(lu - h) > dh + dlu
    accept = ok_t & (squeeze | logt)
    # certainty: the t > 0 test always decides; the squeeze only when t > 0; the log test only when the
    # squeeze fails (or is itself uncertain)
    need_log = ok_t & (~squeeze | ~sq_certain)
    certain &= ~ok_t | sq_certain | log_certain
    certain &= ~need_log | log_certain | (squeeze & sq_certain)
    # lambda = theta d max(v, 0) boost, boost = U^(1/r) for r < 1
    uw = u01(w[:, 3]).astype(np.float64)
    barg = np.log(uw) / np.where(lt1, r, 1.0)
    boost = np.where(lt1, np.exp(barg), 1.0)
    dboost = np.where(lt1, np.log(2.0) * LG2_ABS * np.maximum(1.0, np.abs(np.log2(uw))) / r
                      + np.abs(barg) * (RCP_REL + 3 * E24) + EX2_REL, 0.0)
    lam = th * d * np.maximum(v, 0.0) * boost
    rel = SAFETY * (3 * de / np.maximum(np.abs(t), 1e-30) + 12 * E24 + RSQRT_REL) + SAFETY * dboost
    return accept, certain, lam * (1 - rel), lam * (1 + rel)


# ------------------------------------------------------------------------------------------ PTRS
def _lgfact(k):
    from scipy.special import gammaln
    return gammaln(k + 1.0)


def _ptrs_trial(lam_lo, lam_hi, wu, wv):
    """One PTRS trial (Hoermann 1993) from words (wu, wv) for lambda in [lam_lo, lam_hi].  Returns
    (accept, certain, k_lo, k_hi)."""
    U = (u01(wu) - np.float32(0.5)).astype(np.float32)
    V = u01(wv)
    us = (np.float32(0.5) - np.abs(U)).astype(np.float32)
    U = U.astype(np.float64); us64 = us.astype(np.float64); V64 = V.astype(np.float64)

    def consts(lam):
        slam = np.sqrt(lam)
        b = 2.53 * slam + 0.931
        a = 0.02483 * b - 0.059
        return b, a, np.log(1.1239 + 1.1328 / (b - 3.4)), 0.9277 - 3.6224 / (b - 2.0)

    bl, al, lial, vrl = consts(lam_lo)
    bh, ah, liah, vrh = consts(lam_hi)
    argl = (2 * al / us64 + bl) * U + lam_lo + 0.43
    argh = (2 * ah / us64 + bh) * U + lam_hi + 0.43
    e32 = SAFETY * ((np.abs((2 * ah / us64 + bh) * U)) * (RCP_REL + RSQRT_REL + 6 * E24) + (lam_hi + 1) * 2 * E24)
    k_lo = np.floor(np.minimum(argl, argh) - e32)
    k_hi = np.floor(np.maximum(argl, argh) + e32)
    evr = SAFETY * (RCP_REL + RSQRT_REL + 4 * E24) + np.abs(vrh - vrl)
    vr = 0.5 * (vrl + vrh)
    big_us = us >= np.float32(0.07)
    acc1 = big_us & (V64 <= vr)
    cert1 = ~big_us | (np.abs(V64 - vr) > evr)
    rej2 = (k_hi < 0) | ((us < np.float32(0.013)) & (V > us))
    cert2 = (k_lo >= 0) | (k_hi < 0)
    # log test for both ends of the k range
    lhs_l = np.log(V64) + lial - np.log(al / (us64 * us64) + bl)
    lhs_h = np.log(V64) + liah - np.log(ah / (us64 * us64) + bh)
    dl = SAFETY * (3 * np.log(2.0) * LG2_ABS * 4 + E24 * 8 * (np.abs(np.log(V64)) + np.abs(lial) + 4))
    res = []
    for k in (np.maximum(k_lo, 0.0), np.maximum(k_hi, 0.0)):
        bnd_l = -lam_lo + k * np.log(lam_lo) - _lgfact(k)
        bnd_h = -lam_hi + k * np.log(lam_hi) - _lgfact(k)
        km = np.maximum(k, 1.0)
        y = (lam_hi - km) / km
        small = k < 16
        eb = SAFETY * np.where(small, 4 * E24 * (lam_hi + k * np.abs(np.log(lam_hi)) + _lgfact(k)) + 1e-6,
                               4 * E24 * (km * y * y + np.log(2 * np.pi * km) + 2) + np.abs(y) * (lam_hi + km) * 4 * E24)
        lhs_lo = np.minimum(lhs_l, lhs_h) - dl; lhs_hi = np.maximum(lhs_l, lhs_h) + dl
        b_lo = np.minimum(bnd_l, bnd_h) - eb; b_hi = np.maximum(bnd_l, bnd_h) + eb
        res.append((lhs_hi <= b_lo, lhs_lo <= b_hi))        # (surely accepted, possibly accepted)
    sure = res[0][0] & res[1][0]
    maybe = res[0][1] | res[1][1]
    acc3 = sure
    cert3 = sure | ~maybe
    accept = acc1 | (~acc1 & ~rej2 & acc3)
    certain = np.where(acc1, cert1, cert1 & cert2 & (rej2 | cert3))
    return accept, certain, np.maximum(k_lo, 0.0), np.maximum(k_hi, 0.0)


# --------------------------------------------------------------------------------------- mixture
def _mixture(sampler, seed, cell, gene, mu, th):
    """Both samplers' gamma-Poisson mixture (blocks 2a: gamma attempt a; Poisson trials t: block
    2 (t // 2) + 1, words (x, y) for even t and (z, w) for odd t).  Returns lo, hi, path, clamped."""
    n = mu.shape[0]
    lo = np.zeros(n, np.int64); hi = np.full(n, INT_MAX, np.int64)
    path = np.full(n, P_PTRS, np.int64)
    lam_lo = np.zeros(n); lam_hi = np.zeros(n)
    ok = np.zeros(n, bool); cert = np.ones(n, bool)
    idx = np.arange(n)
    for att in range(62):
        if not idx.size:
            break
        w = philox_block(seed, gene[idx], cell[idx], TAG_COUNT, 2 * att)
        acc, c, ll, lh = _gamma_attempt(mu[idx], th[idx], w)
        cert[idx] &= c
        done = acc | ~c
        lam_lo[idx[done]] = ll[done]; lam_hi[idx[done]] = lh[done]
        ok[idx[done]] = acc[done]
        idx = idx[~done]
    cert[idx] = False
    live = np.nonzero(cert)[0]
    # lambda < 10: inversion with one uniform
    split_ok = (lam_hi[live] < 10.0) | (lam_lo[live] >= 10.0)
    cert[live[~split_ok]] = False
    live = live[split_ok]
    small = live[lam_hi[live] < 10.0]
    if small.size:
        if sampler == "hybrid":
            b1 = philox_block(seed, gene[small], cell[small], TAG_COUNT, 1)
            word, low = b1[:, 0], b1[:, 1]
        else:
            bq = philox_block(seed, gene[small] >> 2, cell[small], TAG_QUAD, 1)
            word = bq[np.arange(small.size), gene[small] & 3]
            low = philox_block(seed, gene[small], cell[small], TAG_COUNT, 1)[:, 0]
        far = word >= 0xFFF00000
        path[small] = np.where(far, P_MIX_FAR, P_MIX_SMALL)
        for sel, fp64 in ((~far, False), (far, True)):
            s = small[sel]
            if not s.size:
                continue
            if fp64:
                U = (word[sel].astype(np.float64) + (low[sel].astype(np.float64) + 0.5) * 2.0 ** -32) * 2.0 ** -32
            else:
                U = u01(word[sel]).astype(np.float64)
            _, l, h = poisson_inversion(U, lam_lo[s], lam_hi[s], fp64)
            lo[s] = l; hi[s] = h
    # lambda >= 1.6e7: normal limit; 10 <= lambda < 1.6e7: PTRS
    large = live[lam_lo[live] >= 10.0]
    nsplit = (lam_lo[large] < 1.6e7) != (lam_hi[large] < 1.6e7)
    cert[large[nsplit]] = False
    large = large[~nsplit]
    norm = large[lam_lo[large] >= 1.6e7]
    if norm.size:
        path[norm] = P_NORMAL
        b1 = philox_block(seed, gene[norm], cell[norm], TAG_COUNT, 1)
        u1 = u01(b1[:, 0]).astype(np.float64)
        z = np.sqrt(-2 * np.log(u1)) * np.cos(2 * np.pi * u01(b1[:, 1]).astype(np.float64) - np.pi)
        lm = 0.5 * (lam_lo[norm] + lam_hi[norm])
        v = lm + np.sqrt(lm) * z
        e = 0.5 * (lam_hi[norm] - lam_lo[norm]) + SAFETY * (lm * 2 * E24 + np.sqrt(lm) * (np.abs(z) * 4 * RSQRT_REL
                                                                                            + 1e-5 + COS_ABS * 3))
        lo[norm] = np.clip(np.floor(v - e + 0.5), 0, 2 ** 40).astype(np.int64)
        hi[norm] = np.clip(np.ceil(v + e - 0.5), 0, 2 ** 40).astype(np.int64)
    pt = large[lam_lo[large] < 1.6e7]
    idx = pt
    for trial in range(120):
        if not idx.size:
            break
        w = philox_block(seed, gene[idx], cell[idx], TAG_COUNT, 2 * (trial // 2) + 1)
        wu, wv = (w[:, 0], w[:, 1]) if trial % 2 == 0 else (w[:, 2], w[:, 3])
        acc, c, kl, kh = _ptrs_trial(lam_lo[idx], lam_hi[idx], wu, wv)
        cert[idx[~c]] = False
        fin = acc & c
        lo[idx[fin]] = kl[fin].astype(np.int64); hi[idx[fin]] = kh[fin].astype(np.int64)
        idx = idx[~acc & c]
    cert[idx] = False
    # undetermined decisions of the gamma or PTRS stage: any value
    bad = ~cert
    lo[bad] = 0; hi[bad] = INT_MAX
    clamped_lo = lo > CLAMP_AT
    lo = np.where(lo > CLAMP_AT, INT_MAX, lo); hi = np.where(hi > CLAMP_AT, INT_MAX, hi)
    return lo, hi, path, clamped_lo


# ------------------------------------------------------------------------------------------- API
def replay(sampler, seed, cell, gene, params):
    """Replay counts of pst_draw_counts.  sampler: "hybrid" or "gamma_poisson"; seed: the uint64 seed;
    cell: global cell indices (cell0 + local index); gene: gene indices; params: dict of the hook's fp32
    arrays mu, theta, q, a, log2p0 and route (0 mixture, 1 inversion, 2 domain error), one per count.
    Returns dict lo, hi (int64), path (P_* codes) and flags (the status bits these counts set)."""
    cell = np.asarray(cell, np.uint64); gene = np.asarray(gene, np.uint64)
    n = cell.shape[0]
    mu = np.asarray(params["mu"], np.float32); th = np.asarray(params["theta"], np.float32)
    route = np.asarray(params["route"])
    lo = np.zeros(n, np.int64); hi = np.zeros(n, np.int64); path = np.full(n, P_DOMAIN, np.int64)
    flags = 0
    dom = (route == 2) | ~((mu > 0) & (th > 0) & (mu < 3e38) & (th < 3e38))
    if dom.any():
        flags |= FLAG_DOMAIN
    inv = (route == 1) & ~dom if sampler == "hybrid" else np.zeros(n, bool)
    if inv.any():
        i = np.nonzero(inv)[0]
        wq = philox_block(seed, gene[i] >> np.uint64(2), cell[i], TAG_QUAD, 0)
        w = wq[np.arange(i.size), (gene[i] & np.uint64(3)).astype(np.int64)]
        fw = w.astype(np.float32)
        far = fw >= np.float32(4294705152.0)
        q = np.asarray(params["q"], np.float32)[i]; a = np.asarray(params["a"], np.float32)[i]
        e2 = np.asarray(params["log2p0"], np.float32)[i]
        # head and drains: u = (float)w 2^-32 (1 + 2^-15), exact in fp64
        h = np.nonzero(~far)[0]
        U = fw[h].astype(np.float64) * 2.0 ** -32 * (1.0 + 2.0 ** -15)
        _, l, hh, _ = nb_inversion(U, q[h], a[h], e2[h], False, mu[i[h]])
        lo[i[h]] = l; hi[i[h]] = hh
        path[i[h]] = np.where(hh < 10, P_HEAD, P_SEARCH)
        f = np.nonzero(far)[0]
        if f.size:
            path[i[f]] = P_TAIL
            ff = i[f]
            pending = np.arange(f.size)
            for attempt in range(16):
                if not pending.size:
                    break
                g = ff[pending]
                wt = philox_block(seed, gene[g], cell[g], TAG_COUNT, 0xFFFFFFFF - attempt)
                hiw = (w[f[pending]] if attempt == 0 else wt[:, 1]).astype(np.float64)
                U = (hiw + (wt[:, 0].astype(np.float64) + 0.5) * 2.0 ** -32) * 2.0 ** -32 * (1.0 + 2.0 ** -15)
                sub = f[pending]
                _, l, hh, top = nb_inversion(U, q[sub], a[sub], e2[sub], True, mu[g])
                cross = top < 0
                lo[g[cross]] = l[cross]; hi[g[cross]] = hh[cross]
                und = top == 0
                lo[g[und]] = 0; hi[g[und]] = INT_MAX
                pending = pending[top == 1]
            if pending.size:                       # 16 redraws above the top: the kernel keeps the last k
                g = ff[pending]; lo[g] = 0; hi[g] = INT_MAX
    mix = ~dom & ~inv
    if mix.any():
        i = np.nonzero(mix)[0]
        l, h, p, cl = _mixture(sampler, seed, cell[i], gene[i], mu[i], th[i])
        lo[i] = l; hi[i] = h; path[i] = p
        if cl.any():
            flags |= FLAG_CLAMPED
    return {"lo": lo, "hi": hi, "path": path, "flags": flags}
