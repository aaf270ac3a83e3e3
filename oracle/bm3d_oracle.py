"""BM3D / CBM3D restated in numpy: exact int64 block distances, fp64 everything else.

The contract is the one include/b200dn.h states for b200dn_bm3d (Dabov et al. 2007; CBM3D in the opponent space;
'np' parameters with a DCT in both stages).  It is not pinned against the compiled ``bm3d`` package.  The block
matching is vectorised per search offset (a box sum of the squared difference image), the filtering per group size.
The keyword arguments of :func:`stage1` / :func:`stage2` exist so that tests can build wrong references (near misses).
"""
from __future__ import annotations

import math
from fractions import Fraction

import numpy as np

BS = 8
A = np.array([[1 / 3, 1 / 3, 1 / 3], [1 / 2, 0, -1 / 2], [1 / 4, -1 / 2, 1 / 4]])
A_INV = np.array([[1, 1, 2 / 3], [1, 0, -4 / 3], [1, -1, 2 / 3]])
CHANNEL_NORM = np.sqrt((A ** 2).sum(axis=1))          # sigma_c = sigma * ||A_c||_2
TAU_HT, TAU_WIE = 3000, 400
N2_HT, N2_WIE = 16, 32
NS = 39
LAMBDA_HARD = 2.7
KAISER_BETA = 2.0
WIENER_FLOOR = 2.0 ** -10
NEAR = 1e-5                                            # relative distance to the threshold that flags a group


def tau_int(tau) -> int:
    """floor(tau * 64 * 2^20 / 255^2): the threshold on the sum of squared differences of q = rint(1024 Y)."""
    return math.floor(Fraction(tau) * 64 * 2 ** 20 / 255 ** 2)


def n_ref(n: int) -> int:
    return (n - BS) // 3 + 1 + ((n - BS) % 3 != 0)


def ref_positions(n: int) -> np.ndarray:
    """{0, 3, 6, ...} u {n - 8}"""
    p = list(range(0, n - BS + 1, 3))
    if p[-1] != n - BS:
        p.append(n - BS)
    return np.array(p)


def dct_matrix() -> np.ndarray:
    k, j = np.meshgrid(np.arange(BS), np.arange(BS), indexing="ij")
    return np.where(k == 0, np.sqrt(1 / BS), np.sqrt(2 / BS)) * np.cos(np.pi * (2 * j + 1) * k / (2 * BS))


def haar_matrix(n: int) -> np.ndarray:
    """H_1 = [1], H_2m = (1/sqrt 2) [H_m (x) [1, 1]; I_m (x) [1, -1]]"""
    if n == 1:
        return np.ones((1, 1))
    h = haar_matrix(n // 2)
    return np.vstack([np.kron(h, [1.0, 1.0]), np.kron(np.eye(n // 2), [1.0, -1.0])]) / np.sqrt(2.0)


def kaiser2d(beta: float = KAISER_BETA) -> np.ndarray:
    k = np.kaiser(BS, beta)
    return np.outer(k, k)


def matching_plane(img: np.ndarray) -> np.ndarray:
    """q = rint(1024 Y) (half to even) from fp32 [C, H, W]: Y = ((R + G) + B) * fl32(1/3) in fp32, or the grey plane."""
    x = np.asarray(img, dtype=np.float32)
    y = x[0] if x.shape[0] == 1 else ((x[0] + x[1]) + x[2]) * np.float32(1 / 3)
    return np.rint(y * np.float32(1024)).astype(np.int64)


def opponent(img: np.ndarray) -> np.ndarray:
    x = np.asarray(img, dtype=np.float64)
    return x if x.shape[0] == 1 else np.einsum("cd,dhw->chw", A, x)


def block_match(q: np.ndarray, N2: int, tau: int, Ns: int = NS, ref_first: bool = True):
    """Groups of every reference block: positions r * W + c [nR, nC, N2] padded with -1, and sizes [nR, nC].

    Candidates are the blocks whose corner is within +-Ns//2 of the reference's (clipped at the border) with
    d = sum (q_R - q)^2 <= tau; the group is the reference, then the kept candidates in ascending (d, r, c), cut to N2
    and then to a power of two.  ref_first=False sorts the reference in with the others (a near miss)."""
    H, W = q.shape
    rows, cols = ref_positions(H), ref_positions(W)
    rr, cc = rows[:, None], cols[None, :]
    half = Ns // 2
    none = np.iinfo(np.int64).max
    keys = np.full((len(rows), len(cols), Ns * Ns), none, dtype=np.int64)
    for dr in range(-half, half + 1):
        for dc in range(-half, half + 1):
            valid = (rr + dr >= 0) & (rr + dr <= H - BS) & (cc + dc >= 0) & (cc + dc <= W - BS)
            if not valid.any() or (ref_first and dr == 0 and dc == 0):
                continue
            y0, y1, x0, x1 = max(0, -dr), min(H, H - dr), max(0, -dc), min(W, W - dc)
            diff = q[y0 + dr:y1 + dr, x0 + dc:x1 + dc] - q[y0:y1, x0:x1]
            ii = np.zeros((y1 - y0 + 1, x1 - x0 + 1), dtype=np.int64)
            ii[1:, 1:] = (diff * diff).cumsum(0).cumsum(1)
            r = np.clip(rr - y0, 0, y1 - y0 - BS)
            c = np.clip(cc - x0, 0, x1 - x0 - BS)
            d = ii[r + BS, c + BS] - ii[r, c + BS] - ii[r + BS, c] + ii[r, c]
            keep = valid & (d <= tau)
            keys[..., (dr + half) * Ns + dc + half] = np.where(keep, d * 2048 + (dr + half) * Ns + dc + half, none)
    take = N2 - 1 if ref_first else N2
    best = np.sort(keys, axis=-1)[..., :take]
    wpos = best % 2048
    cand = (rr[..., None] + wpos // Ns - half) * W + cc[..., None] + wpos % Ns - half
    cand = np.where(best == none, -1, cand)
    if ref_first:
        cand = np.concatenate([(rr * W + cc)[..., None] + np.zeros_like(cand[..., :1]), cand], axis=-1)
    count = (cand >= 0).sum(-1)
    size = (2 ** np.floor(np.log2(np.maximum(count, 1)))).astype(np.int64)
    pos = np.where(np.arange(N2) < size[..., None], cand, -1)
    return pos.astype(np.int32), size.astype(np.int32)


def _filter(noisy: np.ndarray, basic, pos, size, sigma: float, stage: int, lam: float, beta: float, haar: bool):
    """Collaborative filtering + aggregation of one stage on opponent planes [C, H, W]; returns the estimate in the
    same planes and, for stage 1, per group whether a coefficient lies within NEAR (relative) of the threshold."""
    Cn, H, W = noisy.shape
    D, K = dct_matrix(), kaiser2d(beta).ravel()
    offs = (np.arange(BS)[:, None] * W + np.arange(BS)[None, :]).ravel()
    num, den = np.zeros((Cn, H * W)), np.zeros((Cn, H * W))
    near = np.zeros(size.shape, dtype=bool)
    for n in np.unique(size):
        gi = np.nonzero(size == n)
        pix = pos[gi][:, :n, None].astype(np.int64) + offs                      # [G, n, 64]
        Hn = haar_matrix(int(n)) if haar else np.eye(int(n))
        for c in range(Cn):
            sc = sigma * (CHANNEL_NORM[c] if Cn == 3 else 1.0)
            coef = D @ noisy[c].ravel()[pix].reshape(-1, n, BS, BS) @ D.T
            gam = np.einsum("mn,gnkl->gmkl", Hn, coef)
            if stage == 1:
                thr = lam * sc
                keep = np.abs(gam) > thr
                near[gi] |= (np.abs(np.abs(gam) - thr) <= NEAR * thr).any(axis=(1, 2, 3))
                gam = np.where(keep, gam, 0.0)
                w = 1.0 / np.maximum(keep.sum(axis=(1, 2, 3)), 1)
            else:
                gb = np.einsum("mn,gnkl->gmkl", Hn, D @ basic[c].ravel()[pix].reshape(-1, n, BS, BS) @ D.T)
                wie = gb * gb / (gb * gb + sc * sc)
                gam = wie * gam
                w = 1.0 / np.maximum((wie * wie).sum(axis=(1, 2, 3)), WIENER_FLOOR)
            est = D.T @ np.einsum("nm,gnkl->gmkl", Hn, gam) @ D
            wk = w[:, None, None] * K
            num[c] += np.bincount(pix.ravel(), weights=(wk * est.reshape(-1, n, 64)).ravel(), minlength=H * W)
            den[c] += np.bincount(pix.ravel(), weights=np.broadcast_to(wk, pix.shape).ravel(), minlength=H * W)
    return (num / den).reshape(Cn, H, W), near


def _to_image(planes: np.ndarray) -> np.ndarray:
    return planes if planes.shape[0] == 1 else np.einsum("cd,dhw->chw", A_INV, planes)


def stage1(z: np.ndarray, sigma: float, lam: float = LAMBDA_HARD, beta: float = KAISER_BETA, haar: bool = True,
           N2: int = N2_HT, ref_first: bool = True, Ns: int = NS, tau_scale: float = 1.0) -> dict:
    """Hard-thresholding stage of fp32 [C, H, W] (C = 1 or 3).  Returns the basic estimate ``out`` (fp64, image
    space), the groups ``match`` / ``size``, the per-group ``near`` flags and their pixel ``footprint``."""
    z = np.asarray(z, dtype=np.float32)
    pos, size = block_match(matching_plane(z), N2, tau_int(Fraction(TAU_HT) * Fraction(tau_scale)), Ns, ref_first)
    est, near = _filter(opponent(z), None, pos, size, sigma, 1, lam, beta, haar)
    foot = np.zeros(z.shape[1] * z.shape[2], dtype=bool)
    for g in zip(*np.nonzero(near)):
        p = pos[g][:size[g]].astype(np.int64)
        foot[(p[:, None] + (np.arange(BS)[:, None] * z.shape[2] + np.arange(BS)).ravel()).ravel()] = True
    return {"out": _to_image(est), "match": pos, "size": size, "near": near,
            "footprint": foot.reshape(z.shape[1:])}


def stage2(z: np.ndarray, basic: np.ndarray, sigma: float, beta: float = KAISER_BETA, haar: bool = True,
           N2: int = N2_WIE, ref_first: bool = True, Ns: int = NS, tau_scale: float = 1.0) -> dict:
    """Wiener stage of fp32 [C, H, W] on the fp32 basic estimate (groups matched on the basic estimate)."""
    z, basic = np.asarray(z, dtype=np.float32), np.asarray(basic, dtype=np.float32)
    pos, size = block_match(matching_plane(basic), N2, tau_int(Fraction(TAU_WIE) * Fraction(tau_scale)), Ns,
                            ref_first)
    est, _ = _filter(opponent(z), opponent(basic), pos, size, sigma, 2, LAMBDA_HARD, beta, haar)
    return {"out": _to_image(est), "match": pos, "size": size}


def bm3d(z: np.ndarray, sigma: float) -> np.ndarray:
    """stage2(z, basic = stage1(z) rounded to fp32), as the device composes the two."""
    return stage2(z, stage1(z, sigma)["out"].astype(np.float32), sigma)["out"]


def synthetic(C: int, H: int, W: int, seed: int) -> np.ndarray:
    """A seeded low-passed image in [0.15, 0.85] with a few step edges, fp32 [C, H, W]."""
    from scipy.ndimage import gaussian_filter
    rng = np.random.default_rng(seed)
    x = gaussian_filter(rng.standard_normal((C, H, W)), sigma=(0, 3, 3))
    for _ in range(4):
        r0, c0 = rng.integers(0, H), rng.integers(0, W)
        x[:, r0:r0 + H // 3, c0:c0 + W // 3] += rng.normal(0, 2 * x.std(), size=(C, 1, 1))
    lo, hi = x.min(axis=(1, 2), keepdims=True), x.max(axis=(1, 2), keepdims=True)
    return ((x - lo) / np.maximum(hi - lo, 1e-12) * 0.7 + 0.15).astype(np.float32)


def noisy(clean: np.ndarray, sigma: float, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    return (clean + sigma * rng.standard_normal(clean.shape)).astype(np.float32)
