"""Host-side parameter tables for the CUDA kernels.

Everything that depends on species parameters or frame geometry but NOT on pixel values is built
here, on the host, with the same NumPy / torch expressions (and therefore the same dtype
promotions and roundings) the reference evaluates per frame, then uploaded once and cached:
  * 256-entry sRGB decode LUTs            (animals/animal_utils.py:5-11, :41-50; uv_helpers.py:15-19)
  * encode quantiser thresholds           (animals/dog.py:54-59 with animal_utils.py:13-19)
  * the 3x3 colour matrices               (animal_utils.py:52-119, animals/cat.py:95-101)
  * Gaussian taps                         (cv2.getGaussianKernel as called by cv2.GaussianBlur)
  * cat wide-FOV per-column maps/weights  (animals/cat_widevision_utils.py:61-96)
  * centre-zoom fixed-point resize tables (cat_widevision_utils.py:11-29 -> cv2.resize INTER_LINEAR)
  * streak-blur per-row taps + 3x3         (animal_utils.py:147-172)
  * S-cone row gain                       (animal_utils.py:236-247)
  * honeybee spectral tables              (classic_rgb_to_hsi.py:55-78, uv_helpers.py:187-192, honeybee.py:81-93,179-192)
This is the safe route to <=1 LSB (SURVEY.md section 7): the device only does per-pixel arithmetic.
"""
from __future__ import annotations

import math
from functools import lru_cache
from typing import NamedTuple

import numpy as np

# ----------------------------------------------------------------------------- colour
_RGB2LMS = np.array([[0.31399022, 0.63951294, 0.04649755],
                     [0.15537241, 0.75789446, 0.08670142],
                     [0.01775239, 0.10944209, 0.87256922]], dtype=np.float32)   # animal_utils.py:56-62
_LMS2RGB = np.array([[5.472213, -4.6419606, 0.16963711],
                     [-1.125242, 2.2931712, -0.16789523],
                     [0.02980164, -0.19318072, 1.1636479]], dtype=np.float64)   # animal_utils.py:70-75


def _eotf(x):
    return np.where(x <= 0.04045, x / 12.92, ((x + 0.055) / (1 + 0.055)) ** 2.4)


def _oetf(x):
    return np.where(x <= 0.0031308, 12.92 * x, (1 + 0.055) * (x ** (1 / 2.4)) - 0.055)


@lru_cache(maxsize=None)
def decode_lut(div255: bool = True) -> np.ndarray:
    """decode(normalise(v)), v = 0..255, float32.  div255=False is the `max <= 1` branch of
    get_normalized_image: bytes are only clipped to [0,1]."""
    v = np.arange(256, dtype=np.float32)
    if div255:
        v /= 255.0
    v = np.clip(v, 0.0, 1.0)
    lut = _eotf(v).astype(np.float32)
    lut.setflags(write=False)
    return lut


@lru_cache(maxsize=None)
def decode_lut_torch() -> np.ndarray:
    """uint8 -> to_float01 (always /255) -> the torch expression of classic_rgb_to_hsi.py:16-22."""
    import torch
    t = torch.arange(256, dtype=torch.float32).numpy().astype(np.float32) / 255.0
    t = torch.from_numpy(t)
    lut = torch.where(t <= 0.04045, t / 12.92, ((t + 0.055) / (1.0 + 0.055)) ** 2.4).numpy().astype(np.float32)
    lut.setflags(write=False)
    return lut


def _quantise(x32: np.ndarray, *, f64: bool) -> np.ndarray:
    """The reference's encode tail as a function of a float32 linear value."""
    x = x32.astype(np.float64) if f64 else x32
    s = np.clip(_oetf(np.clip(x, 0.0, 1.0)), 0.0, 1.0)
    return (s * 255.0 + 0.5).astype(np.uint8)


@lru_cache(maxsize=None)
def encode_thresholds(f64: bool = False) -> np.ndarray:
    """thr[i-1] = smallest float32 x with quantise(x) >= i (i = 1..255), by bisection over float32
    bit patterns using the reference's own NumPy expression.  f64=True: the float64 tail Cat runs
    (cat.py:101-109), still as a function of a float32 input."""
    lo = np.zeros(255, np.uint32)                       # quantise(0) = 0 < i
    hi = np.full(255, np.float32(1.0).view(np.uint32))  # quantise(1) = 255 >= i
    want = np.arange(1, 256)
    while np.any(hi - lo > 1):
        mid = ((lo.astype(np.uint64) + hi) // 2).astype(np.uint32)
        ge = _quantise(mid.view(np.float32), f64=f64) >= want
        hi = np.where(ge, mid, hi)
        lo = np.where(ge, lo, mid)
    thr = hi.view(np.float32).copy()
    thr.setflags(write=False)
    return thr


def dichromat_matrix(alpha: float, s_scale: float) -> np.ndarray:
    """collapse_LMS_matrix (animal_utils.py:88-119): float32 T, applied by the reference as
    `pixels @ T.T`, i.e. out[c] = sum_k T[c,k] lin[k]."""
    lms = np.eye(3, dtype=np.float32) @ _RGB2LMS.T
    D = np.array([[alpha, 1.0 - alpha, 0.0], [alpha, 1.0 - alpha, 0.0], [0.0, 0.0, s_scale]], dtype=np.float32)
    return ((lms @ D.T) @ _LMS2RGB.T).astype(np.float32)


def cat_matrix(alpha: float = 0.5) -> np.ndarray:
    """cat.py:95-101 collapsed to one matrix: RGB->LMS, LM = a L + (1-a) M, LMS->RGB.
    out = lin @ RGB2LMS.T @ Dm.T @ LMS2RGB.T, composed in float64 and rounded once."""
    Dm = np.array([[alpha, 1.0 - alpha, 0.0], [alpha, 1.0 - alpha, 0.0], [0.0, 0.0, 1.0]], dtype=np.float64)
    T = _LMS2RGB @ Dm @ _RGB2LMS.astype(np.float64)
    return T.astype(np.float32)


# ----------------------------------------------------------------------------- Gaussian taps
def gaussian_ksize(sigma: float) -> int:
    """cv2.GaussianBlur(ksize=(0,0)) on float images: cvRound(8 sigma + 1) | 1."""
    return int(round(sigma * 4 * 2 + 1)) | 1


def gaussian_taps(ksize: int, sigma: float) -> np.ndarray:
    """cv2.getGaussianKernel(ksize, sigma, CV_32F) for sigma > 0."""
    x = np.arange(ksize, dtype=np.float64) - (ksize - 1) * 0.5
    w = np.exp(-(x * x) / (2.0 * sigma * sigma))
    return (w / w.sum()).astype(np.float32)


# ----------------------------------------------------------------------------- cat geometry
def cat_zoom_scale(camera_hfov=100.0, half_fov=105.0, ratio=1.30) -> float:
    """cat_widevision_utils.py:31-44."""
    eff = min(float(camera_hfov), 2.0 * float(half_fov))
    ratio = max(1.01, float(ratio))
    return float(math.tan(math.radians(camera_hfov) * 0.5) / max(math.tan(math.radians(eff / ratio) * 0.5), 1e-6))


def cat_warp_tables(W: int, fov_in=100.0, half_fov=105.0, overlap=40.0):
    """(xL, xR, wL, wR) float32[W] of cat_widevision_utils.py:61-96; maps are constant down a column."""
    phi = np.deg2rad(half_fov)
    psi = np.deg2rad(fov_in * 0.5)
    alpha = max(0.0, phi - 0.5 * np.deg2rad(overlap))
    u = np.linspace(-1.0, 1.0, W, dtype=np.float32)
    theta = u * phi
    gL, gR = theta - alpha, theta + alpha
    xL = ((gL / psi) * (W * 0.5) + (W * 0.5)).astype(np.float32)
    xR = ((gR / psi) * (W * 0.5) + (W * 0.5)).astype(np.float32)
    win = (np.cos(0.5 * np.pi * (theta / phi)) ** 2).astype(np.float32)
    wL = win * (np.abs(gL) <= psi).astype(np.float32)
    wR = win * (np.abs(gR) <= psi).astype(np.float32)
    return xL, xR, wL, wR


def cat_warp_device_table(W: int, fov_in=100.0, half_fov=105.0, overlap=40.0) -> np.ndarray:
    """float32 [6*W] for avb_cat_u8: xL, xR, wL, wR, the blend denominator ws = wL + wR + 1e-8
    (float32, cat_widevision_utils.py:97) and its correctly rounded reciprocal."""
    xL, xR, wL, wR = cat_warp_tables(W, fov_in, half_fov, overlap)
    ws = (wL + wR + 1e-8).astype(np.float32)
    rws = (np.float32(1.0) / ws).astype(np.float32)
    return np.concatenate([xL, xR, wL, wR, ws, rws]).astype(np.float32)


def resize_axis_table(src: int, dst: int, *, vertical: bool):
    """cv2.resize INTER_LINEAR, uint8: per output index (i0, i1, w0, w1) with 11-bit weights.
    Horizontal: an out-of-range neighbour zeroes the fraction.  Vertical: only indices clamp."""
    scale = 1.0 / (dst / src)
    f = ((np.arange(dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = f - s.astype(np.float32)
    if not vertical:
        f[s < 0] = 0
        s[s < 0] = 0
        hi = s >= src - 1
        f[hi] = 0
        s[hi] = src - 1
    w1 = np.rint(f * np.float32(2048)).astype(np.int32)
    w0 = np.rint((np.float32(1.0) - f) * np.float32(2048)).astype(np.int32)
    i0 = np.clip(s, 0, src - 1).astype(np.int32)
    i1 = np.clip(s + 1, 0, src - 1).astype(np.int32)
    return i0, i1, w0, w1


def center_zoom_box(W: int, H: int, scale: float):
    """cat_widevision_utils.py:19-25 -> (x0, y0, cw, ch)."""
    cw = max(1, int(round(W / scale)))
    ch = max(1, int(round(H / scale)))
    return (W - cw) // 2, (H - ch) // 2, cw, ch


def center_zoom_tables(W: int, H: int, scale: float) -> np.ndarray:
    """int32 table for avb_cat_u8: W rows {xi0, xi1, xw0, xw1} then H rows {yi0, yi1, yw0, yw1}
    (source indices already offset by the crop origin, 11-bit weights), flattened to 4*W + 4*H."""
    x0, y0, cw, ch = center_zoom_box(W, H, scale)
    xi0, xi1, xw0, xw1 = resize_axis_table(cw, W, vertical=False)
    yi0, yi1, yw0, yw1 = resize_axis_table(ch, H, vertical=True)
    tx = np.stack([xi0 + x0, xi1 + x0, xw0, xw1], axis=1)
    ty = np.stack([yi0 + y0, yi1 + y0, yw0, yw1], axis=1)
    return np.concatenate([tx.ravel(), ty.ravel()]).astype(np.int32)


# ----------------------------------------------------------------------------- streak blur
def streak_sigmas(H: int, y_center: float, s_streak: float, s_far: float, falloff: float):
    """animal_utils.py:155-162 in the reference's float32 arithmetic."""
    yy = np.linspace(0, 1, H, dtype=np.float32)[:, None]
    d = np.abs(yy - y_center)
    smap = s_streak + (s_far - s_streak) * (1.0 - np.exp(-falloff * d ** 2))
    sx = np.maximum(0.4, 0.5 * smap)
    return sx[:, 0].astype(np.float64), smap[:, 0].astype(np.float64)


def _reflect101(i: int, n: int) -> int:
    if n == 1:
        return 0
    p = 2 * n - 2
    m = i % p
    return p - m if m >= n else m


STREAK_RMAX = 16      # combined radius limit of the device kernel (k2_streak.cu ST_RMAX)
STREAK_TAB = 56       # floats per row: 33 taps (centred at index 16), 9 matrix entries, radius, two-plane factors


def rank2_factor(M: np.ndarray):
    """M (3x3, float32 values) = P (3x2) Q (2x3) if it has rank <= 2, else None.  Q is an exact copy of the two
    most independent rows of M, P the coefficients of every row in that basis (least squares, float64);
    accepted when the residual is within a few float32 ulps of the largest entry (M itself was rounded)."""
    M = np.asarray(M, np.float64)
    best, pair = -1.0, (0, 1)
    for i, j in ((0, 1), (0, 2), (1, 2)):
        a = np.linalg.norm(np.cross(M[i], M[j]))
        if a > best:
            best, pair = a, (i, j)
    Q = M[list(pair)]
    if best <= 0.0:
        return None
    P = M @ np.linalg.pinv(Q)
    if np.abs(P @ Q - M).max() > 4e-7 * np.abs(M).max():
        return None
    return P, Q


def streak_row_table(H: int, M: np.ndarray, y_center: float, s_streak: float, s_far: float, falloff: float) -> np.ndarray:
    """Per-row table [H, 48] float32 for the streak blur as it actually behaves (SURVEY.md 8a-6):
      [0:33]  the two x passes (taps of sigmaX(y), then taps of sigmaY(y)) composed into one
              symmetric tap vector, centred at index 16, zero padded;
      [33:42] row-major 3x3 = (REFLECT_101 channel mix of the sigmaX taps over a width of 3) @ M,
              M being the species' dichromat matrix (applied as out = A @ lin);
      [42]    combined radius r1 + r2;
      [43:49] row-major 3x2 P_y, [49:55] row-major 2x3 Q, [55] 1.0 when they are valid: every dichromat matrix
              has rank 2 (L and M are merged), M = P Q, so the row's 3x3 is (mix_y P) Q and only the TWO
              planes Q lin need filtering; the 3x2 expansion P_y = mix_y P follows the filter.
    Composed in float64 from the float32 taps OpenCV would use, rounded once."""
    sx, sy = streak_sigmas(H, y_center, s_streak, s_far, falloff)
    tab = np.zeros((H, STREAK_TAB), np.float32)
    M64 = np.asarray(M, np.float64)
    fac = rank2_factor(M64)
    cache = {}
    for y in range(H):
        key = (sx[y], sy[y])
        if key not in cache:
            k1, k2 = gaussian_ksize(sx[y]), gaussian_ksize(sy[y])
            g1, g2 = gaussian_taps(k1, sx[y]).astype(np.float64), gaussian_taps(k2, sy[y]).astype(np.float64)
            r1, r2 = k1 // 2, k2 // 2
            if r1 + r2 > STREAK_RMAX:
                raise ValueError(f"streak blur sigma too large for the device kernel (radius {r1}+{r2} > {STREAK_RMAX})")
            mix = np.zeros((3, 3), np.float64)
            for c in range(3):
                for t in range(k1):
                    mix[c, _reflect101(c + t - r1, 3)] += g1[t]
            row = np.zeros(STREAK_TAB, np.float32)
            comb = np.convolve(g1, g2)
            r = r1 + r2
            row[STREAK_RMAX - r:STREAK_RMAX + r + 1] = comb.astype(np.float32)
            row[33:42] = (mix @ M64).astype(np.float32).ravel()
            row[42] = float(r)
            if fac is not None:
                P, Q = fac
                row[43:49] = (mix @ P).astype(np.float32).ravel()
                row[49:55] = Q.astype(np.float32).ravel()
                row[55] = 1.0
            cache[key] = row
        tab[y] = cache[key]
    return tab


def scone_row_gain(H: int, s_top=1.0, s_bottom=0.6, power=1.0, extra_boost=0.0) -> np.ndarray:
    """animal_utils.py:236-247 (band=None): float32 per-row gain of channel 2."""
    w = np.linspace(s_top, s_bottom, H, dtype=np.float32)
    if power != 1.0:
        t = (w - s_bottom) / max(1e-8, (s_top - s_bottom))
        t = np.clip(t, 0.0, 1.0) ** power
        w = s_bottom + (s_top - s_bottom) * t
    if extra_boost != 0.0:
        w = 1.0 + extra_boost * (w - 1.0)
    return w.astype(np.float32)


# ----------------------------------------------------------------------------- honeybee spectra
def analytic_lobes(wavelengths: np.ndarray):
    """(G [B,3], denom): G[:,c] is the Gaussian lobe driven by INPUT CHANNEL c, evaluated with the
    reference's torch float32 expressions (classic_rgb_to_hsi.py:60-78); denom is the scalar
    normaliser including the reference's differently-parenthesised third term (:75)."""
    import torch
    wl = torch.as_tensor(np.asarray(wavelengths, np.float32))
    g2 = torch.exp(-0.5 * ((wl - 610.0) / 60.0) ** 2)     # input channel 2
    g1 = torch.exp(-0.5 * ((wl - 545.0) / 60.0) ** 2)     # input channel 1
    g0 = torch.exp(-0.5 * ((wl - 460.0) / 55.0) ** 2)     # input channel 0
    denom = (g2 + g1 + torch.exp(-0.5 * ((wl - 460.0) ** 2) / (55.0 ** 2))).mean()
    G = torch.stack([g0, g1, g2], dim=1).numpy().astype(np.float32)
    return G, np.float32(denom.item())


def d65_like(lam: np.ndarray) -> np.ndarray:
    """uv_helpers.py:187-192."""
    x = (lam - 560.0) / 50.0
    base = np.exp(-0.5 * x ** 2) + 0.3 * np.exp(-0.5 * ((lam - 450.0) / 35.0) ** 2)
    base /= base.mean()
    return base.astype(np.float32)


def honeybee_curves(lam: np.ndarray) -> np.ndarray:
    """[3, B] float32 UV/Blue/Green sensitivities, each sum-normalised (honeybee.py:88-93, :179-192)."""
    rows = []
    for peak, sigma in ((350.0, 25.0), (440.0, 30.0), (540.0, 35.0)):
        v = np.exp(-0.5 * ((lam - peak) / sigma) ** 2).astype(np.float32)
        s = v.sum()
        if s > 0:
            v /= s
        rows.append(v)
    return np.stack(rows)


def uv_band_table(lam: np.ndarray, sens: np.ndarray, illuminant: np.ndarray | None):
    """Device table for the per-pixel band loop: [B, 8] rows {g0,g1,g2, E, s0,s1,s2, 0} and the
    float32 normaliser denom + 1e-8 (torch adds the Python float to a float32 tensor)."""
    G, denom = analytic_lobes(lam)
    B = len(lam)
    E = np.ones(B, np.float32) if illuminant is None else np.asarray(illuminant, np.float32)
    tab = np.zeros((B, 8), np.float32)
    tab[:, 0:3] = G
    tab[:, 3] = E
    tab[:, 4:4 + sens.shape[0]] = sens.T
    return tab, np.float32(np.float32(denom) + np.float32(1e-8))


def uv_collapsed_matrix(lam: np.ndarray, sens: np.ndarray, illuminant: np.ndarray | None) -> np.ndarray:
    """[R,3] float32: catches = M @ lin.  M[k,c] = sum_l sens[k,l] E[l] G[l,c] / (denom + 1e-8),
    composed in float64 from the float32 tables (SURVEY.md 8a-11: the chain is linear)."""
    tab, denom_eps = uv_band_table(lam, sens, illuminant)
    G, E = tab[:, 0:3].astype(np.float64), tab[:, 3].astype(np.float64)
    M = (sens.astype(np.float64) * E[None, :]) @ G / np.float64(denom_eps)
    return M.astype(np.float32)


def uv_blur_taps(sigma: float) -> np.ndarray:
    """uv_helpers.py:67-73: ksize = 2*ceil(3 sigma)+1 (empty array: no blur)."""
    if sigma <= 0:
        return np.zeros(0, np.float32)
    return gaussian_taps(int(2 * np.ceil(3 * sigma) + 1), sigma)


def uv_map_params(custom_matrix=None) -> np.ndarray:
    """15 floats for avb_uv_map_u8: [0:9] the custom 3x3 (uv_mappers.py:45-50, applied as C @ M.T),
    [9:12] / [12:15] the purple and warm anchors of map_uv_purple_yellow_soft in linear light
    (uv_mappers.py:107-116, same NumPy expressions)."""
    out = np.zeros(15, np.float32)
    if custom_matrix is not None:
        out[:9] = np.asarray(custom_matrix, np.float32).reshape(9)

    def s2l(v):
        return np.where(v <= 0.04045, v / 12.92, ((v + 0.055) / (1 + 0.055)) ** 2.4).astype(np.float32)
    out[9:12] = s2l(np.array([176, 124, 232], np.float32) / 255.0)
    out[12:15] = s2l(np.array([255, 211, 138], np.float32) / 255.0)
    return out


def bandpass_weights(lam: np.ndarray, lo: float, hi: float) -> np.ndarray:
    """uv_helpers.py:125-139 (uniform 1/B fallback when the band holds no sample / no mass)."""
    wl = lam.astype(np.float32)
    w = np.zeros_like(wl, dtype=np.float32)
    inside = (wl >= lo) & (wl <= hi)
    if not np.any(inside):
        return np.ones_like(wl, dtype=np.float32) / float(wl.size)
    x = (wl[inside] - lo) / (hi - lo)
    w[inside] = 0.5 * (1.0 - np.cos(2.0 * np.pi * x))
    s = float(np.sum(w))
    if s > 1e-12:
        w /= s
    else:
        w = np.ones_like(wl, dtype=np.float32) / float(wl.size)
    return w


MANTIS_BANDS = ((320, 360), (360, 400), (400, 430), (430, 460), (460, 490),
                (490, 520), (520, 550), (550, 580), (580, 610), (610, 680))   # mantis_shrimp.py:49-60


def mantis_band_matrix(lam: np.ndarray) -> np.ndarray:
    return np.stack([bandpass_weights(lam, float(lo), float(hi)) for lo, hi in MANTIS_BANDS]).astype(np.float32)


# ----------------------------------------------------------------------------- cv2.resize tap tables (float images)
def _cubic_coeffs(x: np.ndarray) -> np.ndarray:
    """OpenCV interpolateCubic (A = -0.75), float32 arithmetic; taps at sx-1 .. sx+2."""
    A = np.float32(-0.75)
    x = x.astype(np.float32)
    one = np.float32(1.0)
    c0 = ((A * (x + one) - np.float32(5) * A) * (x + one) + np.float32(8) * A) * (x + one) - np.float32(4) * A
    c1 = ((A + np.float32(2)) * x - (A + np.float32(3))) * x * x + one
    c2 = ((A + np.float32(2)) * (one - x) - (A + np.float32(3))) * (one - x) * (one - x) + one
    c3 = one - c0 - c1 - c2
    return np.stack([c0, c1, c2, c3], axis=1).astype(np.float32)


def resize_taps(src: int, dst: int, interp: str, *, vertical: bool = False):
    """(idx int32 [dst, taps], w float32 [dst, taps]) such that one axis of cv2.resize on a float image is
    out[d] = sum_t w[d, t] * in[idx[d, t]]  (borders already resolved in idx), restating OpenCV's own coordinate
    arithmetic (imgproc/resize.cpp): `linear` / `cubic` (fx = (d + 0.5) * scale - 0.5 in float32; the horizontal
    linear pass zeroes the fraction at the borders, everything else clamps indices) and `area` (downscale only:
    computeResizeAreaTab; integer factors give the uniform 1/factor block mean of resizeAreaFast).
    Used by uv_helpers.py:57-64 / :84-99 / :155-183 and cat_widevision_utils.py:26 on float frames."""
    src, dst = int(src), int(dst)
    scale = float(src) / float(dst)
    if interp in ("linear", "cubic"):
        f = ((np.arange(dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
        s = np.floor(f).astype(np.int64)
        f = f - s.astype(np.float32)
        if interp == "linear":
            if not vertical:
                lo = s < 0
                f[lo] = 0
                s[lo] = 0
                hi = s >= src - 1
                f[hi] = 0
                s[hi] = src - 1
            idx = np.stack([s, s + 1], axis=1)
            w = np.stack([np.float32(1.0) - f, f], axis=1)
        else:
            idx = np.stack([s - 1, s, s + 1, s + 2], axis=1)
            w = _cubic_coeffs(f)
        return np.clip(idx, 0, src - 1).astype(np.int32), np.ascontiguousarray(w, np.float32)
    if interp == "nearest":
        # resizeNN: sx = min(floor(x * ifx), src - 1), ifx = 1 / (dst / src) in double (morpho.py:93 mosaic up-sampling)
        ifx = 1.0 / (float(dst) / float(src))
        s = np.minimum(np.floor(np.arange(dst, dtype=np.float64) * ifx).astype(np.int64), src - 1)
        return s.astype(np.int32)[:, None], np.ones((dst, 1), np.float32)
    if interp != "area":
        raise ValueError(f"unknown interpolation {interp}")
    if dst > src:
        raise ValueError("INTER_AREA tables are for down-scaling")
    rows = []
    for d in range(dst):
        fsx1 = d * scale
        fsx2 = fsx1 + scale
        cell = min(scale, src - fsx1)
        sx1, sx2 = int(math.ceil(fsx1)), int(math.floor(fsx2))
        sx2 = min(sx2, src - 1)
        sx1 = min(sx1, sx2)
        taps = []
        if sx1 - fsx1 > 1e-3:
            taps.append((sx1 - 1, np.float32((sx1 - fsx1) / cell)))
        for sx in range(sx1, sx2):
            taps.append((sx, np.float32(1.0 / cell)))
        if fsx2 - sx2 > 1e-3:
            taps.append((sx2, np.float32(min(min(fsx2 - sx2, 1.0), cell) / cell)))
        rows.append(taps)
    nt = max(len(r) for r in rows)
    idx = np.zeros((dst, nt), np.int32)
    w = np.zeros((dst, nt), np.float32)
    for d, taps in enumerate(rows):
        for t, (i, a) in enumerate(taps):
            idx[d, t], w[d, t] = i, a
        for t in range(len(taps), nt):
            idx[d, t] = taps[-1][0]          # zero-weight padding reads a valid sample
    return idx, w


def panorama_geometry(W: int, scale_x: float):
    """uv_helpers.py:84-99 panorama_warp: (newW, start) of the widen + centre crop, or None when it is the identity."""
    if abs(scale_x - 1.0) < 1e-3:
        return None
    newW = max(2, int(round(W * scale_x)))
    if newW == W:
        return newW, 0
    return newW, (newW - W) // 2


def scaled_hw(H: int, W: int, scale: float):
    """uv_helpers.py:169-171 classic_rgb_to_hsi_scaled: size of the down-sampled frame."""
    return max(1, int(round(H * scale))), max(1, int(round(W * scale)))


# ---------------------------------------------------------------------------------------------------- JPEG (K8)
# What libjpeg(-turbo) writes for cv2.imencode(".jpg", frame, [IMWRITE_JPEG_QUALITY, q]) with OpenCV's defaults.
JPEG_ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,
                        7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,
                        39, 46, 53, 60, 61, 54, 47, 55, 62, 63])
_JPEG_STD_Q = (  # ITU-T T.81 Annex K.1, natural order: luminance, chrominance
    [16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22, 29, 51, 87, 80,
     62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, 49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98,
     112, 100, 103, 99],
    [17, 18, 24, 47] + [99] * 4 + [18, 21, 26, 66] + [99] * 4 + [24, 26, 56] + [99] * 5 + [47, 66] + [99] * 38)
_JPEG_STD_HUFF = (  # ITU-T T.81 Annex K.3 as (table class/id, bits[1..16], values): DC0, AC0, DC1, AC1
    (0x00, "00010501010101010100000000000000", "000102030405060708090a0b"),
    (0x10, "0002010303020403050504040000017d",
     "01020300041105122131410613516107227114328191a1082342b1c11552d1f02433627282090a161718191a25262728292a3435363738"
     "393a434445464748494a535455565758595a636465666768696a737475767778797a838485868788898a92939495969798999aa2a3a4a5"
     "a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8e9eaf1f2f3f4f5f6f7f8f9fa"),
    (0x01, "00030101010101010101010000000000", "000102030405060708090a0b"),
    (0x11, "00020102040403040705040400010277",
     "000102031104052131061241510761711322328108144291a1b1c109233352f0156272d10a162434e125f11718191a262728292a35363738"
     "393a434445464748494a535455565758595a636465666768696a737475767778797a82838485868788898a92939495969798999aa2a3a4a5"
     "a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7e8e9eaf2f3f4f5f6f7f8f9fa"),
)


def jpeg_quant_tables(quality: int) -> np.ndarray:
    """[2, 64] uint8 quantisers in zigzag order (luma, chroma), i.e. the payloads of the two DQT segments:
    jcparam.c jpeg_quality_scaling (5000/q below 50, 200-2q otherwise), (std*scale + 50)/100 clamped to [1, 255]."""
    q = int(quality)
    if not 1 <= q <= 100:
        raise ValueError(f"JPEG quality must lie in [1, 100], got {quality!r}")
    scale = 5000 // q if q < 50 else 200 - 2 * q
    t = np.clip((np.array(_JPEG_STD_Q, np.int64) * scale + 50) // 100, 1, 255)
    return t[:, JPEG_ZIGZAG].astype(np.uint8)


def _jpeg_segment(marker: int, payload: bytes) -> bytes:
    return bytes([0xFF, marker]) + (len(payload) + 2).to_bytes(2, "big") + payload


def jpeg_header(H: int, W: int, quality: int) -> bytes:
    """Every byte cv2.imencode writes before the entropy-coded data: SOI, APP0 JFIF 1.01 (density 1:1, no units),
    DQT luma / chroma, SOF0 (3 components, 4:2:0), DHT DC0 / AC0 / DC1 / AC1, SOS."""
    if not (1 <= int(H) <= 65535 and 1 <= int(W) <= 65535):
        raise ValueError(f"JPEG frame size must lie in [1, 65535]^2, got {H}x{W}")
    qt = jpeg_quant_tables(quality)
    out = b"\xff\xd8" + _jpeg_segment(0xE0, b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    for i in range(2):
        out += _jpeg_segment(0xDB, bytes([i]) + qt[i].tobytes())
    out += _jpeg_segment(0xC0, bytes([8]) + int(H).to_bytes(2, "big") + int(W).to_bytes(2, "big")
                         + bytes([3, 1, 0x22, 0, 2, 0x11, 1, 3, 0x11, 1]))
    for tc, bits, vals in _JPEG_STD_HUFF:
        out += _jpeg_segment(0xC4, bytes([tc]) + bytes.fromhex(bits) + bytes.fromhex(vals))
    return out + _jpeg_segment(0xDA, bytes([3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0]))


# ----------------------------------------------------------------------------- PNG (K10)
PNG_SIGNATURE = b"\x89PNG\r\n\x1a\n"


def _png_chunk(kind: bytes, payload: bytes) -> bytes:
    import zlib
    return len(payload).to_bytes(4, "big") + kind + payload + zlib.crc32(kind + payload).to_bytes(4, "big")


def png_header(H: int, W: int) -> bytes:
    """Every byte of cv2.imencode(".png") that depends only on the frame size: the signature, the IHDR chunk (depth 8,
    colour type 2, no interlace) and the two zlib header bytes that open the first IDAT payload.  zlib writes 78 01
    (32K window, level 1); libpng's optimize_cmf then lowers the window to the smallest that holds the image data
    when that data (H rows of 3W + 1 filtered bytes) is at most 16384 bytes."""
    H, W = int(H), int(W)
    if not (1 <= H <= 65535 and 1 <= W <= 65535):
        raise ValueError(f"PNG frame size must lie in [1, 65535]^2, got {H}x{W}")
    size = H * (3 * W + 1)
    cmf, flg = 0x78, 0x01
    if size <= 16384:
        cinfo, half = 7, 1 << 14
        while cinfo > 0 and size <= half:     # optimize_cmf: halve the window while the data still fits in half
            half >>= 1
            cinfo -= 1
        cmf = (cinfo << 4) | 8
        flg = 0x1F - (cmf << 8) % 0x1F
    ihdr = W.to_bytes(4, "big") + H.to_bytes(4, "big") + bytes([8, 2, 0, 0, 0])
    return PNG_SIGNATURE + _png_chunk(b"IHDR", ihdr) + bytes([cmf, flg])


# ----------------------------------------------------------------------------- split-compare labels (K9)
SPLIT_LABEL_MARGIN = 16            # rows drawn below the lowest label rectangle; they must come out untouched
SPLIT_CLASS_INDEX = np.uint16      # class map dtype (K9 reads uint16)


class SplitLabelStencil(NamedTuple):
    band_rows: int                 # rows [0, band_rows) hold every pixel the labels change
    classes: np.ndarray            # [band_rows, W] SPLIT_CLASS_INDEX: table of each pixel, 0 = identity
    luts: np.ndarray               # [n_classes, 256] uint8: byte b of a pixel of class c becomes luts[c, b]


@lru_cache(maxsize=64)
def split_label_stencil(H: int, W: int, left: str, right: str) -> SplitLabelStencil:
    """`draw_split_labels(frame, left, right)` of an H x W frame as a per-pixel byte map.

    Every step of the label drawing (addWeighted of a black overlay, anti-aliased putText towards two constant grey
    colours) maps one byte of one pixel to one byte of the same pixel and channel, the same way for all three channels.
    So the drawing is out[y, x, c] = F_(y,x)(in[y, x, c]), and F is found by drawing on constant canvases: draw k
    carries the values 3k, 3k + 1, 3k + 2 in the three channels, so 86 draws give all 256 inputs.  Only the top rows
    are drawn (the label rectangles' bottom row plus SPLIT_LABEL_MARGIN rows, with the geometry of the full frame), so
    the cost grows with the band, not the frame; the margin rows must come out unchanged, which shows that no stroke
    was clipped by the shorter canvas.  Pixels sharing a table share a class."""
    from .renderers.video import draw_label_boxes, split_label_geometry
    H, W = int(H), int(W)
    if H < 1 or W < 1:
        raise ValueError(f"split_label_stencil: frame size {H}x{W}")
    boxes = split_label_geometry(H, W, left, right)
    R = min(H, max(b.rect[3] for b in boxes) + 1 + SPLIT_LABEL_MARGIN)
    lut = np.empty((258, R, W), np.uint8)                       # lut[v, y, x]: what the drawing makes of byte v
    canvas = np.empty((R, W, 3), np.uint8)
    for k in range(86):
        canvas[:] = np.minimum(np.arange(3 * k, 3 * k + 3), 255).astype(np.uint8)
        draw_label_boxes(canvas, boxes)
        lut[3 * k:3 * k + 3] = canvas.transpose(2, 0, 1)
    lut = lut[:256]
    for v in (0, 1, 127, 128, 254, 255):                        # grey canvases: the channels must agree with the table
        canvas[:] = v
        draw_label_boxes(canvas, boxes)
        if not (np.array_equal(canvas[..., 0], canvas[..., 1]) and np.array_equal(canvas[..., 0], canvas[..., 2])
                and np.array_equal(canvas[..., 0], lut[v])):
            raise ValueError("split_label_stencil: the label drawing treats the three channels differently "
                             "(a label colour that is not grey); it has no per-pixel byte table")
    changed = (lut != np.arange(256, dtype=np.uint8)[:, None, None]).any(axis=0)      # [R, W]
    if R < H and changed[R - SPLIT_LABEL_MARGIN:].any():
        raise ValueError("split_label_stencil: the labels reach the margin below their rectangles")
    rows = np.flatnonzero(changed.any(axis=1))
    band = int(rows[-1]) + 1 if rows.size else 0
    rows256 = np.ascontiguousarray(lut[:, changed].T)                                 # [changed pixels, 256]
    keys, inverse = np.unique(rows256.view(np.dtype((np.void, 256))).ravel(), return_inverse=True)
    tabs = np.frombuffer(keys.tobytes(), np.uint8).reshape(-1, 256)
    if tabs.shape[0] + 1 > int(np.iinfo(SPLIT_CLASS_INDEX).max) + 1:
        raise ValueError(f"split_label_stencil: {tabs.shape[0] + 1} tables do not fit a {np.dtype(SPLIT_CLASS_INDEX)} "
                         "class index")
    classes = np.zeros((R, W), SPLIT_CLASS_INDEX)
    classes[changed] = inverse.reshape(-1) + 1
    luts = np.concatenate([np.arange(256, dtype=np.uint8)[None], tabs])
    classes = np.ascontiguousarray(classes[:band])
    classes.flags.writeable = False
    luts.flags.writeable = False
    return SplitLabelStencil(band, classes, luts)
