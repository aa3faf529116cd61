"""TEST INFRASTRUCTURE ONLY (oracle): `TextBlock.get_transformed_region(img, idx, textheight)` (reference
utils/textblock.py:162-194) -- the crop of one text line, straightened by a homography, that a downstream OCR stage
reads.

Two restatements live here:
  * `get_transformed_region` / `transformed_regions`: the reference's geometry (quad expansion, clip, aspect ratio,
    output size) followed by the very cv2 calls it makes (`findHomography(src, dst, RANSAC, 5.0)`,
    `warpPerspective(img, M, (w, h))`, `rotate(.., ROTATE_90_COUNTERCLOCKWISE)` for vertical lines).  A failing line
    raises what the reference raises.
  * `homography_4pt` / `warp_perspective_u8`: numpy restatements of what those two cv2 calls compute for four points
    and an 8-bit image, i.e. the arithmetic csrc/regions.cu implements.  OpenCV 4.x is an un-vendored binary here, so
    both are PINNED against the installed cv2 itself (tests/test_cpu_regions.py):
      - findHomography with exactly 4 points skips RANSAC and runs the normalised DLT kernel on float32 points: each
        side is shifted to its centroid and scaled by count / sum|p - c| per axis (a zero spread fails -> None), the
        9x9 LtL is accumulated, the eigenvector of its smallest eigenvalue (OpenCV's pivoting Jacobi) is de-normalised and scaled by 1/H[2][2]
        (skipped when |H[2][2]| <= FLT_EPSILON, e.g. three corners collinear after the clip);
      - warpPerspective inverts M in double (lapack.cpp's 3x3 cofactor formula; a singular M becomes all zeros) and
        maps every output pixel through it in blocks of bw0 = min(1024 / min(16, h), w) columns:
        X0 = Mi0*xb + Mi1*y + Mi2 at the block's first column xb, then per column W = W0 + Mi6*x1, W = W ? 32/W : 0,
        X = cvRound((X0 + Mi0*x1) * W) (INTER_BITS = 5; same for Y).  The integer part (X >> 5) picks the top-left tap,
        the 5-bit fractions pick a bilinear weight quadruple of a 32x32 int16 table (weights sum to 32768), and
        dst = (sum w*p + 2^14) >> 15.  Taps outside the page read 0 (BORDER_CONSTANT).
Nothing under comic-text-detector_b200/ imports this module.
"""
import math

import numpy as np

INTER_BITS = 5
TAB = 1 << INTER_BITS
INT_MIN, INT_MAX = float(-2 ** 31), float(2 ** 31 - 1)
EPS = float(np.finfo(np.float64).eps)
FLT_EPSILON = float(np.finfo(np.float32).eps)


# ---- the reference's geometry (textblock.py:163-186) ------------------------------------------------------------------
def expands(language, vertical):
    """textblock.py:168: the quad is grown by font_size / 3 for English lines and for horizontal lines of unknown
    language."""
    return language == "eng" or (language == "unknown" and not vertical)


def line_geometry(line, expand, vertical, font_size, im_w, im_h, textheight):
    """-> (src_pts float64 [4,2], w, h) exactly as the reference computes them; raises where the reference raises
    (OverflowError / ValueError from round() when the aspect ratio is 0, inf or nan)."""
    src_pts = np.array(line, dtype=np.float64)
    if expand:
        e_size = font_size / 3
        src_pts[..., 0] += np.array([-e_size, e_size, e_size, -e_size])
        src_pts[..., 1] += np.array([-e_size, -e_size, e_size, e_size])
        src_pts[..., 0] = np.clip(src_pts[..., 0], 0, im_w)
        src_pts[..., 1] = np.clip(src_pts[..., 1], 0, im_h)
    middle_pnt = (src_pts[[1, 2, 3, 0]] + src_pts) / 2
    vec_v = middle_pnt[2] - middle_pnt[0]
    vec_h = middle_pnt[1] - middle_pnt[3]
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.linalg.norm(vec_v) / np.linalg.norm(vec_h)
        if vertical:
            w = int(textheight)
            h = int(round(textheight * ratio))
        else:
            h = int(textheight)
            w = int(round(textheight / ratio))
    return src_pts, w, h


def dst_points(w, h):
    return np.array([[0, 0], [w - 1, 0], [w - 1, h - 1], [0, h - 1]]).astype(np.float32)


def get_transformed_region(blk, img, idx, textheight):
    """The reference method with cv2 (raises where it raises: OverflowError / ValueError from round(), cv2.error from
    warpPerspective when findHomography returns None)."""
    import cv2
    im_h, im_w = img.shape[:2]
    src_pts, w, h = line_geometry(blk.lines[idx], expands(blk.language, blk.vertical), blk.vertical, blk.font_size,
                                  im_w, im_h, textheight)
    M, _ = cv2.findHomography(src_pts, dst_points(w, h), cv2.RANSAC, 5.0)
    region = cv2.warpPerspective(img, M, (w, h))
    if blk.vertical:
        region = cv2.rotate(region, cv2.ROTATE_90_COUNTERCLOCKWISE)
    return region


def transformed_regions(img, blk_list, textheight):
    """what `TextDetector.get_transformed_regions` returns: per block a list of crops, None where the reference
    raises."""
    out = []
    for blk in blk_list:
        row = []
        for i in range(len(blk.lines)):
            try:
                row.append(get_transformed_region(blk, img, i, textheight))
            except Exception:
                row.append(None)
        out.append(row)
    return out


# ---- numpy restatement of cv2.findHomography for 4 points (calib3d/src/fundam.cpp, HomographyEstimatorCallback) -------
def cv_hypot(a, b):
    """lapack.cpp's own hypot, which JacobiImpl_ calls (not libm's): with libm's, M differs from cv2's in the last bits"""
    a, b = abs(a), abs(b)
    if a > b:
        b /= a
        return a * math.sqrt(1 + b * b)
    if b > 0:
        a /= b
        return b * math.sqrt(1 + a * a)
    return 0.0


def jacobi_smallest(A):
    """cv::eigen of a symmetric matrix (core/src/lapack.cpp JacobiImpl_: the largest off-diagonal element is rotated
    away until it is <= DBL_EPSILON, eigenvalues sorted descending) -> the eigenvector of the smallest eigenvalue."""
    n = len(A)
    A = [[float(v) for v in r] for r in A]
    V = [[1.0 if i == j else 0.0 for j in range(n)] for i in range(n)]
    W = [A[k][k] for k in range(n)]
    indR, indC = [0] * n, [0] * n

    def row_max(k):
        m, mv = k + 1, abs(A[k][k + 1])
        for i in range(k + 2, n):
            if mv < abs(A[k][i]):
                mv, m = abs(A[k][i]), i
        indR[k] = m

    def col_max(k):
        m, mv = 0, abs(A[0][k])
        for i in range(1, k):
            if mv < abs(A[i][k]):
                mv, m = abs(A[i][k]), i
        indC[k] = m

    for k in range(n):
        if k < n - 1:
            row_max(k)
        if k > 0:
            col_max(k)
    for _ in range(n * n * 30):
        k, mv = 0, abs(A[0][indR[0]])
        for i in range(1, n - 1):
            if mv < abs(A[i][indR[i]]):
                mv, k = abs(A[i][indR[i]]), i
        l = indR[k]
        for i in range(1, n):
            if mv < abs(A[indC[i]][i]):
                mv, k, l = abs(A[indC[i]][i]), indC[i], i
        p = A[k][l]
        if abs(p) <= EPS:
            break
        y = (W[l] - W[k]) * 0.5
        t = abs(y) + cv_hypot(p, y)
        s = cv_hypot(p, t)
        c = t / s
        s = p / s
        t = (p / t) * p
        if y < 0:
            s, t = -s, -t
        A[k][l] = 0.0
        W[k] -= t
        W[l] += t

        def rot(a0, b0):
            return a0 * c - b0 * s, a0 * s + b0 * c
        for i in range(0, k):
            A[i][k], A[i][l] = rot(A[i][k], A[i][l])
        for i in range(k + 1, l):
            A[k][i], A[i][l] = rot(A[k][i], A[i][l])
        for i in range(l + 1, n):
            A[k][i], A[l][i] = rot(A[k][i], A[l][i])
        for i in range(n):
            V[k][i], V[l][i] = rot(V[k][i], V[l][i])
        for idx in (k, l):
            if idx < n - 1:
                row_max(idx)
            if idx > 0:
                col_max(idx)
    for k in range(n - 1):
        m = k
        for i in range(k + 1, n):
            if W[m] < W[i]:
                m = i
        if k != m:
            W[m], W[k] = W[k], W[m]
            V[m], V[k] = V[k], V[m]
    return np.array(V[n - 1])


def _mul3(A, B):
    """3x3 product, every element summed k = 0, 1, 2 from 0 (cv::gemm)"""
    return np.array([[((0.0 + A[i][0] * B[0][j]) + A[i][1] * B[1][j]) + A[i][2] * B[2][j] for j in range(3)]
                     for i in range(3)])


def homography_4pt(src, dst):
    """-> 3x3 float64 H or None (a zero spread of either point set along x or y).  Scalar python floats, in OpenCV's
    order of evaluation."""
    M = [[float(v) for v in r] for r in np.asarray(src, np.float64).astype(np.float32)]
    m = [[float(v) for v in r] for r in np.asarray(dst, np.float64).astype(np.float32)]
    n = len(M)
    cm, cM = [0.0, 0.0], [0.0, 0.0]
    for i in range(n):
        for a in range(2):
            cm[a] += m[i][a]
            cM[a] += M[i][a]
    cm, cM = [v / n for v in cm], [v / n for v in cM]
    sm, sM = [0.0, 0.0], [0.0, 0.0]
    for i in range(n):
        for a in range(2):
            sm[a] += abs(m[i][a] - cm[a])
            sM[a] += abs(M[i][a] - cM[a])
    if min(abs(sm[0]), abs(sm[1]), abs(sM[0]), abs(sM[1])) < EPS:
        return None
    sm, sM = [n / v for v in sm], [n / v for v in sM]
    inv_hnorm = [[1.0 / sm[0], 0.0, cm[0]], [0.0, 1.0 / sm[1], cm[1]], [0.0, 0.0, 1.0]]
    hnorm2 = [[sM[0], 0.0, -cM[0] * sM[0]], [0.0, sM[1], -cM[1] * sM[1]], [0.0, 0.0, 1.0]]
    LtL = [[0.0] * 9 for _ in range(9)]
    for i in range(n):
        x, y = (m[i][0] - cm[0]) * sm[0], (m[i][1] - cm[1]) * sm[1]
        X, Y = (M[i][0] - cM[0]) * sM[0], (M[i][1] - cM[1]) * sM[1]
        Lx = [X, Y, 1.0, 0.0, 0.0, 0.0, -x * X, -x * Y, -x]
        Ly = [0.0, 0.0, 0.0, X, Y, 1.0, -y * X, -y * Y, -y]
        for j in range(9):
            for k in range(j, 9):
                LtL[j][k] += Lx[j] * Lx[k] + Ly[j] * Ly[k]
    for j in range(9):
        for k in range(j):
            LtL[j][k] = LtL[k][j]
    h0 = jacobi_smallest(LtL).reshape(3, 3)
    H = _mul3(_mul3(inv_hnorm, h0), hnorm2)
    if abs(H[2, 2]) > FLT_EPSILON:     # cv2 leaves a nearly degenerate H (|H22| <= FLT_EPSILON) unscaled
        return H * (1.0 / H[2, 2])
    return H


def invert3(M):
    """cv::invert(M, DECOMP_LU) for a 3x3 double matrix (core/src/lapack.cpp): cofactors times 1/det, evaluated in the
    same order; a singular matrix gives all zeros."""
    s = [float(v) for v in np.asarray(M, np.float64).reshape(9)]
    S = lambda r, c: s[r * 3 + c]  # noqa: E731
    d = S(0, 0) * (S(1, 1) * S(2, 2) - S(1, 2) * S(2, 1)) - S(0, 1) * (S(1, 0) * S(2, 2) - S(1, 2) * S(2, 0)) + \
        S(0, 2) * (S(1, 0) * S(2, 1) - S(1, 1) * S(2, 0))
    if d == 0.0:
        return np.zeros((3, 3))
    d = 1.0 / d
    t = [(S(1, 1) * S(2, 2) - S(1, 2) * S(2, 1)) * d, (S(0, 2) * S(2, 1) - S(0, 1) * S(2, 2)) * d,
         (S(0, 1) * S(1, 2) - S(0, 2) * S(1, 1)) * d,
         (S(1, 2) * S(2, 0) - S(1, 0) * S(2, 2)) * d, (S(0, 0) * S(2, 2) - S(0, 2) * S(2, 0)) * d,
         (S(0, 2) * S(1, 0) - S(0, 0) * S(1, 2)) * d,
         (S(1, 0) * S(2, 1) - S(1, 1) * S(2, 0)) * d, (S(0, 1) * S(2, 0) - S(0, 0) * S(2, 1)) * d,
         (S(0, 0) * S(1, 1) - S(0, 1) * S(1, 0)) * d]
    return np.array(t).reshape(3, 3)


def bilinear_table():
    """int16 [32*32][4] weights of (top-left, top-right, bottom-left, bottom-right) for fractions (fy, fx); every
    product (1 - i/32)(1 - j/32) * 32768 is an exact integer, so the table needs no sum correction."""
    i = np.arange(TAB)[:, None]
    j = np.arange(TAB)[None, :]
    t = np.stack([(TAB - i) * (TAB - j), (TAB - i) * j, i * (TAB - j), i * j], -1) * (32768 // (TAB * TAB))
    return t.reshape(TAB * TAB, 4).astype(np.int32)


def warp_coords(Mi, h, w):
    """fixed-point source coordinates (X, Y) = cvRound(32 * (x', y')) of every output pixel, int64 [h, w]."""
    Mi = [float(v) for v in np.asarray(Mi, np.float64).reshape(9)]
    bh0 = min(TAB * TAB // 2 // TAB, h)          # min(16, h)
    bw0 = min(TAB * TAB // bh0, w)               # columns per block (BLOCK_SZ*BLOCK_SZ / bh0)
    x = np.arange(w, dtype=np.int64)[None, :]
    y = np.arange(h, dtype=np.float64)[:, None]
    xb = ((x // bw0) * bw0).astype(np.float64)
    x1 = (x - (x // bw0) * bw0).astype(np.float64)
    X0 = Mi[0] * xb + Mi[1] * y + Mi[2]
    Y0 = Mi[3] * xb + Mi[4] * y + Mi[5]
    W0 = Mi[6] * xb + Mi[7] * y + Mi[8]
    W = W0 + Mi[6] * x1
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        W = np.where(W != 0, TAB / np.where(W != 0, W, 1.0), 0.0)
        fX = np.maximum(INT_MIN, np.minimum(INT_MAX, (X0 + Mi[0] * x1) * W))
        fY = np.maximum(INT_MIN, np.minimum(INT_MAX, (Y0 + Mi[3] * x1) * W))
    return np.rint(fX).astype(np.int64), np.rint(fY).astype(np.int64)


def warp_perspective_u8(img, M, dsize_wh):
    """cv2.warpPerspective(img, M, dsize_wh) (INTER_LINEAR, BORDER_CONSTANT 0) for uint8 [H,W] / [H,W,C]; an empty
    dsize means the page's size, as in OpenCV."""
    img = np.asarray(img)
    assert img.dtype == np.uint8
    squeeze = img.ndim == 2
    src = img[:, :, None] if squeeze else img
    ih, iw, c = src.shape
    w, h = int(dsize_wh[0]), int(dsize_wh[1])
    if w <= 0 or h <= 0:
        w, h = iw, ih
    X, Y = warp_coords(invert3(M), h, w)
    sx = np.clip(X >> INTER_BITS, -32768, 32767)
    sy = np.clip(Y >> INTER_BITS, -32768, 32767)
    wt = bilinear_table()[((Y & (TAB - 1)) * TAB + (X & (TAB - 1)))]            # [h, w, 4]
    acc = np.zeros((h, w, c), np.int64)
    for k, (dy, dx) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):
        yy, xx = sy + dy, sx + dx
        inside = (xx >= 0) & (xx < iw) & (yy >= 0) & (yy < ih)
        p = src[np.clip(yy, 0, ih - 1), np.clip(xx, 0, iw - 1)].astype(np.int64)
        acc += np.where(inside[..., None], p, 0) * wt[..., k, None]
    out = np.clip((acc + (1 << 14)) >> 15, 0, 255).astype(np.uint8)
    return out[:, :, 0] if squeeze else out
