"""CPU restatement of OpenCV's cv::CLAHE::apply (modules/imgproc/src/clahe.cpp) on one plane, the parity reference of the CLAHE
tests and smoke().  Histogram size hs = 2^bits; samples above hs - 1 count as hs - 1.  All float arithmetic is f32, one rounding per
multiply and per add, as in OpenCV.  Pinned against cv2 by test_clahe_host.py."""
import numpy as np

F = np.float32


def _reflect101(p, n):
    """cv::borderInterpolate(p, n, BORDER_REFLECT_101) for an array of indices p >= 0."""
    if n == 1:
        return np.zeros_like(p)
    p = p.copy()
    while True:
        out = p >= n
        if not out.any():
            return p
        p[out] = 2 * n - 2 - p[out]
        p = np.abs(p)


def _tile_terms(n, tile, tiles):
    """First / second tile and the weights along one axis (column or row positions 0..n-1)."""
    f = (np.arange(n, dtype=F) * (F(1) / F(tile))).astype(F) - F(0.5)
    t1 = np.floor(f).astype(np.int64)
    a = (f - t1.astype(F)).astype(F)
    return np.maximum(t1, 0), np.minimum(t1 + 1, tiles - 1), a, (F(1) - a).astype(F)


def clahe_plane(src: np.ndarray, bits: int, limit=15.0, tiles=(3, 3)) -> np.ndarray:
    h, w = src.shape
    tx, ty = int(tiles[0]), int(tiles[1])
    hs = 1 << bits
    s = np.minimum(src.astype(np.int64), hs - 1)
    # both axes are padded (by a whole tile on an axis that divides) as soon as one does not divide
    pad = w % tx != 0 or h % ty != 0
    pw, ph = (w + tx - w % tx, h + ty - h % ty) if pad else (w, h)
    tw, th = pw // tx, ph // ty
    n = tw * th
    ext = s[_reflect101(np.arange(ph), h)][:, _reflect101(np.arange(pw), w)]
    tiles_ = ext.reshape(ty, th, tx, tw).transpose(0, 2, 1, 3).reshape(ty * tx, n)
    hist = np.bincount((tiles_ + (np.arange(ty * tx) * hs)[:, None]).ravel(), minlength=ty * tx * hs).reshape(ty * tx, hs)
    if limit > 0:
        c = limit * n / hs
        clip = 2147483647 if c >= 2147483647.0 else max(int(c), 1)
        clipped = np.maximum(hist - clip, 0).sum(axis=1)
        hist = np.minimum(hist, clip) + (clipped // hs)[:, None]
        i = np.arange(hs)
        for t, res in enumerate(clipped % hs):
            if res:  # OpenCV's residual loop: one count to bins 0, step, 2 step, ... (res of them)
                step = max(hs // int(res), 1)
                hist[t] += (i % step == 0) & (i // step < res)
    scale = F(hs - 1) / F(n)
    lut = np.clip(np.rint((np.cumsum(hist, axis=1).astype(F) * scale).astype(F)), 0, hs - 1).astype(F)
    x1, x2, xa, xa1 = _tile_terms(w, tw, tx)
    y1, y2, ya, ya1 = _tile_terms(h, th, ty)
    Y1, Y2 = (y1 * tx)[:, None], (y2 * tx)[:, None]
    l11, l12 = lut[Y1 + x1[None, :], s], lut[Y1 + x2[None, :], s]
    l21, l22 = lut[Y2 + x1[None, :], s], lut[Y2 + x2[None, :], s]
    top = ((l11 * xa1).astype(F) + (l12 * xa).astype(F)).astype(F)
    bot = ((l21 * xa1).astype(F) + (l22 * xa).astype(F)).astype(F)
    res = ((top * ya1[:, None]).astype(F) + (bot * ya[:, None]).astype(F)).astype(F)
    return np.clip(np.rint(res), 0, hs - 1).astype(src.dtype)
