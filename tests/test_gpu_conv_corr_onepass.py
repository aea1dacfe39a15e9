"""One-pass correlation Grams of 3x3 conv layers: G1 = Xq X^T is read as x centre x an xq window below it (the point
reflection of G2's xq centre x xq window above it), so its records are split by the region of the x pixel.  These tests
give x and xq different supports, signs and image splits, and compare every Gram entry with an fp64 patch-form Gram."""
import contextlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
RTOL = 1e-15   # relative to |Xq| |X|^T: fp64 re-association of the same exact fp32 x fp32 products


def patch_gram(act, actq):
    """(C, 2, 9, 9) fp64 [G1 | G2] of the 3x3 'SAME' patch matrices, lower triangles, and the |Xq||X|^T bounds."""
    n, H, Wd, C = act.shape
    # extended-precision sums of the exact fp32 x fp32 products: the reference adds no re-association error of its own
    pad = lambda a: np.pad(a.astype(np.longdouble), ((0, 0), (1, 1), (1, 1), (0, 0)))
    px, pq = pad(act), pad(actq)
    P = lambda p, c: np.stack([p[:, ty:ty + H, tx:tx + Wd, c].ravel() for ty in range(3) for tx in range(3)])
    g, b = np.zeros((C, 2, 9, 9)), np.zeros((C, 2, 9, 9))
    low = np.tril(np.ones((9, 9), dtype=bool))
    for c in range(C):
        X, Xq = P(px, c), P(pq, c)
        for k, (A, B) in enumerate(((Xq, X), (Xq, Xq))):
            g[c, k] = np.where(low, np.einsum("ip,jp->ij", A, B).astype(np.float64), 0.0)
            b[c, k] = np.where(low, np.einsum("ip,jp->ij", np.abs(A), np.abs(B)).astype(np.float64), 0.0)
    return g, b


@contextlib.contextmanager
def options(engine, **opts):
    for k, v in opts.items():
        engine.set_option(k, v)
    try:
        yield
    finally:
        for k in opts:
            engine.set_option(k, 0)


def gram(engine, act, actq, **opts):
    with options(engine, **opts):
        g = engine.conv_gram_nhwc(act, actq).cpu().numpy()
    # the correlation form ran (4: straight from the activations, 5: packed images), not a patch-form fallback
    assert engine.last_stats["gram_kernel"] == (5 if opts.get("corr_pack") == 1 else 4), (opts, engine.last_stats["gram_kernel"])
    return g


def check(G, ref, bound, what):
    low = np.tril(np.ones((9, 9), dtype=bool))
    G = np.where(low, G, 0.0)
    err = np.abs(G - ref)
    assert np.all(err <= RTOL * bound), (what, float((err / np.maximum(bound, 1e-300)).max()))
    # an entry that is an empty sum or a sum of zero products in the patch form is a literal zero here
    assert np.all(G[ref == 0] == 0), (what, int(np.count_nonzero(G[ref == 0])))


# the band kernel (widths not a multiple of 5, so the last 5-column stage is ragged), the strip kernels (14, 28: two passes;
# 8: one pass) and the band kernel forced onto the strip widths
RUNS = {"direct": dict(corr_small=1, corr_pack=2), "band": dict(corr_small=1, corr_pack=2, corr_strip=2),
        "rows4": dict(corr_small=1, corr_pack=2, corr_rows=4), "rows6": dict(corr_small=1, corr_pack=2, corr_rows=6),
        "rows8": dict(corr_small=1, corr_pack=2, corr_rows=8)}


@pytest.mark.parametrize("H,Wd", [(6, 13), (7, 7), (9, 11), (14, 14), (28, 28), (112, 17), (8, 8), (11, 8)])
def test_onepass_gram_matches_patch_form(engine, H, Wd):
    rng = np.random.default_rng(H * 1000 + Wd)
    n_img, C = 3, 40
    act = np.maximum(rng.standard_normal((n_img, H, Wd, C)), 0).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    # signed channels: G1 entries with cancellation, and x / xq of opposite signs
    act[..., 5] = rng.standard_normal((n_img, H, Wd)).astype(np.float32)
    actq[..., 5] = (act[..., 5] + 0.1 * rng.standard_normal((n_img, H, Wd))).astype(np.float32)
    act[..., 6] = rng.standard_normal((n_img, H, Wd)).astype(np.float32)
    actq[..., 6] = -act[..., 6]
    # different dead borders: x lives on the bottom row only (xq dense), xq on the right column only (x dense), and
    # x on the top row / xq on the left column
    act[:, :-1, :, 1] = 0
    actq[:, :, :-1, 2] = 0
    act[:, 1:, :, 3] = 0
    actq[:, :, 1:, 4] = 0
    ref, bound = patch_gram(act, actq)
    for name, opts in RUNS.items():
        check(gram(engine, act, actq, **opts), ref, bound, (name, H, Wd))
    # packed images (few channels: G images side by side as virtual channels)
    sub = np.ascontiguousarray(act[..., :6]), np.ascontiguousarray(actq[..., :6])
    check(gram(engine, *sub, corr_pack=1), ref[:6], bound[:6], ("packed", H, Wd))


@pytest.mark.parametrize("H,Wd", [(112, 23), (28, 28), (8, 8)])
def test_onepass_gram_image_split(engine, H, Wd):
    """One image set split two ways: the two Grams summed by hand equal the one-call Gram (and the patch form)."""
    rng = np.random.default_rng(H + Wd)
    n_img, C = 5, 32
    act = rng.standard_normal((n_img, H, Wd, C)).astype(np.float32)
    actq = np.maximum(act + 0.05 * rng.standard_normal(act.shape), 0).astype(np.float32)
    act[:, :-1, :, 7] = 0
    ref, bound = patch_gram(act, actq)
    whole = gram(engine, act, actq)
    check(whole, ref, bound, "whole")
    for k in (1, 3):
        a = gram(engine, np.ascontiguousarray(act[:k]), np.ascontiguousarray(actq[:k]))
        b = gram(engine, np.ascontiguousarray(act[k:]), np.ascontiguousarray(actq[k:]))
        check(a + b, ref, bound, ("split", k))
        check(a + b, whole, bound, ("split vs whole", k))
