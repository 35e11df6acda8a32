"""align2d_kernel bit for bit against a NumPy float32 restatement of its exact operation order: the reference's weight expressions
(two in fp64, narrowed), each column summed sequentially over the four rows of its row group, the Jres tree (row groups, then
columns c ^ 4, c ^ 2, c ^ 1), the Hinv rows left to right. Every NumPy float32 operation is one IEEE round-to-nearest operation
and no multiply-add is fused, as on the device."""
import numpy as np
import pytest

import helpers as H
import oracle as O

pytestmark = pytest.mark.gpu

F = np.float32


def restated_align2d(img, p10, max_iters, px):
    """-> (u, v) as float64 and the converged flag"""
    rows, cols = img.shape
    flat = img.reshape(-1)
    p = p10.reshape(10, 10).astype(np.int64)
    ddx = p[1:9, 2:10] - p[1:9, 0:8]
    ddy = p[2:10, 1:9] - p[0:8, 1:9]
    rdx = F(0.5) * ddx.astype(F)
    rdy = F(0.5) * ddy.astype(F)
    rref = p[1:9, 1:9].astype(F)
    h00, h01, h02 = F(0.25) * F((ddx * ddx).sum()), F(0.25) * F((ddx * ddy).sum()), F(0.5) * F(ddx.sum())
    h11, h12, h22 = F(0.25) * F((ddy * ddy).sum()), F(0.5) * F(ddy.sum()), F(64)
    m = [[h00, h01, h02], [h01, h11, h12], [h02, h12, h22]]

    def cof(i, j):
        return m[(i + 1) % 3][(j + 1) % 3] * m[(i + 2) % 3][(j + 2) % 3] - m[(i + 1) % 3][(j + 2) % 3] * m[(i + 2) % 3][(j + 1) % 3]
    c00, c10, c20 = cof(0, 0), cof(1, 0), cof(2, 0)
    det = (c00 * m[0][0] + c10 * m[1][0]) + c20 * m[2][0]
    invdet = F(1) / det
    Hi = [c00 * invdet, c10 * invdet, c20 * invdet, cof(0, 1) * invdet, cof(1, 1) * invdet, cof(2, 1) * invdet,
          cof(0, 2) * invdet, cof(1, 2) * invdet, cof(2, 2) * invdet]

    def tree(S):                     # S[g, c]: column c summed over the rows of row group g
        T = S[0] + S[1]
        U = T + T[np.arange(8) ^ 4]
        V = U + U[np.arange(8) ^ 2]
        return V[0] + V[1]

    u, v = F(px[0]), F(px[1])
    mean_diff = F(0)
    conv = False
    rr, cc = np.mgrid[0:9, 0:9]
    for _ in range(max_iters):
        uf, vf = np.floor(u), np.floor(v)
        if not (uf >= 4 and vf >= 4 and uf <= cols - 4 and vf <= rows - 4):
            break
        u_r, v_r = int(uf), int(vf)
        sx, sy = u - uf, v - vf
        wTL = F((1.0 - np.float64(sx)) * (1.0 - np.float64(sy)))
        wTR = sx * (F(1) - sy)
        wBL = F((1.0 - np.float64(sx)) * np.float64(sy))
        wBR = sx * sy
        o = (v_r + rr - 4) * cols + (u_r - 4 + cc)             # linear addressing, zeros past the end of the level (Q4)
        T = np.where(o < flat.size, flat[np.minimum(o, flat.size - 1)], 0).astype(F)
        s = ((wTL * T[:8, :8] + wTR * T[:8, 1:]) + wBL * T[1:, :8]) + wBR * T[1:, 1:]
        res = (s - rref) + mean_diff
        j = np.zeros((3, 2, 8), F)
        for k in range(4):
            r = res[[k, 4 + k]]
            j[0] = j[0] - r * rdx[[k, 4 + k]]
            j[1] = j[1] - r * rdy[[k, 4 + k]]
            j[2] = j[2] - r
        J0, J1, J2 = tree(j[0]), tree(j[1]), tree(j[2])
        d0 = (Hi[0] * J0 + Hi[1] * J1) + Hi[2] * J2
        d1 = (Hi[3] * J0 + Hi[4] * J1) + Hi[5] * J2
        d2 = (Hi[6] * J0 + Hi[7] * J1) + Hi[8] * J2
        u, v, mean_diff = u + d0, v + d1, mean_diff + d2
        if d0 * d0 + d1 * d1 < F(0.03 * 0.03):
            conv = True
            break
    return np.array([u, v], np.float64), conv


def _check(ctx, sc, levels, patches, start, iters):
    packed, offs, ws, hs = sc["cur_pyr"]
    px, conv = ctx.align2d(1, levels, patches, start, iters)
    for i in range(len(levels)):
        if levels[i] < 0:
            assert not conv[i] and (px[i].view(np.uint64) == np.asarray(start[i], np.float64).view(np.uint64)).all(), i
            continue
        img = O.pyr_level(packed, offs, ws, hs, int(levels[i]))
        with np.errstate(invalid="ignore", over="ignore"):
            p, c = restated_align2d(img, patches[i], iters, start[i])
        assert c == conv[i], i
        assert (p.view(np.uint64) == px[i].view(np.uint64)).all(), (i, p, px[i])


@pytest.mark.parametrize("iters", [3, 10])
def test_align2d_bits_300_patches(ctx, scenario, iters):
    ctx.upload(1, scenario["cur_img"])
    levels, patches, truth, start = H.make_patches(scenario["cur_pyr"], 300, 21, max_level=2)
    _check(ctx, scenario, levels, patches, start, iters)


def test_align2d_bits_border_nan_q4(ctx, scenario):
    ctx.upload(1, scenario["cur_img"])
    rng = np.random.default_rng(4)
    starts = np.array([[636.3, 200.2], [300.5, 476.4], [636.0, 476.0], [3.9, 100.0], [100.0, 3.2], [637.2, 50.0], [50.0, 477.1],
                       [np.nan, 100.0], [1e9, 5.0], [4.0, 4.0], [-5.0, 30.0]])
    patches = rng.integers(0, 256, (len(starts), 100), dtype=np.uint8)
    _check(ctx, scenario, np.zeros(len(starts), np.int32), patches, starts, 10)


@pytest.mark.parametrize("n", [1, 2, 3, 5, 37])
def test_align2d_bits_partial_warps_and_unused(ctx, scenario, n):
    """batches that end inside a warp of four patches (missing groups shadow the last patch and must not write), with unused
    (level < 0) entries at several positions of a warp"""
    ctx.upload(1, scenario["cur_img"])
    levels, patches, truth, start = H.make_patches(scenario["cur_pyr"], n, 100 + n, max_level=2)
    for j in (1, 6, n - 1):
        if n >= 3 and j < n:
            levels[j] = -1
    _check(ctx, scenario, levels, patches, start, 10)
