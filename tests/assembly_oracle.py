"""TEST INFRASTRUCTURE — restatement of the assembly mass properties (DESIGN.md 4.11,
cc_assembly_mass_properties_exact) on top of the C oracle's per-block evaluation: oracle.host.mass_properties'
hierarchy and Kahan sums, with every block carrying the parts undecided at its parent cell (`eval`) and the parts
decided inside at an ancestor cell (`inside`), one set of sums per part and per pair of parts."""
import math

import numpy as np

import oracle
from oracle import host


def pair_index(n, a, b):
    a, b = min(a, b), max(a, b)
    return n + a * n - a * (a + 1) // 2 + (b - a - 1)


def _bits(mask):
    return [k for k in range(32) if (mask >> k) & 1]


def _index_sums(cells):
    """mass_properties.cl:34-41 over the cells (k, 3) of a boolean grid: xx,xy,xz,x,yy,yz,y,zz,z,n (uint32 wrap)"""
    x, y, z = (cells[:, i].astype(np.int64) for i in range(3))
    s = (x * x, x * y, x * z, x, y * y, y * z, y, z * z, z)
    return [int(v.sum()) % 2 ** 32 for v in s] + [len(x) % 2 ** 32]


def _block_integrals(sums, shifted, s):
    """mass_properties.py:119-148, as oracle.host.mass_properties"""
    sxx, sxy, sxz, sx, syy, syz, sy, szz, sz, n = sums
    s2 = s * s
    s3 = s * s2
    bx, by, bz = shifted
    tx, ty, tz = s * sx, s * sy, s * sz
    txx, tyy, tzz = s2 * sxx, s2 * syy, s2 * szz
    txy, txz, tyz = s2 * sxy, s2 * sxz, s2 * syz
    return (s3 * n, s3 * (n * bx + tx), s3 * (n * by + ty), s3 * (n * bz + tz),
            s3 * (n * (bx * bx + s2 / 12) + 2 * bx * tx + txx), s3 * (n * (by * by + s2 / 12) + 2 * by * ty + tyy),
            s3 * (n * (bz * bz + s2 / 12) + 2 * bz * tz + tzz), s3 * (n * bx * by + bx * ty + by * tx + txy),
            s3 * (n * bx * bz + bx * tz + bz * tx + txz), s3 * (n * by * bz + by * tz + bz * ty + tyz))


def assembly_mass_properties(words_list, box_a, box_b, resolution, grid_size=64):
    """-> float64 integrals [sets][10] (one,x,y,z,xx,yy,zz,xy,xz,yz): the parts of words_list, then the pairs {a < b}
    at pair_index.  Blocks are visited in oracle.host.mass_properties' order, so a single part's integrals are that
    function's to the bit."""
    n = len(words_list)
    assert 1 <= n <= 32
    assert resolution > 0 and grid_size > 1 and grid_size ** 5 <= 2 ** 32
    sets = n + n * (n - 1) // 2
    bs = host.calculate_block_sizes(box_a, box_b, 3, resolution, grid_size, False)
    bs = [(resolution * cs, dims) for cs, dims in bs]
    acc = [[host._Kahan() for _ in range(10)] for _ in range(sets)]
    stack = [(tuple(float(c) for c in box_a), 0, (1 << n) - 1, 0)]
    while stack:
        corner, level, eval_mask, inside = stack.pop()
        s, dims = bs[level]
        shifted = tuple(c + s / 2 for c in corner)
        thr = np.float32(s * math.sqrt(3) / 2 if level < len(bs) - 1 else 0)
        c32 = np.array(shifted, np.float64).astype(np.float32)
        now = np.zeros(tuple(dims), np.uint32)
        near = np.zeros(tuple(dims), np.uint32)
        for k in _bits(eval_mask):
            d = oracle.grid_eval(words_list[k], c32, s, dims)[..., 3]
            ins = d <= -thr                       # mass_properties.cl:31 (NaN: outside)
            nr = ~ins & (d < thr)                 # :43
            now |= ins.astype(np.uint32) << np.uint32(k)
            near |= nr.astype(np.uint32) << np.uint32(k)
        member = now | np.uint32(inside)
        for k in _bits(eval_mask):  # (every block of the part's own hierarchy, as oracle.host adds them: zeros too)
            cells = np.argwhere((now >> np.uint32(k)) & 1)
            for a, v in zip(acc[k], _block_integrals(_index_sums(cells), shifted, s)):
                a.add(v)
        for a in range(n):
            for b in range(a + 1, n):
                if not ((eval_mask >> a) | (eval_mask >> b)) & 1:
                    continue  # (the blocks where a member of the pair is undecided, zeros too: [A, A] sums as A)
                bit_a, bit_b = np.uint32(a), np.uint32(b)
                cell = (((now >> bit_a) & 1) & ((member >> bit_b) & 1)) | (((now >> bit_b) & 1) & ((member >> bit_a) & 1))
                cells = np.argwhere(cell)
                for acc_i, v in zip(acc[pair_index(n, a, b)], _block_integrals(_index_sums(cells), shifted, s)):
                    acc_i.add(v)
        hits = np.argwhere(near != 0)              # INDEX3 order
        assert level + 1 < len(bs) or len(hits) == 0
        stack.extend(((i * s + corner[0], j * s + corner[1], k * s + corner[2]), level + 1, int(near[i, j, k]),
                      inside | int(now[i, j, k])) for i, j, k in hits.tolist())
    return np.array([[a.result for a in row] for row in acc])
