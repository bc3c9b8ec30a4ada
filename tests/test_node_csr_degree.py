"""CPU model of the degree pass of the CSR node form (ncsr_row_degree): summing a row's stored entries in the windows, lanes
and trips of row_sum_window (k_degree over the dense block) gives the same float64 bits, whatever the node's offset in its
chunk, because every missing entry is a +0 and every affinity is >= 0."""
import numpy as np
import pytest


def warp_sum(acc):
    v = np.array(acc, dtype=np.float64)
    for o in (16, 8, 4, 2, 1):
        v = v + v[np.arange(32) ^ o]
    return v[0]


def row_sum_window(row, c_lo, c_hi):
    """kernels_graph.cuh row_sum_window on a dense float32 row (absolute columns)."""
    acc = [np.float64(0.0)] * 32
    a0 = c_lo & ~3
    for lane in range(32):
        c = a0 + lane * 4
        while c < c_hi:
            w = [np.float64(row[c + q]) if c + q < len(row) else np.float64(0.0) for q in range(4)]
            if c >= c_lo and c + 3 < c_hi:
                s = (w[0] + w[1]) + (w[2] + w[3])
            else:
                s = np.float64(0.0)
                for q in range(4):
                    if c_lo <= c + q < c_hi:
                        s = s + w[q]
            acc[lane] = acc[lane] + s
            c += 128
    return warp_sum(acc)


def degree_csr(cols, vals, pad, n):
    """ncsr_row_degree: ascending local columns, lane = window & 31, empty windows skipped."""
    acc = [np.float64(0.0)] * 32
    cur = [None] * 32
    xs = [[np.float32(0)] * 4 for _ in range(32)]

    def flush(lane):
        win = cur[lane]
        x = [np.float64(v) for v in xs[lane]]
        cl = 4 * win - pad
        if cl >= 0 and cl + 3 < n:
            s = (x[0] + x[1]) + (x[2] + x[3])
        else:
            s = np.float64(0.0)
            for v in x:
                s = s + v
        acc[lane] = acc[lane] + s

    for c, v in zip(cols, vals):
        q = c + pad
        win, lane = q >> 2, (q >> 2) & 31
        if cur[lane] != win:
            if cur[lane] is not None:
                flush(lane)
            cur[lane] = win
            xs[lane] = [np.float32(0)] * 4
        xs[lane][q & 3] = v
    for lane in range(32):
        if cur[lane] is not None:
            flush(lane)
    return warp_sum(acc)


@pytest.mark.parametrize("seed", range(6))
def test_csr_degree_matches_the_dense_window_sum(seed):
    rng = np.random.default_rng(seed)
    for _ in range(40):
        n = int(rng.integers(3, 700))
        ro = int(rng.integers(0, 64))
        ld = ((ro + n + 31) // 32) * 32 + 32
        row = np.zeros(ld, dtype=np.float32)
        i = int(rng.integers(0, n))
        dens = rng.choice([0.02, 0.1, 0.6, 1.0])
        mask = rng.random(n) < dens
        v = np.exp(-rng.uniform(0.0, 40.0, size=n)).astype(np.float32)
        v[rng.random(n) < 0.05] = np.float32(0)                   # exp underflow: a 0 in the block, no CSR entry
        block = np.where(mask, v, np.float32(0))
        block[i] = np.float32(1.0)
        row[ro:ro + n] = block
        row[max(0, ro - 4):ro] = np.float32(0)
        cols = np.nonzero(block)[0]
        want = row_sum_window(row, ro, ro + n)
        got = degree_csr(cols, block[cols], ro & 3, n)
        assert want.tobytes() == got.tobytes(), (seed, n, ro)
