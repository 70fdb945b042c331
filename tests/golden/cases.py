"""Case lists shared by make_golden.py (which runs the reference) and the tests (which run
the oracle / the CUDA path on the same seeded inputs)."""
import numpy as np

# (B, T, seed, realistic)
GEN_CASES = [(1, 1, 0, False), (2, 7, 1, False), (1, 32, 0, False), (2, 33, 2, False), (1, 16, 3, True)]
# (B, L, seed)
MSD_CASES = [(2, 8192, 0), (1, 1031, 1)]

CONV_CASES = [  # (Cin, Cout, K, stride, pad, dil, groups, L)
    (3, 5, 3, 1, 1, 1, 1, 17), (4, 4, 3, 1, 9, 9, 1, 11), (8, 16, 41, 4, 20, 1, 4, 103),
    (1, 16, 15, 1, 7, 1, 1, 33), (6, 2, 7, 1, 3, 1, 1, 1), (16, 16, 41, 1, 20, 1, 4, 5),
]
CONVT_CASES = [(6, 4, 16, 8, 4, 5), (5, 3, 4, 2, 1, 9), (4, 2, 16, 8, 4, 1)]  # Cin,Cout,K,s,p,L
POOL_CASES = [(4, 2, 2, 8192), (4, 4, 2, 4097), (4, 2, 2, 7), (4, 4, 2, 5)]  # k,s,p,L


def gen_key(B, T, seed, realistic):
    return "gen_B%d_T%d_s%d_r%d" % (B, T, seed, int(realistic))


CONFIG2_SAMPLES = 1024  # of each item's 8192 output samples kept in config2_outputs.npz (keeps the file under 1 MB)
CONFIG2_BLOCK = 64      # samples per float64 block sum; the block sums cover every sample


def config2_sample_index():
    return np.sort(np.random.RandomState(8192).choice(8192, CONFIG2_SAMPLES, replace=False))


def config2_digest(y, index):
    """What config2_outputs.npz keeps of a [B, 1, 8192] generator output: the samples at `index` (the same positions in
    every item) and the float64 sums of every block of CONFIG2_BLOCK consecutive samples."""
    y = np.asarray(y).reshape(len(y), -1)
    return y[:, index], y.astype(np.float64).reshape(len(y), -1, CONFIG2_BLOCK).sum(axis=2)


def op_inputs():
    """Yields (key, kind, params, x, w, b) in a fixed draw order from RandomState(99)."""
    rs = np.random.RandomState(99)
    for n, (cin, cout, k, s, p, d, g, L) in enumerate(CONV_CASES):
        x = rs.standard_normal((2, cin, L)).astype(np.float32)
        w = rs.standard_normal((cout, cin // g, k)).astype(np.float32)
        b = rs.standard_normal((cout,)).astype(np.float32)
        yield "op_conv_%d" % n, "conv", (s, p, d, g), x, w, b
    for n, (cin, cout, k, s, p, L) in enumerate(CONVT_CASES):
        x = rs.standard_normal((2, cin, L)).astype(np.float32)
        w = rs.standard_normal((cin, cout, k)).astype(np.float32)
        b = rs.standard_normal((cout,)).astype(np.float32)
        yield "op_convT_%d" % n, "convT", (s, p), x, w, b
    for n, (k, s, p, L) in enumerate(POOL_CASES):
        x = rs.standard_normal((2, 1, L)).astype(np.float32)
        yield "op_pool_%d" % n, "pool", (k, s, p), x, None, None
