"""NumPy twin of the minibatch stream of include/mfgp.h ("Minibatch stream"), which minibatch_gather_kernel evaluates on the
GPU.  The rule, stated once here:

    position p -> epoch e = p // N, offset i = p % N, row = pi_{seed,e}(i)
    pi_{seed,e}: 8-round balanced Feistel network on 2k-bit values (k smallest with 4**k >= N), cycle-walked below N;
                 round j: (l, r) <- (r, l ^ (mix32(r ^ key_j) & (2**k - 1)))
    key_j      = low 32 bits of splitmix64(splitmix64(splitmix64(seed) ^ e) ^ j)

All arithmetic is on uint64 / uint32 arrays, so it wraps exactly as the C code does."""
import numpy as np

ROUNDS = 8
_M64 = (1 << 64) - 1


def splitmix64(z):
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = z + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def mix32(x):
    x = np.asarray(x, dtype=np.uint32)
    with np.errstate(over="ignore"):
        x = x ^ (x >> np.uint32(16))
        x = x * np.uint32(0x7FEB352D)
        x = x ^ (x >> np.uint32(15))
        x = x * np.uint32(0x846CA68B)
    return x ^ (x >> np.uint32(16))


def half_bits(N):
    k = 0
    while 4**k < N:
        k += 1
    return k


def round_keys(seed, e):
    """[..., ROUNDS] uint32 keys for epoch(s) e."""
    se = splitmix64(splitmix64(np.uint64(seed & _M64)) ^ np.asarray(e, dtype=np.uint64))
    return np.stack([splitmix64(se ^ np.uint64(j)).astype(np.uint32) for j in range(ROUNDS)], axis=-1)


def permute(i, N, seed, e):
    """pi_{seed,e}(i) for an array of offsets i in [0, N) (e a scalar or an array like i)."""
    i = np.asarray(i, dtype=np.uint64)
    k = half_bits(N)
    mask = np.uint32((1 << k) - 1)
    keys = np.broadcast_to(round_keys(seed, e), i.shape + (ROUNDS,))
    x = i.copy()
    todo = np.ones(i.shape, dtype=bool)  # every offset takes at least one pass of the network
    while todo.any():
        xs, ks = x[todo], keys[todo]
        l = (xs >> np.uint64(k)).astype(np.uint32)
        r = (xs & np.uint64(mask)).astype(np.uint32)
        for j in range(ROUNDS):
            l, r = r, l ^ (mix32(r ^ ks[:, j]) & mask)
        x[todo] = (l.astype(np.uint64) << np.uint64(k)) | r.astype(np.uint64)
        todo = x >= np.uint64(N)
    return x.astype(np.int64)


def rows(positions, N, seed):
    """Rows of stream positions (int64 array)."""
    p = np.asarray(positions, dtype=np.int64)
    return permute(p % N, N, seed, (p // N).astype(np.uint64))


def batch_rows(N, seed, pos0, step, B, lo=0, count=None):
    """Rows of positions pos0 + step * B + lo + j, j < count (default B - lo): what mfgp_minibatch_gather returns."""
    count = B - lo if count is None else count
    return rows(pos0 + step * B + lo + np.arange(count, dtype=np.int64), N, seed)
