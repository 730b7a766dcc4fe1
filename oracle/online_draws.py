"""Host restatement of the online path's random draws (k_draw_schedule and k_draw_world in csrc/r3d_resident.cu),
entry for entry, for the tests that compare the device draws with ``==``.

Every draw is integer arithmetic on Philox4x32-10 words, plus float32 steps with one rounding each, so numpy can
decide every entry.  The shuffle heads are rebuilt with the plain array Fisher-Yates shuffle, not with the kernel's
sparse (position, value) map, so the two implementations are independent.  Test infrastructure: imported by tests only.
"""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)
PHILOX_M = (np.uint64(0xD2511F53), np.uint64(0xCD9E8D57))
PHILOX_W = (np.uint64(0x9E3779B9), np.uint64(0xBB67AE85))
MAX_CLASSES = 16               # R3D_MAX_CLASSES: the event stride of the head stream ids
WORLD_STREAM = 0xFFFFFFFF


def _u64(v):
    return np.asarray(v, dtype=np.uint64) & M32


def philox4x32_10(ctr, key):
    """Philox4x32-10 of counters ``ctr`` = (c0, c1, c2, c3) and key (k0, k1); every entry an integer or an array of
    32-bit values (broadcast together).  Returns the four output words as uint64 arrays."""
    c0, c1, c2, c3 = np.broadcast_arrays(*(_u64(c) for c in ctr))
    k0, k1 = _u64(key[0]), _u64(key[1])
    for _ in range(10):
        p0, p1 = PHILOX_M[0] * c0, PHILOX_M[1] * c2                  # 32 x 32 -> 64 bits: exact in uint64
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & M32
        k0, k1 = (k0 + PHILOX_W[0]) & M32, (k1 + PHILOX_W[1]) & M32
    return c0, c1, c2, c3


def key_of(seed, epoch):
    """(seed low word, seed high word ^ epoch high word)"""
    seed, epoch = int(seed) & (2**64 - 1), int(epoch) & (2**64 - 1)
    return seed & 0xFFFFFFFF, (seed >> 32) ^ (epoch >> 32)


def bounded(x, r):
    """Lemire's bounded integer: (v in [0, r), accepted) for 32-bit words x (uint64 arrays or ints) and range r >= 1."""
    m = _u64(x) * np.uint64(r)
    low = m & M32
    return m >> np.uint64(32), (low >= np.uint64(r)) | (low >= np.uint64((2**32 - r) % r))


# ------------------------------------------------------------------------------------------------ class counts
def draw_counts(sidx, seed, epoch, n_classes, number_of_object):
    """Class counts of store scan ``sidx``: (int64 [n_classes], rejected words).  Round q calls Philox on (q * 32 +
    lane, 0, sidx, epoch low word) for lanes 0..31; the words are consumed word-major (word 0 of lanes 0..31, then
    word 1, ...), and every accepted word adds one to its class until number_of_object are taken."""
    key, elo = key_of(seed, epoch), int(epoch) & 0xFFFFFFFF
    counts = np.zeros(n_classes, dtype=np.int64)
    taken = rejected = 0
    rnd = 0
    while taken < number_of_object:
        words = philox4x32_10((np.arange(32) + rnd * 32, 0, sidx, elo), key)
        for w in words:
            if taken >= number_of_object:
                break
            v, ok = bounded(w, n_classes)
            rejected += int((~ok).sum())
            acc = v[ok][:number_of_object - taken].astype(np.int64)
            np.add.at(counts, acc, 1)
            taken += len(acc)
        rnd += 1
    return counts, rejected


def draw_counts_scalar(sidx, seed, epoch, n_classes, number_of_object):
    """draw_counts one word at a time, in the order the kernel comment states."""
    k0, k1 = key_of(seed, epoch)
    counts = [0] * n_classes
    taken = rejected = rnd = 0
    while taken < number_of_object:
        lanes = [[int(w) for w in philox4x32_10((rnd * 32 + lane, 0, sidx, int(epoch) & 0xFFFFFFFF), (k0, k1))]
                 for lane in range(32)]
        for word in range(4):
            if taken >= number_of_object:
                break
            for lane in range(32):
                m = lanes[lane][word] * n_classes
                low = m & 0xFFFFFFFF
                if not (low >= n_classes or low >= (2**32 - n_classes) % n_classes):
                    rejected += 1
                elif taken < number_of_object:
                    counts[m >> 32] += 1
                    taken += 1
        rnd += 1
    return np.array(counts, dtype=np.int64), rejected


# ------------------------------------------------------------------------------------------------ shuffle heads
def head_steps(sidx, seed, epoch, stream, n_c, k):
    """The Fisher-Yates targets r_j = j + uniform [0, n_c - j) of the heads on ``stream`` for j < k, vectorised over
    heads (sidx and stream broadcast together): (int64 [heads, k], rejected words per head int64 [heads]).  Step j
    calls Philox on (j | att << 16, stream, sidx, epoch low word) for att = 0, 1, ... and takes the first accepted of
    its four words."""
    key, elo = key_of(seed, epoch), int(epoch) & 0xFFFFFFFF
    sidx, stream = np.broadcast_arrays(_u64(sidx), _u64(stream))
    sidx, stream = sidx.ravel(), stream.ravel()
    r = np.zeros((len(sidx), k), dtype=np.int64)
    rejected = np.zeros(len(sidx), dtype=np.int64)
    for j in range(k):
        todo = np.arange(len(sidx))
        att = 0
        while len(todo):
            words = philox4x32_10(((j | att << 16), stream[todo], sidx[todo], elo), key)
            got = np.zeros(len(todo), dtype=bool)
            for w in words:
                v, ok = bounded(w, n_c - j)
                new = ok & ~got
                r[todo[new], j] = j + v[new].astype(np.int64)
                rejected[todo] += ~ok & ~got
                got |= ok
            todo = todo[~got]
            att += 1
    return r, rejected


def fisher_yates_heads(r, n_c, T, chunk=64):
    """Heads [heads, T]: perm[:k] of the array shuffle perm = arange(n_c), step j swapping perm[j] and perm[r_j],
    then -1 up to T."""
    h, k = r.shape
    out = np.full((h, T), -1, dtype=np.int32)
    for a in range(0, h, chunk):
        rr = r[a:a + chunk]
        rows = np.arange(len(rr))
        perm = np.tile(np.arange(n_c, dtype=np.int32), (len(rr), 1))
        for j in range(k):
            pj, pr = perm[rows, j].copy(), perm[rows, rr[:, j]]
            perm[rows, j] = pr
            perm[rows, rr[:, j]] = pj
        out[a:a + chunk, :k] = perm[:, :k]
    return out


def draw_heads(indices, seed, epoch, n_events, list_lens, T):
    """Heads of the scans ``indices`` (store indices): (int32 [n, n_events, classes, T], rejected words).  Head (ev, c)
    of a scan is on stream 1 + ev * 16 + c and holds min(T, n_c) entries."""
    idx = np.asarray(indices, dtype=np.int64)
    C = len(list_lens)
    out = np.full((len(idx), n_events, C, T), -1, dtype=np.int32)
    rejected = 0
    ev = np.arange(n_events)
    for c, n_c in enumerate(list_lens):
        k = min(T, int(n_c))
        if k == 0:
            continue
        sid = np.broadcast_to(idx[:, None], (len(idx), n_events))
        stream = np.broadcast_to(1 + ev[None, :] * MAX_CLASSES + c, (len(idx), n_events))
        r, rej = head_steps(sid, seed, epoch, stream, int(n_c), k)
        rejected += int(rej.sum())
        out[:, :, c, :] = fisher_yates_heads(r, int(n_c), T).reshape(len(idx), n_events, T)
    return out, rejected


def draw_head_scalar(sidx, seed, epoch, ev, c, n_c, T):
    """One head, one word at a time, as the kernel comment states: (int32 [T], rejected words)."""
    k0, k1 = key_of(seed, epoch)
    stream = 1 + ev * MAX_CLASSES + c
    k = min(T, n_c)
    perm = list(range(n_c))
    rejected = 0
    for j in range(k):
        rng = n_c - j
        v = None
        att = 0
        while v is None:
            words = philox4x32_10(((j | att << 16), stream, sidx, int(epoch) & 0xFFFFFFFF), (k0, k1))
            for w in words:
                m = int(w) * rng
                low = m & 0xFFFFFFFF
                if low >= rng or low >= (2**32 - rng) % rng:
                    v = m >> 32
                    break
                rejected += 1
            att += 1
        perm[j], perm[j + v] = perm[j + v], perm[j]
    return np.array(perm[:k] + [-1] * (T - k), dtype=np.int32), rejected


def draw_schedule(indices, seed, epoch, n_events, list_lens, T, random=True, number_of_object=0, fixed=None):
    """(counts int64 [n, classes], heads int32 [n, n_events, classes, T], rejected words) of a load_resident batch."""
    C = len(list_lens)
    rejected = 0
    if random:
        counts = np.zeros((len(indices), C), dtype=np.int64)
        for b, i in enumerate(indices):
            counts[b], rej = draw_counts(i, seed, epoch, C, number_of_object)
            rejected += rej
    else:
        counts = np.tile(np.asarray(fixed, dtype=np.int64), (len(indices), 1))
    heads, rej = draw_heads(indices, seed, epoch, n_events, list_lens, T)
    return counts, heads, rejected + rej


# ------------------------------------------------------------------------------------------------ world draw
def uniform24(w):
    return (np.asarray(w) >> np.uint64(8)).astype(np.float32) * np.float32(2.0**-24)


def draw_world(indices, seed, epoch, flip_x_prob, flip_y_prob, rot_max, scale_lo, scale_hi):
    """(fx, fy, theta, k) float32 arrays [n] of the scans ``indices``: one Philox call on (0, 0xFFFFFFFF, sidx, epoch
    low word); every float32 step rounds once, as the kernel's __fmul_rn / __fsub_rn / __fadd_rn do."""
    f32 = np.float32
    x = philox4x32_10((0, WORLD_STREAM, np.asarray(indices, dtype=np.int64), int(epoch) & 0xFFFFFFFF), key_of(seed, epoch))
    u = [uniform24(w) for w in x]
    fx = (u[0] < f32(flip_x_prob)).astype(np.float32)
    fy = (u[1] < f32(flip_y_prob)).astype(np.float32)
    theta = f32(rot_max) * ((f32(2.0) * u[2]).astype(np.float32) - f32(1.0)).astype(np.float32)
    k = f32(scale_lo) + ((f32(scale_hi) - f32(scale_lo)) * u[3]).astype(np.float32)
    return fx, fy, theta.astype(np.float32), k.astype(np.float32)


# ------------------------------------------------------------------------------------------------ world transform
def world_points(w, xyz):
    """A scan's world parameters ``w`` (fx, fy, theta, c, s, k, ...) on points in float32: flip, rotate, scale (numpy
    rounds every float32 operation)."""
    fx, fy, _, c, s, k = (np.float32(v) for v in w[:6])
    x, y, z = (np.asarray(xyz[:, i], dtype=np.float32) for i in range(3))
    x1 = -x if fy else x
    y1 = -y if fx else y
    return np.stack([(c * x1 - s * y1) * k, (s * x1 + c * y1) * k, z * k], axis=1)


def world_boxes(w, b7):
    """Target boxes (x, y, z, dx, dy, dz, heading) through the same transform; the heading in float64, wrapped."""
    from pcl_augmentation_b200 import boxes as bx
    out = np.array(b7, dtype=np.float32, copy=True)
    out[:, :3] = world_points(w, out[:, :3])
    out[:, 3:6] *= np.float32(w[5])
    h = out[:, 6].astype(np.float64)
    if w[0]:
        h = -h
    if w[1]:
        h = -(h + np.pi)
    out[:, 6] = bx.wrap_pi(h + np.float64(np.float32(w[2]))).astype(np.float32)
    return out
