"""Test helper: a numpy restatement of the closed loop's noise generator (mpcb_sim_set_noise, csrc/mpcb_philox.cuh).

``philox4x32_10`` is Philox4x32-10 with curand's round and key schedule, ``normal_pairs`` one call's two normals,
``sim_normals`` the twelve normals of a vehicle and step in the layout include/mpcb200.h states.  The device's recorded
disturbances are checked against these (test_gpu_sim_noise.py); they are themselves checked without a GPU against
Philox's known answers and against the g++ build of the device header."""
import numpy as np


def philox4x32_10(ctr, key):
    """Philox4x32-10 (curand's round and key schedule): ctr [..., 4], key [..., 2] uint32 -> [..., 4] uint32."""
    ctr, key = np.asarray(ctr, np.uint64), np.asarray(key, np.uint64)
    c = list(np.broadcast_arrays(*(ctr[..., i] for i in range(4)), key[..., 0], key[..., 1]))
    c, k0, k1 = c[:4], c[4], c[5]
    m32 = np.uint64(0xFFFFFFFF)
    for r in range(10):
        if r:
            k0 = (k0 + np.uint64(0x9E3779B9)) & m32
            k1 = (k1 + np.uint64(0xBB67AE85)) & m32
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & m32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & m32]
    return np.stack(c, axis=-1).astype(np.uint32)


def normal_pairs(seed, id, t, j):
    """Two standard normals of Philox call (seed, id, t, j): counter (t, id, j, 0), key (seed low, seed high), the two
    64-bit words as (0, 1) uniforms ((W >> 11) + 0.5) 2^-53, Box-Muller.  Broadcasts; returns [..., 2] and the words."""
    seed = np.asarray(seed, np.uint64)
    t, id, j = (np.asarray(a, np.uint64) for a in (t, id, j))
    t, id, j, seed = np.broadcast_arrays(t, id, j, seed)
    w = philox4x32_10(np.stack([t, id, j, np.zeros_like(t)], axis=-1),
                      np.stack([seed & np.uint64(0xFFFFFFFF), seed >> np.uint64(32)], axis=-1))
    W = w.astype(np.uint64)
    W1 = (W[..., 0] << np.uint64(32)) | W[..., 1]
    W2 = (W[..., 2] << np.uint64(32)) | W[..., 3]
    u1 = ((W1 >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53
    u2 = ((W2 >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53
    rho = np.sqrt(-2.0 * np.log(u1))
    return np.stack([rho * np.cos(2.0 * np.pi * u2), rho * np.sin(2.0 * np.pi * u2)], axis=-1), w


def sim_normals(seed, id, t):
    """The standard normals of vehicle id at step t under seed (mpcb_sim_set_noise): [..., 12] = measurement 5 (calls
    j = 0..2), actuation 2 (j = 3), process 5 (j = 4..6); component i of a channel is output i mod 2 of call base + i/2."""
    z = normal_pairs(seed, np.asarray(id)[..., None], np.asarray(t)[..., None], np.arange(7))[0]
    return np.concatenate([z[..., 0:3, :].reshape(*z.shape[:-2], 6)[..., :5], z[..., 3, :],
                           z[..., 4:7, :].reshape(*z.shape[:-2], 6)[..., :5]], axis=-1)
