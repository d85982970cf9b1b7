"""Host restatements of the counter-based dropout RNG (rng64 / rng_keep in adapter4rec_b200/csrc/a4r_common.cuh) and of
the two counter layouts the kernels draw from it, so a test can rebuild the exact mask a kernel applied.

rng64(seed, counter) is the splitmix64 finaliser of counter * 0x9E3779B97F4A7C15 + seed: 64 bits = four 16-bit lanes, and
an element is kept iff its lane >= thr16 = round(p * 65536); kept values are scaled by 65536 / (65536 - thr16).

`rng64_np` is the plain uint64 statement.  `rng64` states the same thing in torch int64, so masks of hundreds of millions
of elements can be built on the GPU: the constants are written as signed int64, multiplication wraps, and a logical right
shift is an arithmetic shift with the sign-extended bits masked off."""
import numpy as np
import torch


def thr16(p):
    """the keep threshold the kernels derive from p (float32 arithmetic, as on the device)"""
    return int(np.float32(p) * np.float32(65536.0) + np.float32(0.5))


def keep_scale(p):
    """the scale of a kept element (float32, as on the device)"""
    return float(np.float32(65536.0) / np.float32(65536 - thr16(p)))


def rng64_np(seed, counter):
    """numpy uint64 statement of rng64(); counter: uint64 array"""
    with np.errstate(over="ignore"):
        z = counter.astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(seed)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def _i64(u):
    """the int64 with the bit pattern of the uint64 u"""
    u &= (1 << 64) - 1
    return u - (1 << 64) if u >= 1 << 63 else u


_C0, _C1, _C2 = _i64(0x9E3779B97F4A7C15), _i64(0xBF58476D1CE4E5B9), _i64(0x94D049BB133111EB)


def _lsr(z, k):
    return (z >> k) & ((1 << (64 - k)) - 1)


def rng64(seed, counter):
    """torch int64 statement of rng64(): the result's bit pattern equals rng64_np's; counter: int64 tensor (< 2^63)"""
    z = counter * _C0 + _i64(seed)
    z = (z ^ _lsr(z, 30)) * _C1
    z = (z ^ _lsr(z, 27)) * _C2
    return z ^ _lsr(z, 31)


def _keep(seed, counter, lane, p):
    return ((rng64(seed, counter) >> (16 * lane)) & 0xFFFF) >= thr16(p)


def element_keep(seed, offset, p, rows, N):
    """keep mask [len(rows), N] of rows `rows` (int64 tensor) of a logical [M, N] tensor in the element layout of
    a4r_dropout, the GEMM LINEAR epilogue and a4r_layernorm_bwd's dz_masked: element (r, c) uses lane (r*N + c) & 3 of
    counter offset + (r*N + c) / 4."""
    e = rows.to(torch.int64)[:, None] * N + torch.arange(N, dtype=torch.int64, device=rows.device)[None, :]
    return _keep(seed, offset + (e >> 2), e & 3, p)


def prob_keep(seed, offset, p, seqs, heads, L):
    """keep mask [len(seqs), heads, L, L] of the attention probabilities of sequences `seqs` (int64 tensor) in the layout
    of the short-sequence attention kernel (attention_small.cu): element (i, j) of (sequence n, head h), with nt = j / 8,
    t = (j % 8) / 2, e = j % 2, uses lane (nt & 1) * 2 + e of counter offset + ((n*heads + h) * 32 + i) * 8 + (nt >> 1) * 4 + t."""
    dev = seqs.device
    n = seqs.to(torch.int64).view(-1, 1, 1, 1)
    h = torch.arange(heads, dtype=torch.int64, device=dev).view(1, -1, 1, 1)
    i = torch.arange(L, dtype=torch.int64, device=dev).view(1, 1, -1, 1)
    j = torch.arange(L, dtype=torch.int64, device=dev).view(1, 1, 1, -1)
    nt = j // 8
    ctr = offset + ((n * heads + h) * 32 + i) * 8 + (nt >> 1) * 4 + (j % 8) // 2
    return _keep(seed, ctr, (nt & 1) * 2 + j % 2, p)
