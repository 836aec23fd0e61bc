"""Host model of the kernels' dropout masks (numpy uint32 arithmetic, vectorised).

A mask is a pure function of (seed, site, element index), csrc/common.cuh: `mix32`, `drop_bits64`, `make_drop`,
`drop_factor` / `drop_factor4`, and the attention pair hash (`pair_hash` in attention_bf16.cu, inlined in attention_tc.cu,
attention_tc_long_bwd.cu and attn_block_tc.cu).  The functions here rebuild the exact float32 factor (0 or 1/(1-p)) of any
launch, so a float64 reference can apply the very mask the kernel drew.

Element-indexed sites (`elem_mask`): the factor of flat element e is lane (e & 3) of quad e >> 2 -- word a for e & 2 == 0,
word b otherwise; the low 16 bits for even e, the high 16 bits for odd e.  Every element-indexed kernel uses e = row * ncols
+ col of its own output, ncols being the width of that output:
  - patch_embed.cu (emb-dropout, site 1): tokens [B*T, D], forward and backward;
  - gemm_f32.cu / gemm_bf16.cu epilogues: y [M, N] (the ragged tail N % 4 != 0 through `drop_factor`), and the act-2
    data-gradient epilogue (GELU'(aux) * mask) on dx [M, K] of the forward's [M, N] = its hidden output;
  - mlp_block_tc.cu: hidden [R, M] (site_hidden) and output [R, D] (site_out);
  - the attn_block_tc.cu tail: xmid [R, D] (site_out);
  - cast_rows (bf16_util.cu), the LayerNorm backward's fused cast (layernorm.cu) and msst_dropout_apply: flat [R, D].
No exception was found: all of them index row * ncols + col with the row of the residual-stream matrix.

`seed` is the descriptor's seed plus the device seed offset when one is set (`seed_dev`, CUDA-graph replays), mod 2^64.
"""
import numpy as np

_M32 = 0xFFFFFFFF


def mix32(x):
    """lowbias32 finaliser (common.cuh `mix32`) on a uint32 array."""
    x = np.asarray(x, dtype=np.uint32)
    with np.errstate(over="ignore"):
        x = x ^ (x >> np.uint32(16))
        x = x * np.uint32(0x7FEB352D)
        x = x ^ (x >> np.uint32(15))
        x = x * np.uint32(0x846CA68B)
        x = x ^ (x >> np.uint32(16))
    return x


def drop_bits64(seed, site, quad):
    """(a, b): the two 32-bit words of quad `quad` (uint64 array) of (seed, site) -- common.cuh `drop_bits64`."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    quad = np.asarray(quad, dtype=np.uint64)
    lo = (quad & np.uint64(_M32)).astype(np.uint32)
    hi = (quad >> np.uint64(32)).astype(np.uint32)
    with np.errstate(over="ignore"):
        x = (lo + np.uint32(seed >> 32)) * np.uint32(0x9E3779B1)
        x = x ^ (hi * np.uint32(0x85EBCA77)) ^ np.uint32(seed & _M32) ^ np.uint32((int(site) * 0xC2B2AE3D) & _M32)
        a = mix32(x)
        b = mix32(a + np.uint32(0x9E3779B9))
    return a, b


def drop_params(p):
    """(thresh, scale) of `make_drop` for a float32 p: thresh = floor(p * 2^32) clamped to [1, 2^32 - 1] (0: disabled),
    scale = 1/(1-p) in float32 (0 for p >= 1)."""
    p = np.float32(p)
    if not p > 0:
        return 0, np.float32(1.0)
    t = float(p) * 4294967296.0
    thresh = _M32 if t >= 4294967295.0 else int(t)
    thresh = max(thresh, 1)
    scale = np.float32(0.0) if p >= 1 else np.float32(1.0) / (np.float32(1.0) - p)
    return thresh, scale


def _factor(lanes16, p):
    thresh, scale = drop_params(p)
    if thresh == 0:
        return np.ones(lanes16.shape, dtype=np.float32)
    return np.where(lanes16 >= np.uint32(thresh >> 16), scale, np.float32(0.0)).astype(np.float32)


def elem_mask(p, seed, site, n):
    """float32 factors of elements 0..n-1 of an element-indexed site (any n, not only multiples of 4)."""
    e = np.arange(n, dtype=np.uint64)
    a, b = drop_bits64(seed, site, e >> np.uint64(2))
    w = np.where((e & np.uint64(2)) != 0, b, a)
    lane = np.where((e & np.uint64(1)) != 0, w >> np.uint32(16), w & np.uint32(0xFFFF))
    return _factor(lane, p)


def attn_mask_f32(p, seed, site, n_seq, N, inner, H):
    """[n_seq, H, N, N] factors of attention_f32.cu: element ((seq*H + h)*N + q)*N + k (inner does not enter)."""
    return elem_mask(p, seed, site, n_seq * H * N * N).reshape(n_seq, H, N, N)


def _slot_of(n_seq, N, inner):
    """(group, slot) of every (seq, pos) under the N <= 64 packing of attn_geom.cuh (`slot_to` inverted)."""
    G = 64 // N
    seq = np.arange(n_seq, dtype=np.int64)[:, None]
    pos = np.arange(N, dtype=np.int64)[None, :]
    if inner == 1:                      # sequence-major: group = G consecutive sequences, slot = j * N + pos
        group, slot = seq // G + 0 * pos, (seq % G) * N + pos
    else:                               # position-major: G sequences of one block of `inner`, slot = pos * G + j
        gpb = -(-inner // G)
        blk, s = seq // inner, seq % inner
        group, slot = blk * gpb + s // G + 0 * pos, pos * G + s % G
    return group, slot


def attn_mask_bf16(p, seed, site, n_seq, N, inner, H):
    """[n_seq, H, N, N] factors of the bf16 attention kernels (mma.sync, tcgen05, long forward / backward, fused block).
    One hash word (word a of `drop_bits64` at the pair index) decides two neighbouring key slots: the low 16 bits the even
    slot, the high 16 bits the odd one (`pair_factors`: f0 = low half for key column 2*tq, f1 = high half for 2*tq + 1).
      N <= 64: pair = (group*H + h)*2048 + qslot*32 + kslot/2     (slot packing of attn_geom.cuh)
      N  > 64: pair = ((((seq*H + h)*tiles + q/64)*tiles + k/64)*2048 + (q mod 64)*32 + (k mod 64)/2,  tiles = ceil(N/64)."""
    h = np.arange(H, dtype=np.int64)[None, :, None, None]
    if N <= 64:
        group, slot = _slot_of(n_seq, N, inner)
        qs = slot[:, None, :, None]
        ks = slot[:, None, None, :]
        idx = (group[:, None, :, None] * H + h) * 2048 + qs * 32 + ks // 2
        odd = ks % 2
    else:
        tiles = -(-N // 64)
        seq = np.arange(n_seq, dtype=np.int64)[:, None, None, None]
        q = np.arange(N, dtype=np.int64)[None, None, :, None]
        k = np.arange(N, dtype=np.int64)[None, None, None, :]
        idx = (((seq * H + h) * tiles + q // 64) * tiles + k // 64) * 2048 + (q % 64) * 32 + (k % 64) // 2
        odd = k % 2
    idx, odd = np.broadcast_arrays(idx, odd)
    a, _ = drop_bits64(seed, site, idx.astype(np.uint64))
    lane = np.where(odd != 0, a >> np.uint32(16), a & np.uint32(0xFFFF))
    return _factor(lane, p)
