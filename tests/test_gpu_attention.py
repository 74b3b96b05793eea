"""
Kernel-level parity of the attention kernels that MCTS rollouts depend on, through the C ABI test hooks:
  * decode_attn_kernel (decode.cu): split-KV single-query attention over the slot cache, the last-CTA merge and its
    self-resetting counters, the switch from the lender's slot to the row's own slot at share_len, grouped KV heads;
  * the shared-prefix ("cascade") pass of batched decode: flash_attn_kernel in partial mode over the prefix slot, merged by
    decode_attn_kernel with key_begin = prefix_len (the pairing engine.cu's decode_launches runs);
  * flash_attn_kernel prefill (attn_mma.cu) over a suffix with grouped KV heads and borrowed prefix rows (k2 / v2);
  * one model-level check at the product's configuration (v2-8b shapes, GQA 32/8, 32 rollouts borrowing a long prefix).

Reference: plain fp64 softmax attention (torch on the device) over the same bf16 K/V, built from each row's logical
sequence (keys [0, share_len) from the lender, the rest from the row's own rows, keys [0, pos]).

The inputs make a wrong key visible far above the tolerance:
  * every query of a head leans on a fixed +-1 direction of its KV head; every cache row the kernel must NOT read (rows of
    other slots, the borrower's own rows below share_len, rows past pos, k rows below split_row, k2 rows from split_row
    on) holds 4x that direction in K (score ~ +22) and 24 in V, so reading one moves the output by O(10);
  * keys at the boundaries a kernel can get wrong (pos, share_len - 1 and share_len, the first and last key of every
    split range, every 64-key tile edge, the last key of the ragged last prefix range) hold the direction itself
    (score ~ +5.7, e^5.7 ~ 300 times a background key) and a V of 8 on one distinct column, so dropping or duplicating
    any one of them moves that column by >= 0.05 (most by far more); random background keys keep the softmax non-degenerate.

Tolerances (from the arithmetic):
  * decode_attn_kernel alone: fp32 q, fp32 scores / softmax / accumulation over bf16 K/V -> rtol 1e-4,
    atol 1e-4 * max|V| (a few fp32 ulps of the largest term);
  * cascade and prefill flash: q and P are rounded to bf16 for the mma.sync products -> rtol 2e-2 / atol 2e-2, as in
    test_gpu_kernels.py.
"""
import ctypes as C
import math

import pytest
import torch

from conftest import engine_for, model_bundle

pytestmark = pytest.mark.gpu

D = 128
SCALE = 1.0 / math.sqrt(D)
PLANT_V = 8.0
POISON_K, POISON_V = 4.0, 24.0
DEV = "cuda"


def _lib():
    from detikzify_b200 import _lib as L
    return L.load_library()


def _p(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _nsplit_for(heads, B):
    """engine.cu nsplit_for: key ranges per (row, head) so that heads * B * nsplit covers 2 CTAs per SM."""
    return max(1, min(16, (2 * 148 + heads * B - 1) // (heads * B)))


def _cascade_tiles(prefix_len, nsplit):
    """engine.cu decode_launches: 64-key tiles per prefix CTA with nsplit capped at 4 for cascade steps."""
    ctiles = (prefix_len + 63) // 64
    return max(2, -(-ctiles // (16 - nsplit)))


def _split_edges(T, key_begin, nsplit):
    """First and last key of every non-empty key range of decode_attn_kernel (ranges rounded up to 8 keys)."""
    chunk = (T - key_begin + nsplit - 1) // nsplit
    chunk = (chunk + 7) & ~7
    edges = set()
    for s in range(nsplit):
        j0 = key_begin + s * chunk
        j1 = min(T, j0 + chunk)
        if j0 < j1:
            edges |= {j0, j1 - 1}
    return edges


def _tile_edges(lo, hi):
    return {j for j in range(lo, hi) if j % 64 in (0, 63)}


class Cache:
    """One layer of the engine's slot cache, [slot][K | V][kv_head][max_len][128] bf16, filled with poison; `fill` writes
    background and planted rows into a range of one slot."""

    def __init__(self, nslots, kv_heads, max_len, gen):
        self.kv_heads, self.max_len, self.gen = kv_heads, max_len, gen
        self.dirs = (torch.randint(0, 2, (kv_heads, D), generator=gen, device=DEV) * 2 - 1).float()
        self.kv = torch.empty(nslots, 2, kv_heads, max_len, D, device=DEV, dtype=torch.bfloat16)
        self.kv[:, 0] = (POISON_K * self.dirs)[None, :, None, :].to(torch.bfloat16)
        self.kv[:, 1] = POISON_V

    def fill(self, slot, lo, hi, planted):
        n = hi - lo
        if n <= 0:
            return
        k = 0.5 * torch.randn(self.kv_heads, n, D, generator=self.gen, device=DEV)
        v = 0.5 * torch.randn(self.kv_heads, n, D, generator=self.gen, device=DEV)
        idx = sorted(j for j in planted if lo <= j < hi)
        if idx:
            rows = torch.tensor(idx, device=DEV)
            k[:, rows - lo] = self.dirs[:, None, :]
            v[:, rows - lo] = 0.0
            v[:, rows - lo, (rows * 37) % D] = PLANT_V
        self.kv[slot, 0, :, lo:hi] = k.to(torch.bfloat16)
        self.kv[slot, 1, :, lo:hi] = v.to(torch.bfloat16)

    def logical(self, own, lender, share_len, T):
        """K, V [kv_heads, T, D] fp64 of a row: keys below share_len from the lender's slot, the others from its own."""
        k = torch.cat([self.kv[lender, 0, :, :share_len], self.kv[own, 0, :, share_len:T]], 1).double()
        v = torch.cat([self.kv[lender, 1, :, :share_len], self.kv[own, 1, :, share_len:T]], 1).double()
        return k, v


def _queries(rows, heads, dirs, gen):
    """fp32 [rows, heads, D]: each query leans on its KV head's direction (planted keys score ~ 5.7, background ~ N(0, 0.3^2))."""
    g = heads // dirs.shape[0]
    return 0.5 * dirs.repeat_interleave(g, 0)[None] + 0.3 * torch.randn(rows, heads, D, generator=gen, device=DEV)


def _attend(q, k, v):
    """fp64 softmax attention of q [heads, D] over k, v [kv_heads, T, D] (query head h reads KV head h // group)."""
    kvh = k.shape[0]
    qg = q.double().view(kvh, -1, D)
    s = torch.einsum("kgd,ktd->kgt", qg, k) * SCALE
    return torch.einsum("kgt,ktd->kgd", torch.softmax(s, -1), v).reshape(-1, D)


def _decode_call(cache, q, rows, heads, nsplit, counters, q16=None, prefix_slot=0, prefix_len=0, part_tiles=0):
    """rows: (own slot, lender slot, share_len, pos) per row. Returns (out fp32 [B, heads, D], out bf16)."""
    B = q.shape[0]
    i32 = lambda xs: torch.tensor(xs, device=DEV, dtype=torch.int32)
    slots, lenders, slens, pos = (i32([r[i] for r in rows]) for i in range(4))
    part_o = torch.full((B, heads, 16, D), float("nan"), device=DEV)
    part_ml = torch.full((B, heads, 16, 2), float("nan"), device=DEV)
    out = torch.full((B, heads * D), float("nan"), device=DEV)
    out16 = torch.full((B, heads * D), float("nan"), device=DEV, dtype=torch.bfloat16)
    rc = _lib().dtk_dbg_decode_attn(_p(q), _p(cache.kv), cache.kv.shape[0], _p(slots), _p(pos), _p(lenders), _p(slens), B,
                                    heads, cache.kv_heads, cache.max_len, nsplit, SCALE, _p(part_o), _p(part_ml),
                                    _p(counters), _p(out), _p(out16), _p(q16), prefix_slot, prefix_len, part_tiles,
                                    _stream())
    assert rc == 0
    torch.cuda.synchronize()
    assert int(counters.count_nonzero()) == 0, "merge counters must reset themselves"
    assert torch.equal(out16, out.to(torch.bfloat16))
    return out.view(B, heads, D), out16


# ---------------------------------------------------------------------------------------------------------- decode
T_LIST = [1, 7, 8, 9, 31, 32, 33, 243, 244, 300, 1025, 2048]
SHARE_LENS = [0, 16, 48, 240, 288]      # 243 and 300 rounded down to whole 16-position blocks, and shorter ones

DECODE_CASES = [
    # (heads, kv_heads, B, max_len, nsplit, t0): row b has T = T_LIST[(t0 + b) % 12] (capped at max_len) and borrows
    # SHARE_LENS[(t0 + b) % 5] positions from that length's lender when they fit below its pos
    (16, 16, 1, 2048, _nsplit_for(16, 1), 11),    # ds-1.3b, batch 1 at the full context: 16 ranges of 128 keys
    (32, 32, 1, 2048, _nsplit_for(32, 1), 9),     # ds-7b, T = 300
    (32, 8, 1, 2048, _nsplit_for(32, 1), 10),     # v2-8b, T = 1025: ragged last range
    (32, 8, 1, 2048, 16, 3),                      # T = 9 over 16 ranges: 14 empty ranges
    (4, 2, 1, 2048, 5, 0),                        # tiny-v2, T = 1
    (4, 2, 3, 2048, _nsplit_for(4, 3), 1),        # 16 ranges
    (16, 16, 3, 2048, _nsplit_for(16, 3), 6),     # 7 ranges
    (32, 32, 4, 2048, _nsplit_for(32, 4), 5),
    (32, 8, 4, 2048, _nsplit_for(32, 4), 7),
    (16, 16, 4, 2048, 9, 8),
    (32, 8, 4, 2048, 2, 2),
    (16, 16, 17, 2048, _nsplit_for(16, 17), 0),
    (32, 8, 17, 2048, 5, 4),
    (4, 2, 17, 2048, 16, 3),
    (32, 32, 32, 2048, _nsplit_for(32, 32), 2),
    (32, 8, 32, 2048, 3, 9),
    (16, 16, 64, 2048, _nsplit_for(16, 64), 5),
    (32, 8, 64, 2048, 4, 1),
    (32, 8, 6, 320, 3, 7),                        # short max_len: other slot and head strides
    (16, 16, 17, 272, 9, 0),
]


def _decode_setup(heads, kv_heads, B, max_len, nsplit, t0, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    lens = sorted({s for s in SHARE_LENS if s > 0})
    nslots = B + len(lens) + 1
    order = torch.randperm(nslots, generator=gen, device=DEV).tolist()   # own slots and lenders interleave in the buffer
    lender_of = {s: order[B + i] for i, s in enumerate(lens)}
    cache = Cache(nslots, kv_heads, max_len, gen)
    rows, planted = [], []
    for b in range(B):
        T = min(T_LIST[(t0 + b) % len(T_LIST)], max_len)
        sl = SHARE_LENS[(t0 + b) % len(SHARE_LENS)]
        sl = sl if sl < T else 0
        own = order[b]
        lender = lender_of[sl] if sl else own
        rows.append((own, lender, sl, T - 1))
        p = {T - 1} | _split_edges(T, 0, nsplit) | _tile_edges(0, T)
        if sl:
            p |= {sl - 1, sl}
        planted.append(p)
    for sl, lender in lender_of.items():   # a lender's rows are the prefix of all its borrowers
        borrowers = [planted[b] for b in range(B) if rows[b][2] == sl]
        if borrowers:
            cache.fill(lender, 0, sl, set().union(*borrowers))
    for b, (own, lender, sl, pos) in enumerate(rows):
        cache.fill(own, sl, pos + 1, planted[b])
    q = _queries(B, heads, cache.dirs, gen)
    return cache, q, rows


def _reference(cache, q, rows):
    ref, vmax = [], 0.0
    for b, (own, lender, sl, pos) in enumerate(rows):
        k, v = cache.logical(own, lender, sl, pos + 1)
        vmax = max(vmax, v.abs().max().item())
        ref.append(_attend(q[b], k, v))
    return torch.stack(ref), vmax


@pytest.mark.parametrize("heads,kv_heads,B,max_len,nsplit,t0", DECODE_CASES)
def test_decode_attention_split_kv_matches_fp64(heads, kv_heads, B, max_len, nsplit, t0):
    """decode_attn_kernel against fp64 attention over each row's logical sequence: ragged positions, empty and ragged key
    ranges, per-row lenders, grouped KV heads; the merge counters reset themselves and a second call through the same
    counters gives a bit-identical output (fixed merge order)."""
    cache, q, rows = _decode_setup(heads, kv_heads, B, max_len, nsplit, t0, seed=B * 1000 + heads * 10 + nsplit + t0)
    q2 = q.reshape(B, heads * D).contiguous()
    counters = torch.zeros(B * heads, device=DEV, dtype=torch.int32)
    out, _ = _decode_call(cache, q2, rows, heads, nsplit, counters)
    ref, vmax = _reference(cache, q, rows)
    torch.testing.assert_close(out.double(), ref, rtol=1e-4, atol=1e-4 * vmax)
    again, _ = _decode_call(cache, q2, rows, heads, nsplit, counters)
    assert torch.equal(again, out)


# --------------------------------------------------------------------------------------------------------- cascade
def _cascade_cases():
    """Prefix lengths of whole 16-position blocks (what seq_share lends), at the engine's own nsplit / part_tiles and at
    forced part_tiles that take csplit from 1 up to 16 - nsplit, most with a ragged last key range."""
    layouts = [(32, 32), (32, 8)]
    batches = [4, 6, 32, 64]
    cases = []
    for i, P in enumerate([64, 96, 128, 192, 240, 288, 1024, 2032]):
        heads, kv_heads = layouts[i % 2]
        B = batches[i % 4]
        ns = min(4, _nsplit_for(heads, B))
        tiles = (P + 63) // 64
        p_min = next(p for p in range(1, tiles + 1) if -(-tiles // p) <= 16 - ns)
        forced = {_cascade_tiles(P, ns), p_min, tiles, (p_min + tiles) // 2}
        max_len = 2048 if P > 1024 else P + 64
        cases += [(heads, kv_heads, B, P, ns, pt, max_len) for pt in sorted(forced)]
    # all 16 partial slots in use: more suffix ranges than the engine would pick next to one-tile prefix CTAs
    cases += [(32, 8, 6, 288, 11, 1, 352), (32, 32, 4, 2032, 5, 3, 2048), (16, 16, 64, 1024, 1, 2, 1088)]
    return cases


@pytest.mark.parametrize("heads,kv_heads,B,P,nsplit,part_tiles,max_len", _cascade_cases())
def test_cascade_prefix_pass_matches_fp64_and_per_row_kernel(heads, kv_heads, B, P, nsplit, part_tiles, max_len):
    """B rollouts borrow [0, P) from one slot: the tensor-core prefix pass writes partial slots [nsplit, nsplit + csplit)
    and decode_attn_kernel covers each row's 1..40-key suffix and merges all of them. Against fp64 attention and against
    the per-row kernel alone (prefix_len = 0) over the same logical sequence."""
    gen = torch.Generator(device=DEV).manual_seed(P * 7 + B + part_tiles * 1000 + nsplit)
    nslots = B + 1
    order = torch.randperm(nslots, generator=gen, device=DEV).tolist()
    prefix_slot = order[B]
    cache = Cache(nslots, kv_heads, max_len, gen)
    csplit = -(-((P + 63) // 64) // part_tiles)
    ranges = {min(P, c * part_tiles * 64) for c in range(csplit)} | {min(P, (c + 1) * part_tiles * 64) - 1 for c in range(csplit)}
    cache.fill(prefix_slot, 0, P, _tile_edges(0, P) | ranges | {P - 1})
    rows = []
    for b in range(B):
        pos = P + (b * 7) % min(40, max_len - P)
        rows.append((order[b], prefix_slot, P, pos))
        cache.fill(order[b], P, pos + 1, {P, pos} | _split_edges(pos + 1, P, nsplit) | _tile_edges(P, pos + 1))
    q = _queries(B, heads, cache.dirs, gen)
    q2 = q.reshape(B, heads * D).contiguous()
    q16 = q2.to(torch.bfloat16)
    counters = torch.zeros(B * heads, device=DEV, dtype=torch.int32)
    out, _ = _decode_call(cache, q2, rows, heads, nsplit, counters, q16, prefix_slot, P, part_tiles)
    ref, vmax = _reference(cache, q, rows)
    torch.testing.assert_close(out.double(), ref, rtol=2e-2, atol=2e-2)
    plain, _ = _decode_call(cache, q2, rows, heads, nsplit, counters)
    torch.testing.assert_close(plain.double(), ref, rtol=1e-4, atol=1e-4 * vmax)
    torch.testing.assert_close(out, plain, rtol=2e-2, atol=2e-2)
    again, _ = _decode_call(cache, q2, rows, heads, nsplit, counters, q16, prefix_slot, P, part_tiles)
    assert torch.equal(again, out)


def test_decode_hook_rejects_out_of_range_arguments():
    """The hook refuses, without launching, what would index outside its buffers."""
    gen = torch.Generator(device=DEV).manual_seed(5)
    heads, kv_heads, max_len = 4, 2, 256
    cache = Cache(3, kv_heads, max_len, gen)
    counters = torch.zeros(65 * heads, device=DEV, dtype=torch.int32)

    def call(B, rows, nsplit=2, prefix_len=0, part_tiles=0, prefix_slot=0):
        q = torch.zeros(B, heads * D, device=DEV)
        i32 = lambda xs: torch.tensor(xs, device=DEV, dtype=torch.int32)
        slots, lenders, slens, pos = (i32([r[i] for r in rows]) for i in range(4))
        part_o = torch.zeros(B, heads, 16, D, device=DEV)
        part_ml = torch.zeros(B, heads, 16, 2, device=DEV)
        out = torch.zeros(B, heads * D, device=DEV)
        return _lib().dtk_dbg_decode_attn(_p(q), _p(cache.kv), 3, _p(slots), _p(pos), _p(lenders), _p(slens), B, heads,
                                          kv_heads, max_len, nsplit, SCALE, _p(part_o), _p(part_ml), _p(counters), _p(out),
                                          None, _p(q.to(torch.bfloat16)), prefix_slot, prefix_len, part_tiles, _stream())
    ok = [(0, 1, 16, 200)]
    assert call(1, ok) == 0
    assert call(1, ok, nsplit=13, prefix_len=192, part_tiles=1) == 0   # 13 + 3 partial slots: all 16 in use
    assert call(65, ok * 65) == -1                              # more rows than one 64-row prefix tile
    assert call(1, [(3, 1, 16, 200)]) == -1                     # slot outside the buffer
    assert call(1, [(0, 7, 16, 200)]) == -1                     # lender outside the buffer
    assert call(1, [(0, 1, 16, max_len)]) == -1                 # position past max_len
    assert call(1, ok, nsplit=17) == -1
    assert call(1, ok, nsplit=14, prefix_len=192, part_tiles=1) == -1   # 14 + 3 partial slots > 16
    assert call(1, ok, prefix_len=208, part_tiles=4) == -1              # pos 200 inside the prefix
    assert call(1, ok, prefix_len=64, part_tiles=1, prefix_slot=3) == -1
    assert call(1, ok, prefix_len=64, part_tiles=0) == -1
    torch.cuda.synchronize()
    assert int(counters.count_nonzero()) == 0


# --------------------------------------------------------------------------------------------------------- prefill
FLASH_CASES = [
    # (B, heads, kv_heads, q_pos0, Tq, split_row): causal suffix prefill over a cache, Tk = q_pos0 + Tq
    (1, 16, 16, 243, 57, 240),    # ds-1.3b: prompt suffix after a borrowed image prefix (split_row below q_pos0)
    (1, 32, 8, 288, 40, 16),
    (2, 32, 8, 48, 200, 64),      # split_row above q_pos0, on a tile edge
    (1, 4, 2, 16, 100, 48),
    (1, 16, 16, 200, 100, 240),   # split_row above q_pos0, inside the query span
    (3, 4, 2, 64, 64, 64),
    (1, 32, 32, 240, 1, 48),      # one query row
    (1, 32, 8, 1000, 129, 240),
]


@pytest.mark.parametrize("B,heads,kv_heads,q_pos0,Tq,split_row", FLASH_CASES)
def test_prefill_flash_gqa_borrowed_prefix_matches_fp64(B, heads, kv_heads, q_pos0, Tq, split_row):
    """flash_attn_kernel prefill with grouped KV heads: key rows below split_row from k2 / v2 (a lender's slot), the others
    from k / v; causal over positions q_pos0 + i."""
    Tk = q_pos0 + Tq
    gen = torch.Generator(device=DEV).manual_seed(q_pos0 * 31 + Tq + split_row + heads)
    dirs = (torch.randint(0, 2, (kv_heads, D), generator=gen, device=DEV) * 2 - 1).float()
    planted = torch.tensor(sorted(_tile_edges(0, Tk) | {split_row - 1, split_row, Tk - 1} - {Tk}), device=DEV)
    k = 0.5 * torch.randn(B, Tk, kv_heads, D, generator=gen, device=DEV)
    v = 0.5 * torch.randn(B, Tk, kv_heads, D, generator=gen, device=DEV)
    k[:, planted] = dirs
    v[:, planted] = 0.0
    v[:, planted, :, (planted * 37) % D] = PLANT_V
    k, v = k.to(torch.bfloat16), v.to(torch.bfloat16)
    poison_k = (POISON_K * dirs).to(torch.bfloat16)
    k1, v1, k2, v2 = k.clone(), v.clone(), k.clone(), v.clone()
    k1[:, :split_row], v1[:, :split_row] = poison_k, POISON_V     # rows the kernel must take from k2 / v2
    k2[:, split_row:], v2[:, split_row:] = poison_k, POISON_V
    g = heads // kv_heads
    q = (0.5 * dirs.repeat_interleave(g, 0) + 0.3 * torch.randn(B, Tq, heads, D, generator=gen, device=DEV)).to(torch.bfloat16)
    o = torch.full((B, Tq, heads, D), float("nan"), device=DEV, dtype=torch.bfloat16)
    rc = _lib().dtk_dbg_flash_attn_ex(_p(q), _p(k1), _p(v1), _p(k2), _p(v2), _p(o), B, heads, kv_heads, Tq, Tk, D, 1, q_pos0,
                                      split_row, SCALE, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    qd = q.double().view(B, Tq, kv_heads, g, D)
    s = torch.einsum("bqkgd,btkd->bkgqt", qd, k.double()) * SCALE
    mask = torch.arange(Tk, device=DEV)[None, :] > (q_pos0 + torch.arange(Tq, device=DEV))[:, None]
    s = s.masked_fill(mask, float("-inf"))
    ref = torch.einsum("bkgqt,btkd->bqkgd", torch.softmax(s, -1), v.double()).reshape(B, Tq, heads, D)
    torch.testing.assert_close(o.double(), ref, rtol=2e-2, atol=2e-2)


def test_flash_hook_rejects_bad_arguments():
    x = torch.zeros(1, 64, 4, D, device=DEV, dtype=torch.bfloat16)
    f = _lib().dtk_dbg_flash_attn_ex
    assert f(_p(x), _p(x), _p(x), None, None, _p(x), 1, 4, 3, 64, 64, D, 1, 0, 0, SCALE, _stream()) == -1   # 4 % 3
    assert f(_p(x), _p(x), _p(x), None, None, _p(x), 1, 4, 4, 64, 64, D, 1, 0, 16, SCALE, _stream()) == -1  # no k2 / v2
    assert f(_p(x), _p(x), _p(x), _p(x), _p(x), _p(x), 1, 4, 4, 64, 64, D, 1, 0, 65, SCALE, _stream()) == -1
    assert f(_p(x), _p(x), _p(x), None, None, _p(x), 1, 4, 4, 64, 64, 64, 1, 0, 0, SCALE, _stream()) == -1


# ------------------------------------------------------------------------------------------------------ model level
def _tol(ref):   # test_gpu_ds7b.py: 8 % of the reference logits' RMS
    return max(3e-2, 0.08 * ref.float().pow(2).mean().sqrt().item())


def test_v2_8b_rollouts_borrowing_a_long_prefix():
    """32 rollouts of one figure borrow a 421-position prefix (image span + prompt; seq_share lends 416 positions, so the
    cascade pass runs 4 prefix CTAs over 7 key tiles with a ragged last range) at the v2-8b shapes (GQA 32/8, llama3 RoPE):
    cascade on and off agree, the first and last rows match the fp32 oracle, and one borrower decoded at batch 1 on the
    persistent kernel (the borrowed prefix under GQA, read per 16-position item) matches the per-op kernels."""
    from oracle.hf_oracle import synthetic_pixels
    name, R, cut = "v2-8b-2l", 32, 421
    cfg, sd, oracle = model_bundle(name)
    eng = engine_for(name, max_seqs=R + 1, max_batch=R)
    pix = synthetic_pixels(1, cfg.vision_config.image_size, 1000)
    img = eng.image_embeds(pix.cuda())[0]
    P = cfg.num_patches
    g = torch.Generator().manual_seed(8100)
    prefix = torch.cat([torch.full((P,), cfg.patch_token_id), torch.randint(0, 128000, (cut - P,), generator=g)]).long()
    sufs = [torch.randint(0, 128000, (1 + (i * 7) % 40,), generator=g) for i in range(R)]
    toks = torch.randint(0, 128000, (R,), generator=g)
    base = eng.seq_alloc()
    subs = [eng.seq_alloc() for _ in range(R)]
    try:
        eng.prefill(base, prefix.cuda(), 0, img, 0)
        lens = []
        for s_, suf in zip(subs, sufs):
            eng.seq_share(base, s_, cut)
            eng.prefill(s_, suf.cuda(), cut, None, 0)
            lens.append(cut + suf.numel())
        out = {}
        for cas in (1, 0):
            eng.set_option("cascade_attn", cas)
            out[cas] = eng.decode(subs, lens, toks.cuda()).clone()
        eng.set_option("cascade_attn", 1)
        one = {}
        for impl in (1, 0):
            eng.set_option("decode_impl", impl)
            if impl == 1:
                assert eng.get_option("decode_persistent") == 1
            one[impl] = eng.decode([subs[-1]], [lens[-1]], toks[-1:].cuda())[0].clone()
        torch.cuda.synchronize()
        ref0, _ = oracle.forward_logits(torch.cat([prefix, sufs[0], toks[:1]])[None], pix)
        refl, _ = oracle.forward_logits(torch.cat([prefix, sufs[-1], toks[-1:]])[None], pix)
        TOL = _tol(ref0)
        d_cas = (out[1] - out[0]).abs().max().item()
        d_one = (one[1] - one[0]).abs().max().item()
        print(f"cascade on/off max diff {d_cas:.3e}; batch-1 persistent/per-op max diff {d_one:.3e}; oracle tol {TOL:.3e}")
        assert d_cas < TOL
        assert (out[1][0].cpu() - ref0[0, -1]).abs().max().item() < TOL
        assert (out[1][-1].cpu() - refl[0, -1]).abs().max().item() < TOL
        assert (one[0].cpu() - refl[0, -1]).abs().max().item() < TOL
        assert d_one < 5e-3
    finally:
        eng.set_option("cascade_attn", 1)
        eng.set_option("decode_impl", 1)
        for s_ in subs:
            eng.seq_free(s_)
        eng.seq_free(base)
