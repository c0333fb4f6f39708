"""GQA group 5 (Qwen3-14B: 40 q / 8 kv heads) in the attention kernels, the fused QKV-RoPE
epilogue at 40 / 8 heads and RMSNorm at d = 5120, called through the C-ABI.

The prefill q tile is 128 / 5 = 25 tokens: 125 of the tcgen05 kernel's 128 tile rows are real
(rows 125..127 are padding), and the paged kernel's second 16-token sub-tile ends inside the
tile.  Sequence lengths around 25 / 50 probe both edges; output rows outside every sequence are
pre-filled with a sentinel that must survive."""
import math

import pytest
import torch

import kv_layout as KV
import test_kernels_gpu as TK
from sutro_b200 import _lib as L

pytestmark = pytest.mark.gpu

DEV = TK.DEV
bf = TK.bf
SENTINEL = 7.0          # exact in bf16, far from any attention output of unit-scale inputs
GAP = 3                 # unused output rows between consecutive sequences
SCALE = 1.0 / math.sqrt(KV.HD)
SPECS = [(0, 1), (0, 16), (0, 17), (0, 100), (32, 5), (32, 70), (48, 200), (3, 33),
         (46, 111), (130, 140), (200, 300), (0, 129), (1, 128),
         (0, 24), (0, 25), (0, 26), (0, 50), (0, 51), (7, 25), (7, 51)]


def i32(x):
    return torch.tensor(x, dtype=torch.int32, device=DEV)


def layout(specs, qt):
    """q_start per sequence (GAP unused rows after each) and the (sequence, q tile) work list."""
    q_start, work, acc = [], [], 0
    for i, (_, q) in enumerate(specs):
        q_start.append(acc)
        acc += q + GAP
        work += [x for t0 in range(0, q, qt) for x in (i, t0)]
    return q_start, work, acc


def check_out(out, ref, specs, q_start, hq, tol=2e-2):
    """Every sequence row against the reference; every other row still holds the sentinel."""
    got = out.view(out.shape[0], hq, KV.HD).float()
    used = torch.zeros(out.shape[0], dtype=torch.bool, device=DEV)
    for i, (_, q) in enumerate(specs):
        lo = q_start[i]
        err = (got[lo:lo + q] - ref[i]).abs()
        assert torch.allclose(got[lo:lo + q], ref[i], rtol=tol, atol=tol), (i, specs[i], err.max())
        used[lo:lo + q] = True
    assert bool((out[~used].float() == SENTINEL).all()), "a row outside every sequence was written"


def dense_ref(qkv, pre, hq, hkv, specs, q_start):
    """fp32 softmax(QK^T)V per sequence over [prefix | own rows]: list of [q, hq, 128]."""
    out = []
    for i, (p, q) in enumerate(specs):
        out.append(TK._dense_ref(qkv[q_start[i]:q_start[i] + q], pre, 0, hq, hkv, [(p, q)], [0],
                                 SCALE))
    return out


# --------------------------------------------------------------------------- decode
@pytest.mark.parametrize("variant", [1, 2])   # 1: 4-warp split kernel, 2: warp-per-pair kernel
@pytest.mark.parametrize("hq,hkv", [(40, 8), (10, 2), (5, 1)])
def test_attn_decode_group5(hq, hkv, variant):
    TK.test_attn_decode(hq, hkv, variant)


# --------------------------------------------------------------------------- dense (tcgen05)
def _dense_case(hq, hkv, specs, seed, q_gain=1.0):
    torch.manual_seed(seed)
    qt = L.lib().sb200_attn_prefill_q_tile(hq, hkv)
    assert qt == 25
    q_start, items, rows = layout(specs, qt)
    ldq = (hq + 2 * hkv) * KV.HD
    qkv = bf(torch.randn(rows + 7, ldq, device=DEV))
    qkv[:, :hq * KV.HD] *= q_gain
    prefix_rows = max(max(p for p, _ in specs), 1)
    pre = bf(torch.randn(1, prefix_rows, 2 * hkv * KV.HD, device=DEV))
    return qkv, pre, prefix_rows, q_start, items


def _run_dense(qkv, pre, prefix_rows, hq, hkv, specs, q_start, items):
    out = torch.full((qkv.shape[0], hq * KV.HD), SENTINEL, dtype=torch.bfloat16, device=DEV)
    d_items, d_qs = i32(items), i32(q_start)
    d_ql, d_past = i32([q for _, q in specs]), i32([p for p, _ in specs])
    L.check(L.lib().sb200_attn_prefill_dense(
        L.ptr(qkv), qkv.shape[0], L.ptr(out), L.ptr(pre), prefix_rows, 1, 0, L.ptr(d_items),
        len(items) // 2, L.ptr(d_qs), L.ptr(d_ql), L.ptr(d_past), hq, hkv, SCALE, TK.stream()))
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("hq,hkv", [(40, 8), (10, 2)])
def test_attn_prefill_dense_tcgen05_group5(hq, hkv):
    qkv, pre, prefix_rows, q_start, items = _dense_case(hq, hkv, SPECS, seed=hq * 7 + hkv)
    out = _run_dense(qkv, pre, prefix_rows, hq, hkv, SPECS, q_start, items)
    check_out(out, dense_ref(qkv, pre, hq, hkv, SPECS, q_start), SPECS, q_start, hq)


@pytest.mark.parametrize("hq,hkv", [(40, 8), (10, 2)])
def test_attn_prefill_dense_group5_forced_rescale(hq, hkv):
    """Large scores force the lazy running-max rescale of the TMEM accumulator."""
    specs = [(0, 700), (0, 260), (0, 31), (0, 51)]
    qkv, pre, prefix_rows, q_start, items = _dense_case(hq, hkv, specs, seed=3, q_gain=6.0)
    out = _run_dense(qkv, pre, prefix_rows, hq, hkv, specs, q_start, items)
    check_out(out, dense_ref(qkv, pre, hq, hkv, specs, q_start), specs, q_start, hq, tol=3e-2)


@pytest.mark.parametrize("hq,hkv", [(40, 8), (10, 2)])
def test_attn_prefill_dense_group5_is_batch_invariant(hq, hkv):
    """A sequence's output bits do not depend on which other sequences share the launch (the
    padding rows' scores must not pick up what another item left in shared memory)."""
    qkv, pre, prefix_rows, q_start, items = _dense_case(hq, hkv, SPECS, seed=9)
    full = _run_dense(qkv, pre, prefix_rows, hq, hkv, SPECS, q_start, items)
    for i in (3, 9, 14, 17, 19):
        its = [x for t0 in range(0, SPECS[i][1], 25) for x in (0, t0)]
        alone = _run_dense(qkv, pre, prefix_rows, hq, hkv, [SPECS[i]], [q_start[i]], its)
        lo, hi = q_start[i], q_start[i] + SPECS[i][1]
        assert torch.equal(alone[lo:hi], full[lo:hi]), SPECS[i]


# --------------------------------------------------------------------------- paged (mma.sync)
def _paged_case(hq, hkv, specs, seed):
    torch.manual_seed(seed)
    ks = [bf(torch.randn(p + q, hkv, KV.HD, device=DEV)) for p, q in specs]
    vs = [bf(torch.randn(p + q, hkv, KV.HD, device=DEV)) for p, q in specs]
    pool, pt, max_pages = KV.build_cache(ks, vs, hkv, 400, DEV)
    qt = L.lib().sb200_attn_prefill_q_tile(hq, hkv)
    q_start, work, rows = layout(specs, qt)
    qkv = bf(torch.randn(rows, (hq + 2 * hkv) * KV.HD, device=DEV))
    return ks, vs, pool, pt, max_pages, qkv, q_start, work


def _run_paged(hq, hkv, specs, pool, pt, max_pages, qkv, q_start, work, slots):
    out = torch.full((qkv.shape[0], hq * KV.HD), SENTINEL, dtype=torch.bfloat16, device=DEV)
    d_work, d_slot, d_qs = i32(work), i32(slots), i32(q_start)
    d_ql, d_past = i32([q for _, q in specs]), i32([p for p, _ in specs])
    L.check(L.lib().sb200_attn_prefill(
        L.ptr(qkv), L.ptr(out), L.ptr(pool), L.ptr(pt), max_pages, L.ptr(d_work), len(work) // 2,
        L.ptr(d_slot), L.ptr(d_qs), L.ptr(d_ql), L.ptr(d_past), hq, hkv, SCALE, TK.stream()))
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("hq,hkv", [(40, 8), (10, 2)])
def test_attn_prefill_paged_group5(hq, hkv):
    ks, vs, pool, pt, max_pages, qkv, q_start, work = _paged_case(hq, hkv, SPECS, seed=hq + hkv)
    out = _run_paged(hq, hkv, SPECS, pool, pt, max_pages, qkv, q_start, work,
                     list(range(len(SPECS))))
    ref = []
    for i, (p, q) in enumerate(SPECS):
        rows = []
        for j in range(q):
            qv = qkv[q_start[i] + j].view(hq + 2 * hkv, KV.HD)[:hq]
            rows.append(TK.attn_ref(qv, ks[i][:p + j + 1], vs[i][:p + j + 1], SCALE))
        ref.append(torch.stack(rows))
    check_out(out, ref, SPECS, q_start, hq)
    # batch invariance: a sequence launched alone gives the same bits
    for i in (3, 14, 17, 19):
        its = [x for t0 in range(0, SPECS[i][1], 25) for x in (0, t0)]
        alone = _run_paged(hq, hkv, [SPECS[i]], pool, pt, max_pages, qkv, [q_start[i]], its, [i])
        lo, hi = q_start[i], q_start[i] + SPECS[i][1]
        assert torch.equal(alone[lo:hi], out[lo:hi]), SPECS[i]


@pytest.mark.parametrize("hq,hkv", [(40, 8), (10, 2)])
def test_attn_prefill_paged_group5_forced_rescale(hq, hkv):
    specs = [(0, 300), (0, 51), (20, 26)]
    ks, vs, pool, pt, max_pages, qkv, q_start, work = _paged_case(hq, hkv, specs, seed=5)
    qkv[:, :hq * KV.HD] *= 6.0
    out = _run_paged(hq, hkv, specs, pool, pt, max_pages, qkv, q_start, work,
                     list(range(len(specs))))
    ref = []
    for i, (p, q) in enumerate(specs):
        ref.append(torch.stack([
            TK.attn_ref(qkv[q_start[i] + j].view(hq + 2 * hkv, KV.HD)[:hq], ks[i][:p + j + 1],
                        vs[i][:p + j + 1], SCALE) for j in range(q)]))
    check_out(out, ref, specs, q_start, hq, tol=3e-2)


def test_unsupported_groups_are_refused_by_every_attention_kernel():
    lib = L.lib()
    z = torch.zeros(4096, dtype=torch.int32, device=DEV)
    for hq, hkv in ((24, 8), (48, 8), (56, 8), (128, 8)):       # groups 3, 6, 7, 16
        g = hq // hkv
        rc = lib.sb200_attn_decode(L.ptr(z), L.ptr(z), L.ptr(z), L.ptr(z), 1, L.ptr(z), L.ptr(z),
                                   1, hq, hkv, SCALE, TK.stream())
        assert rc != 0 and f"unsupported GQA group size {g}".encode() in lib.sb200_last_error()
        rc = lib.sb200_attn_prefill(L.ptr(z), L.ptr(z), L.ptr(z), L.ptr(z), 1, L.ptr(z), 1,
                                    L.ptr(z), L.ptr(z), L.ptr(z), L.ptr(z), hq, hkv, SCALE,
                                    TK.stream())
        assert rc != 0 and f"unsupported GQA group size {g}".encode() in lib.sb200_last_error()


# --------------------------------------------------------------------------- QKV epilogue, norm
@pytest.mark.parametrize("block_n", [128, 256, 512, 0])
def test_gemm_qkv_rope_fused_matches_unfused_40_8(block_n):
    """The fused QKV GEMM epilogue (q/k-norm, RoPE, paged K/V write) at Qwen3-14B's 40 / 8
    heads equals the plain GEMM followed by rope_kv_write."""
    torch.manual_seed(14)
    hq, hkv, T, K = 40, 8, 333, 320
    N = (hq + 2 * hkv) * KV.HD
    n_slots, max_pages, num_pages = 4, 12, 60
    a = bf(torch.randn(T, K, device=DEV))
    w = bf(torch.randn(N, K, device=DEV) / math.sqrt(K))
    qn = bf(torch.rand(KV.HD, device=DEV) + 0.5)
    kn = bf(torch.rand(KV.HD, device=DEV) + 0.5)
    cos, sin = TK.rope_tables(256)
    tok_slot = torch.arange(T, dtype=torch.int32) % n_slots
    tok_pos = (torch.arange(T, dtype=torch.int32) // n_slots) + 5
    pt = torch.randperm(num_pages)[: n_slots * max_pages].view(n_slots, max_pages).to(torch.int32)
    d_slot, d_pos, d_pt = tok_slot.to(DEV), tok_pos.to(DEV), pt.to(DEV)
    qkv_a = torch.zeros(T, N, dtype=torch.bfloat16, device=DEV)
    pool_a = torch.zeros(num_pages, hkv, 2, KV.PAGE, KV.HD, dtype=torch.bfloat16, device=DEV)
    L.check(L.lib().sb200_gemm_bf16_tn(L.ptr(a), T, L.ptr(w), L.ptr(qkv_a), 0, T, N, K, N, 0, 0,
                                       TK.stream()))
    L.check(L.lib().sb200_rope_kv_write(L.ptr(qkv_a), L.ptr(qn), L.ptr(kn), L.ptr(cos), L.ptr(sin),
                                        L.ptr(d_slot), L.ptr(d_pos), L.ptr(d_pt), max_pages,
                                        L.ptr(pool_a), T, hq, hkv, 1e-6, TK.stream()))
    qkv_b = torch.zeros(T, N, dtype=torch.bfloat16, device=DEV)
    pool_b = torch.zeros_like(pool_a)
    L.check(L.lib().sb200_gemm_qkv_rope(L.ptr(a), T, L.ptr(w), L.ptr(qkv_b), T, K, block_n,
                                        L.ptr(qn), L.ptr(kn), L.ptr(cos), L.ptr(sin),
                                        L.ptr(d_slot), L.ptr(d_pos), L.ptr(d_pt), max_pages,
                                        L.ptr(pool_b), hq, hkv, 1e-6, TK.stream()))
    torch.cuda.synchronize()
    qa, qb = qkv_a[:, :hq * KV.HD].float(), qkv_b[:, :hq * KV.HD].float()
    assert torch.allclose(qa, qb, rtol=2e-2, atol=2e-2)
    assert (qa != qb).float().mean().item() < 0.01
    assert torch.allclose(pool_a.float(), pool_b.float(), rtol=2e-2, atol=2e-2)
    assert (pool_a != pool_b).float().mean().item() < 0.01
    assert torch.equal(pool_a[:, :, 1], pool_b[:, :, 1])


@pytest.mark.parametrize("rows,d", [(1, 5120), (37, 5120), (513, 5120), (9, 4608)])
def test_rmsnorm_up_to_5120(rows, d):
    TK.test_rmsnorm(rows, d)
