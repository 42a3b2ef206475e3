"""CPU tests of oracle/pool_exact_ref.py, the integer oracle that pins the fp32 pooling kernels bit for bit on dyadic
inputs: it restates the fp64 oracle, its premise (any float32 summation order is exact below 2^24 units) holds for the
orders the kernels use and fails just past the limit, and a single misplaced term changes its result."""
import numpy as np
import pytest
import torch

from oracle import pool_exact_ref as px
from oracle import voxel_pool_ref as vp
from oracle.depth_softmax_ref import online_softmax_f32

f32 = np.float32


SMALL = [  # B, N, D, H, W, C, vn, coherent
    (2, 2, 17, 16, 5, 8, (12, 6, 1), True),
    (1, 3, 7, 17, 4, 4, (9, 5, 2), False),
    (2, 1, 33, 3, 3, 12, (4, 4, 1), True),
]


@pytest.mark.parametrize('case', SMALL)
def test_integer_reference_equals_fp64_oracle(case):
    B, N, D, H, W, C, vn, coherent = case
    geom = px.frustum_geom(1, B, N, D, H, W, vn, coherent)
    a, b, g = px.dyadic_inputs(2, B, N, D, H, W, C, vn)
    cell = px.cells(geom, vn)
    kept, lin, _ = vp.cell_index_ref(geom, vn)
    assert torch.equal(cell, torch.where(kept, lin, torch.tensor(-1)))
    depth, ctx, go = px.to_float(a), px.to_float(b), px.to_float(g)
    out, mag, terms = px.forward_exact(cell, a, b, vn)
    assert px.holds(mag)
    ref64 = vp.voxel_pooling_fused_ref(geom, depth, ctx, vn, acc_dtype=torch.float64)        # (B, C, Y, X)
    assert torch.equal(out.permute(0, 3, 1, 2).double() * 2.0 ** -8, ref64)
    abs64 = vp.voxel_pooling_fused_ref(geom, depth, ctx.abs(), vn, acc_dtype=torch.float64)
    assert torch.equal(mag.permute(0, 3, 1, 2).double() * 2.0 ** -8, abs64)
    assert torch.equal(terms.view(-1), torch.bincount(lin[kept], minlength=B * vn[0] * vn[1]))
    gd, gd_mag, gc, gc_mag = px.grads_exact(cell, a, b, g)
    rd, rc = vp.voxel_pooling_fused_grads_ref(geom, depth, ctx, vn, go)
    assert torch.equal(gd.double() * 2.0 ** -8, rd) and torch.equal(gc.double() * 2.0 ** -8, rc)
    assert bool((gd_mag >= gd.abs()).all()) and bool((gc_mag >= gc.abs()).all())
    # the drop-in op: arbitrary integer rows per point
    f = (a.view(B, N, D, H, W, 1) * b.view(B, N, C, H, W).permute(0, 1, 3, 4, 2).unsqueeze(2)).reshape(B, -1, C)
    dout, _ = px.dropin_forward_exact(cell, f, vn)
    assert torch.equal(dout, out)
    assert torch.equal(px.dropin_backward_exact(cell, g).double(),
                       vp.voxel_pooling_backward_ref(geom, g.double(), vn, (B, N * D * H * W, C)))


# ---------------------------------------------------------------- the premise: float32 is exact below 2^24 units
def _fma(x, y, acc):
    """fp32 fused multiply-add: the fp64 evaluation is exact for these dyadic operands, so one rounding to fp32."""
    return f32(np.float64(x) * np.float64(y) + np.float64(acc))


def _seq(rows):
    s = np.zeros(rows.shape[1], f32)
    for r in rows:
        s = (s + r).astype(f32)
    return s


def _pairwise(rows):
    if len(rows) == 0:
        return np.zeros(rows.shape[1], f32)
    if len(rows) == 1:
        return rows[0].astype(f32)
    m = len(rows) // 2
    return (_pairwise(rows[:m]) + _pairwise(rows[m:])).astype(f32)


def _cell_terms(cell, a, b, N, D, H, W):
    """Per output row: float32 (depth, context row) pairs of its terms in point order, and the run each belongs to
    (same image, bin, column and 16-row block, consecutive rows in one cell: the run plan's rule)."""
    BN, C = a.shape[0], b.shape[1]
    out = {}
    flat = cell.view(BN, D, H, W)
    for i in range(BN):
        for d in range(D):
            for w in range(W):
                prev = -1
                for h in range(H):
                    c = int(flat[i, d, h, w])
                    if c < 0:
                        prev = -1
                        continue
                    new_run = h % 16 == 0 or c != prev
                    lst = out.setdefault(c, [])
                    run = (lst[-1][2] + 1 if lst else 0) if new_run else lst[-1][2]
                    lst.append((f32(a[i, d, h, w] / 16.0), (b[i, :, h, w].numpy() / 16.0).astype(f32), run))
                    prev = c
    return out


def test_float32_orders_equal_the_integer_reference():
    B, N, D, H, W, C, vn = 2, 2, 19, 18, 5, 6, (5, 4, 1)
    geom = px.frustum_geom(3, B, N, D, H, W, vn, True)
    a, b, _ = px.dyadic_inputs(4, B, N, D, H, W, C, vn)
    cell = px.cells(geom, vn)
    out, mag, terms = px.forward_exact(cell, a, b, vn)
    assert px.holds(mag) and int(terms.max()) > 40
    want = px.to_float(out, 8).view(-1, C).numpy()
    rng = np.random.default_rng(5)
    for c, lst in _cell_terms(cell, a, b, N, D, H, W).items():
        prods = np.stack([(dv * row).astype(f32) for dv, row, _ in lst])
        # stage A / B: FMA run sums of <= 16 rows, then the runs of the cell in order
        runs = {}
        for dv, row, r in lst:
            acc = runs.get(r, np.zeros(C, f32))
            runs[r] = np.array([_fma(dv, x, y) for x, y in zip(row, acc)], f32)
        run_rows = np.stack([runs[r] for r in sorted(runs)])
        got = {'runs': _seq(run_rows), 'shuffled': _seq(prods[rng.permutation(len(prods))]), 'pairwise': _pairwise(prods)}
        # even share: the cell's runs cut into slices at random points, each summed, then the fix-up adds the slices
        cuts = np.sort(rng.choice(np.arange(1, len(run_rows) + 1), size=min(3, len(run_rows)), replace=False))
        parts = np.split(run_rows, cuts[:-1])
        got['slices'] = _seq(np.stack([_seq(p) for p in parts]))
        fma = np.zeros(C, f32)
        for dv, row, _ in lst:
            fma = np.array([_fma(dv, x, y) for x, y in zip(row, fma)], f32)
        got['fma'] = fma
        for name, v in got.items():
            assert np.array_equal(v, want[c]), (name, c)


def test_just_past_two_to_the_24_units_the_order_matters():
    t = np.array([[8388608], [8388609], [-1]], f32) * f32(2.0 ** -8)        # sum of |terms| = 2^24 + 2 units
    mag = torch.tensor([8388608 + 8388609 + 1])
    assert not px.holds(mag)
    exact = f32(16777216 * 2.0 ** -8)
    assert _seq(t)[0] != exact                                             # 2^24 + 1 units rounds away first
    assert _seq(t[[1, 2, 0]])[0] == exact
    assert px.holds(mag - 3)


# ---------------------------------------------------------------- sensitivity: one misplaced term changes the result
def _sens_case():
    B, N, D, H, W, C, vn = 1, 2, 18, 17, 5, 8, (6, 5, 1)
    geom = px.frustum_geom(7, B, N, D, H, W, vn, True)
    a, b, g = px.dyadic_inputs(8, B, N, D, H, W, C, vn)
    return geom, a, b, g, vn


def test_every_kind_of_misplaced_term_changes_the_integer_result():
    geom, a, b, g, vn = _sens_case()
    cell = px.cells(geom, vn)
    ref, _, _ = px.forward_exact(cell, a, b, vn)
    rgd, _, rgc, _ = px.grads_exact(cell, a, b, g)
    kept = (cell.view(-1) >= 0).nonzero().squeeze(1)
    p = int(kept[len(kept) // 2])
    fwd = lambda c=cell, aa=a, bb=b: px.forward_exact(c, aa, bb, vn)[0]

    dropped = cell.clone()
    dropped.view(-1)[p] = -1
    dup = a.clone()
    dup.view(-1)[p] *= 2                                                   # the term added twice
    moved = cell.clone()
    X = vn[0]
    moved.view(-1)[p] += 1 if int(cell.view(-1)[p]) % X < X - 1 else -1     # the neighbouring cell
    row_up = torch.cat([b[:, :, 1:], b[:, :, -1:]], 2)                      # row h + 1's context
    bin_up = torch.cat([a[:, 1:], a[:, -1:]], 1)                            # bin d + 1's depth
    swapped = ref[..., [1, 0] + list(range(2, ref.shape[-1]))]
    no_last_col = a.clone()
    no_last_col[..., -1] = 0                                               # W = 5: the ragged last column of a 4-wide tile
    mutants = {'drop': fwd(c=dropped), 'duplicate': fwd(aa=dup), 'neighbour cell': fwd(c=moved),
               'row h+1': fwd(bb=row_up), 'bin d+1': fwd(aa=bin_up), 'swap channels': swapped,
               'ragged column': fwd(aa=no_last_col)}
    for name, m in mutants.items():
        assert not torch.equal(m, ref), name
    # the gradients see the same mutations
    for name, (c, aa, bb) in {'drop': (dropped, a, b), 'neighbour cell': (moved, a, b), 'row h+1': (cell, a, row_up),
                              'bin d+1': (cell, bin_up, b), 'ragged column': (cell, no_last_col, b)}.items():
        gd, _, gc, _ = px.grads_exact(c, aa, bb, g)
        assert not (torch.equal(gd, rgd) and torch.equal(gc, rgc)), name


# ---------------------------------------------------------------- the softmax-folded route
def test_masked_logits_give_exact_reciprocals_and_an_exact_logit_gradient():
    logits, a = px.masked_logits(9, 3, 17, 5, 4)
    assert set(torch.unique((a > 0).sum(1)).tolist()) == {1, 2, 4, 8}
    p = online_softmax_f32(logits.permute(0, 2, 3, 1).reshape(-1, 17).numpy())
    want = px.to_float(a).permute(0, 2, 3, 1).reshape(-1, 17).numpy()
    assert np.array_equal(p, want)                                         # the kernels' loop: expf(0) * (1 / k)
    assert torch.equal(torch.softmax(logits, 1), px.to_float(a))
    gen = torch.Generator().manual_seed(10)
    gd = torch.randint(-3000, 3001, a.shape, generator=gen)                 # a gradient wrt p, units of 2^-8
    r, mag = px.logit_grad_exact(a, gd)
    assert px.holds(mag)
    pf, gf = px.to_float(a), px.to_float(gd, 8)
    dot = torch.zeros(3, 1, 5, 4)
    for d in range(17):                                                    # float32, the kernel's order
        dot = dot + pf[:, d:d + 1] * gf[:, d:d + 1]
    assert torch.equal(pf * (gf - dot), px.to_float(r, 16))
    p64, g64 = pf.double(), gf.double()
    assert torch.equal(p64 * (g64 - (p64 * g64).sum(1, keepdim=True)), r.double() * 2.0 ** -16)
