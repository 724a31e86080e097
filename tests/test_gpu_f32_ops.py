"""Every fp32 C-ABI operator against the fp64 oracle, at the widths, sizes and edges where the kernels could go wrong.

The fp32 operators are the default precision, the only one for models wider than 64 channels and the on-device oracle of
the 16-bit gradient tests, so each is pinned here to a float64 CPU restatement (oracle/fgnn_oracle.py, gradients by
torch.autograd) rather than to the whole-model goldens alone.  The library is called directly through its C ABI so the
test owns every buffer:
  - every output is filled with NaN before the call, so a skipped tile, row or column fails instead of leaving zeros;
  - accumulated parameter-gradient buffers are seeded with a power of two near the gradient's own scale, subtracted
    afterwards (the header's += contract);
  - ragged cases run a second time with the padded input entries set to 1e3: every output must be bitwise equal (the
    parameter gradients too in deterministic mode; the default mode sums them with atomics in any order);
  - padded output entries must be exact zeros.
Ragged references follow the reference's own idiom: each graph's n_g x n_g slice runs alone, with GraphNorm's n = n_g
(constant_n = 0) or the padded N (constant_n = 1).

Tolerances are relative Frobenius errors (parameter gradients: against the magnitude of their summands, see mlp_errors),
about 1.5x the worst measured on one B200 at its 1000 W power limit, each measured number written beside its bar below;
all sit under the ceilings forward 1e-5, matmul / scores / cross-entropy / Adam 1e-5 and MLP gradients 1e-4.  Integer
outputs, arg-max, max-pool values and padding are exact.  The whole file runs in about 12 s on a B200."""
import math

import numpy as np
import pytest
import torch

import graph_neural_net_b200 as pkg
from graph_neural_net_b200 import _lib as L
from graph_neural_net_b200 import _ops
from graph_neural_net_b200.maskedtensors import maskedtensor as mt
from oracle import fgnn_oracle as O
from tests.helpers import rel_fro

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
EPS = 1e-5
DET = L.FGNN_DETERMINISTIC
PAD = 1e3                      # what the padded input entries hold in the second run of a ragged case

# bars: about 1.5x the worst measured on one B200 (1000 W power limit), see each test's docstring
TOL_MLP_FWD = 1.3e-6      # measured 8.8e-7
TOL_MLP_GRAD = 8e-7       # measured 4.8e-7 (against the summands' magnitude; dx in relative Frobenius norm)
TOL_WIDE_FWD = 2.8e-6     # measured 1.9e-6
TOL_WIDE_GRAD = 7.2e-5    # measured 4.8e-5 (the oracle itself in fp32: 4.8e-5)
TOL_PLANES = 1.4e-6       # measured 8.9e-7
TOL_FUSED = 5.6e-7        # measured 3.7e-7
TOL_GN = 8.5e-8           # measured 5.4e-8
TOL_MM = 4.7e-7           # measured 3.1e-7
TOL_SCORES = 3.5e-7       # measured 2.3e-7
TOL_CE = 2e-6             # measured 1.3e-6
TOL_ADAM = 2.6e-6         # measured 1.7e-6


def lib():
    return pkg.get_lib()


def stream():
    return L.stream_ptr(torch.device(DEV))


def nan(shape):
    return torch.full(shape, float("nan"), device=DEV)


def scratch(nbytes):
    """Workspace whose every float reads as NaN: a kernel that consumes scratch it did not write shows it."""
    return torch.full((max(int(nbytes), 1),), 0xFF, dtype=torch.uint8, device=DEV)


def i32(sizes):
    return None if sizes is None else torch.tensor(sizes, dtype=torch.int32, device=DEV)


def outside(G, N1, N2, n1, n2):
    """bool (G,N1,N2): True outside each graph's n1[g] x n2[g] block (all False when the sizes are None)."""
    if n1 is None and n2 is None:
        return torch.zeros((G, N1, N2), dtype=torch.bool)
    n1 = torch.tensor(n1 if n1 is not None else [N1] * G)[:, None, None]
    n2 = torch.tensor(n2 if n2 is not None else [N2] * G)[:, None, None]
    return (torch.arange(N1)[None, :, None] >= n1) | (torch.arange(N2)[None, None, :] >= n2)


def planes_outside(G, N, sizes):
    """bool (G,1,N,N) padding mask of (G,C,N,N) planes."""
    return outside(G, N, N, sizes, sizes)[:, None]


def vec_outside(G, N, sizes):
    """bool (G,1,N) padding mask of (G,C,N) node vectors."""
    if sizes is None:
        return torch.zeros((G, 1, N), dtype=torch.bool)
    return (torch.arange(N)[None, :] >= torch.tensor(sizes)[:, None])[:, None]


def filled(t, mask, value):
    """Copy of the CPU tensor t with the masked (padded) entries set to value."""
    return torch.where(mask, torch.full_like(t, value), t)


def seed_of(ref):
    """A power of two near the rms of the reference gradient: the accumulator's known starting value."""
    rms = float(ref.double().pow(2).mean().sqrt())
    return 2.0 ** round(math.log2(rms)) if rms > 0 else 1.0


def assert_zero(t, mask, what):
    m = mask.expand_as(t)
    assert bool((t[m] == 0).all()), f"{what}: padded entries are not exact zeros"


def ok(status, what):
    L.check(status, what)


# --------------------------------------------------------------------------------------------------------------------
# fgnn_mlp_fwd_f32 / fgnn_mlp_bwd_f32_ex
# --------------------------------------------------------------------------------------------------------------------
MLP_CASES = [
    # (c_in, c_out, depth, N): 11^2 and 12^2 pixels sit on either side of the 128-pixel CTA, 64^2 is a whole number of
    # 64-pixel wgrad chunks and 100^2 is not; the wide cases go with small N to keep the fp64 reference cheap
    *[(1, 1, 1, n) for n in (1, 11, 12, 64, 100)],
    *[(2, 5, 2, n) for n in (1, 11, 12, 64, 100)],
    *[(7, 9, 3, n) for n in (11, 12, 64, 100)],
    *[(33, 127, 8, n) for n in (1, 11, 12)],
    *[(64, 64, 3, n) for n in (11, 12, 64)],
    *[(128, 128, 2, n) for n in (1, 12, 64)],
    *[(130, 64, 2, n) for n in (11, 12, 64)],
    *[(256, 128, 3, n) for n in (11, 12)],
    *[(512, 128, 1, n) for n in (1, 12, 64)],
]


def ragged_sizes(N):
    """n_g in {N, 1, an inner value}."""
    inner = {1: 1, 11: 6, 12: 11, 64: 33, 100: 65}.get(N, max(1, N // 2))
    return [N, 1, inner]


def mlp_params(c_in, c_out, depth, gen):
    """Conv weights / biases and GraphNorm affine (float64, CPU); output channel c_out // 2 of the last conv has zero
    weights, so its pre-norm plane is the constant bias (variance 0)."""
    ws, bs, fin = [], [], c_in
    for _ in range(depth):
        bound = math.sqrt(6.0 / (fin + c_out))
        ws.append(((torch.rand((c_out, fin), generator=gen) * 2 - 1) * bound).double())
        bs.append(((torch.rand(c_out, generator=gen) - 0.5) * 0.2).double())
        fin = c_out
    ws[-1][c_out // 2] = 0
    gw = (1.0 + (torch.rand(c_out, generator=gen) - 0.5)).double()
    gb = ((torch.rand(c_out, generator=gen) - 0.5) * 0.5).double()
    return ws, bs, gw, gb


def plane_stats(z, n_norm):
    """{mean, 1/(2 sqrt(n (var + eps)))} of (1,C,n,n) pre-norm planes."""
    mu = z.mean(dim=(-1, -2))
    var = ((z - mu[..., None, None]) ** 2).mean(dim=(-1, -2))
    return torch.stack([mu, 1.0 / (2.0 * torch.sqrt(n_norm * (var + EPS)))], -1)


def ref_mlp(x, dy, params, sizes, constant_n):
    """fp64 oracle per graph slice (O.mlp_block's conv1x1 / relu / graph_norm chain, each layer's output kept): y,
    stats, dx and the parameter gradients of sum(y * dy), and for every parameter gradient the magnitude of its summands
    (sum over pixels of |d out| |in| for a weight, |d out| for a bias, |dy normalize(z)| and |dy| for the GraphNorm
    affine): the scale an fp32 sum over those pixels is accurate to."""
    ws, bs, gw, gb = [[t.clone().requires_grad_(True) for t in group] if isinstance(group, list)
                      else group.clone().requires_grad_(True) for group in params]
    depth = len(ws)
    G, _, N, _ = x.shape
    xr = x.double().clone().requires_grad_(True)
    y = torch.zeros((G, ws[0].shape[0], N, N), dtype=torch.float64)
    stats = torch.zeros((G, ws[0].shape[0], 2), dtype=torch.float64)
    loss, kept = 0.0, []
    for g in range(G):
        n = sizes[g] if sizes else N
        n_norm = N if (constant_n or not sizes) else n
        h = xr[g:g + 1, :, :n, :n]
        ins, outs = [], []
        for k in range(depth):
            ins.append(h)
            h = O.conv1x1(h, ws[k], bs[k])
            h.retain_grad()
            outs.append(h)
            h = torch.relu(h) if k < depth - 1 else h
        yg = O.graph_norm(h, gw, gb, n_norm, EPS)
        dyg = dy[g:g + 1, :, :n, :n].double()
        loss = loss + (yg * dyg).sum()
        with torch.no_grad():
            stats[g] = plane_stats(h, n_norm)[0]
            y[g, :, :n, :n] = yg[0]
        kept.append((ins, outs, dyg, O.normalize(h.detach(), n_norm, EPS)))
    loss.backward()
    grads = {f"w{k}": ws[k].grad for k in range(depth)}
    grads.update({f"b{k}": bs[k].grad for k in range(depth)})
    grads.update({"gn_w": gw.grad, "gn_b": gb.grad})
    mags = {k: torch.zeros_like(v) for k, v in grads.items()}
    with torch.no_grad():
        for ins, outs, dyg, yn in kept:
            for k in range(depth):
                d, i = outs[k].grad.abs()[0].flatten(1), ins[k].abs()[0].flatten(1)
                mags[f"w{k}"] += d @ i.t()
                mags[f"b{k}"] += d.sum(1)
            mags["gn_w"] += (dyg * yn).abs().sum(dim=(0, 2, 3))
            mags["gn_b"] += dyg.abs().sum(dim=(0, 2, 3))
    return y, stats, xr.grad, grads, mags


def run_mlp(x, dy, params, sizes, constant_n, flags, seeds, want_dx=True, ws_bytes=None):
    """fgnn_mlp_fwd_f32 then fgnn_mlp_bwd_f32_ex on device copies -> (y, stats, dx, grads - seeds, backward launches)."""
    ws, bs, gw, gb = [[t.float().to(DEV) for t in group] if isinstance(group, list) else group.float().to(DEV)
                      for group in params]
    depth, c_out = len(ws), ws[0].shape[0]
    G, c_in, N, _ = x.shape
    keep = []
    p = _ops.make_mlp_params(ws, bs, gw, gb, EPS, keep, constant_n)
    xd, dyd, npg = x.float().to(DEV), dy.float().to(DEV), i32(sizes)
    y, stats = nan((G, c_out, N, N)), nan((G, c_out, 2))
    fws = scratch(lib().fgnn_mlp_workspace_bytes(G, c_in, c_out, depth, N))
    ok(lib().fgnn_mlp_fwd_f32(L.C.byref(p), L.ptr(xd), L.ptr(y), L.ptr(stats), G, N, L.ptr(npg), L.ptr(fws),
                              fws.numel(), stream()), "fgnn_mlp_fwd_f32")
    bufs = {k: torch.full(tuple(v.shape), seeds[k], device=DEV) for k, v in
            [(f"w{k}", ws[k]) for k in range(depth)] + [(f"b{k}", bs[k]) for k in range(depth)] + [("gn_w", gw), ("gn_b", gb)]}
    g = L.MlpGrads()
    for k in range(depth):
        g.w[k], g.b[k] = bufs[f"w{k}"].data_ptr(), bufs[f"b{k}"].data_ptr()
    g.gn_w, g.gn_b = bufs["gn_w"].data_ptr(), bufs["gn_b"].data_ptr()
    dx = nan((G, c_in, N, N)) if want_dx else None
    nbytes = ws_bytes if ws_bytes is not None else lib().fgnn_mlp_workspace_bytes_ex(G, c_in, c_out, depth, N, flags)
    bws = scratch(nbytes)
    lib().fgnn_reset_launch_count()
    ok(lib().fgnn_mlp_bwd_f32_ex(L.C.byref(p), L.C.byref(g), L.ptr(xd), L.ptr(stats), L.ptr(dyd), L.ptr(dx), G, N,
                                 L.ptr(npg), L.ptr(bws), nbytes, stream(), flags), "fgnn_mlp_bwd_f32_ex")
    launches = lib().fgnn_launch_count()
    torch.cuda.synchronize()
    grads = {k: v.cpu() for k, v in bufs.items()}
    return y.cpu(), stats.cpu(), None if dx is None else dx.cpu(), grads, launches


def mlp_errors(got, ref, sizes, G, N):
    """(forward error, worst gradient error) of run_mlp's result against ref_mlp's; checks the padding zeros.  dx, a
    sum over at most c_out terms per entry, is compared in relative Frobenius norm; each parameter gradient, a sum over
    every pixel of the batch, against the magnitude of its summands (ref_mlp): such a sum can cancel to a small fraction
    of its terms (at width 1 and N = 64 the weight gradient is 2.38 from summands of total magnitude 6.9e4), and its fp32
    rounding is relative to the terms, not to the result."""
    y, stats, dx, grads, _ = got
    ry, rstats, rdx, rgrads, mags = ref
    pad = planes_outside(G, N, sizes)
    assert_zero(y, pad, "y")
    fwd = max(rel_fro(y, ry), rel_fro(stats, rstats))
    gerr = []
    if dx is not None:
        assert_zero(dx, pad, "dx")
        gerr.append(rel_fro(dx, rdx))
    for k, r in rgrads.items():
        d = grads[k].double() - seed_of(r)
        gerr.append(float((d - r).norm() / mags[k].norm().clamp_min(1e-30)))
    return fwd, max(gerr)


@pytest.mark.parametrize("layout", ["dense", "ragged"])
@pytest.mark.parametrize("c_in,c_out,depth,N", MLP_CASES)
def test_mlp_matches_fp64(c_in, c_out, depth, N, layout):
    """y, stats, dx and every parameter gradient of one MlpBlock_Real, flags 0 and FGNN_DETERMINISTIC, constant_n 0 and
    1, against the fp64 oracle; dx = NULL leaves the parameter gradients bitwise unchanged; a c_in above 128 exercises the
    sliced input gradient."""
    gen = torch.Generator().manual_seed(1000 * c_in + 10 * c_out + N)
    sizes = ragged_sizes(N) if layout == "ragged" else None
    G = 3 if sizes else 2
    params = mlp_params(c_in, c_out, depth, gen)
    x = torch.randn((G, c_in, N, N), generator=gen)
    dy = torch.randn((G, c_out, N, N), generator=gen)
    pad = planes_outside(G, N, sizes)
    x, dy = filled(x, pad, 0.0), filled(dy, pad, 0.0)
    worst_f = worst_g = 0.0
    for constant_n in ((False, True) if sizes else (True,)):
        ref = ref_mlp(x, dy, params, sizes, constant_n)
        seeds = {k: seed_of(v) for k, v in ref[3].items()}
        for flags in (0, DET):
            got = run_mlp(x, dy, params, sizes, constant_n, flags, seeds)
            f, g = mlp_errors(got, ref, sizes, G, N)
            worst_f, worst_g = max(worst_f, f), max(worst_g, g)
            assert f < TOL_MLP_FWD and g < TOL_MLP_GRAD, (constant_n, flags, f, g)
            if flags == DET:
                no_dx = run_mlp(x, dy, params, sizes, constant_n, flags, seeds, want_dx=False)
                assert all(torch.equal(got[3][k], no_dx[3][k]) for k in got[3]), "dx = NULL changed a gradient"
            if sizes:
                big = run_mlp(filled(x, pad, PAD), filled(dy, pad, PAD), params, sizes, constant_n, flags, seeds)
                assert torch.equal(big[0], got[0]) and torch.equal(big[1], got[1]) and torch.equal(big[2], got[2])
                if flags == DET:
                    assert all(torch.equal(big[3][k], got[3][k]) for k in got[3])
                else:
                    f, g = mlp_errors(big, ref, sizes, G, N)
                    assert f < TOL_MLP_FWD and g < TOL_MLP_GRAD, (constant_n, flags, f, g)
    print(f"PARITY mlp c_in={c_in} c_out={c_out} depth={depth} N={N} {layout}: forward {worst_f:.2e} gradients {worst_g:.2e}")


@pytest.mark.parametrize("flags", [0, DET])
def test_mlp_backward_in_graph_chunks(flags):
    """fgnn_mlp_bwd_f32_ex with a workspace for 1 and for 2 of its 5 graphs runs its graph-chunk loop (5 = 1+1+1+1+1 and
    2+2+1, an uneven last chunk): same result as the full workspace (to the rounding of the per-chunk gradient sums)
    and as fp64."""
    c_in, c_out, depth, N = 7, 9, 3, 12
    sizes = [12, 5, 1, 12, 9]
    G = len(sizes)
    gen = torch.Generator().manual_seed(77)
    params = mlp_params(c_in, c_out, depth, gen)
    pad = planes_outside(G, N, sizes)
    x = filled(torch.randn((G, c_in, N, N), generator=gen), pad, 0.0)
    dy = filled(torch.randn((G, c_out, N, N), generator=gen), pad, 0.0)
    ref = ref_mlp(x, dy, params, sizes, True)
    seeds = {k: seed_of(v) for k, v in ref[3].items()}
    full = lib().fgnn_mlp_workspace_bytes_ex(G, c_in, c_out, depth, N, flags)
    per_graph = (depth + 2) * max(c_in, c_out) * N * N * 4 + 256 * (depth + 2)     # fgnn_f32_bwd.cu's chunk unit
    runs = {k: run_mlp(x, dy, params, sizes, True, flags, seeds, ws_bytes=full - (G - k) * per_graph) for k in (1, 2)}
    runs[G] = run_mlp(x, dy, params, sizes, True, flags, seeds)
    assert runs[1][4] > runs[2][4] > runs[G][4], "the smaller workspaces did not run more chunks"
    worst = 0.0
    for k, got in runs.items():
        f, g = mlp_errors(got, ref, sizes, G, N)
        assert f < TOL_MLP_FWD and g < TOL_MLP_GRAD, (k, f, g)
        assert torch.equal(got[2], runs[G][2])                                  # dx: no cross-graph sum
        worst = max(worst, g, max(float((got[3][n].double() - runs[G][3][n].double()).norm() / ref[4][n].norm())
                                  for n in got[3]))
    print(f"PARITY mlp backward in chunks flags={flags}: worst {worst:.2e}")
    assert worst < TOL_MLP_GRAD


# --------------------------------------------------------------------------------------------------------------------
# fgnn_graphnorm_fwd_f32
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["dense", "ragged"])
@pytest.mark.parametrize("affine", [False, True])
def test_graphnorm_matches_fp64(affine, layout):
    """GraphNorm (affine) and normalize (gn_w = gn_b = NULL), with a graph of one vertex in the ragged batch."""
    G, C, N = 3, 5, 13
    sizes = [13, 1, 7] if layout == "ragged" else None
    gen = torch.Generator().manual_seed(11)
    pad = planes_outside(G, N, sizes)
    x = filled(torch.randn((G, C, N, N), generator=gen) * 3 + 1, pad, 0.0)
    gw = (torch.rand(C, generator=gen) + 0.5) if affine else None
    gb = (torch.rand(C, generator=gen) - 0.5) if affine else None
    worst = 0.0
    for constant_n in ((False, True) if sizes else (True,)):
        ry = torch.zeros((G, C, N, N), dtype=torch.float64)
        rs = torch.zeros((G, C, 2), dtype=torch.float64)
        for g in range(G):
            n = sizes[g] if sizes else N
            n_norm = N if (constant_n or not sizes) else n
            xs = x[g:g + 1, :, :n, :n].double()
            ry[g, :, :n, :n] = (O.graph_norm(xs, gw.double(), gb.double(), n_norm, EPS) if affine
                                else O.normalize(xs, n_norm, EPS))[0]
            rs[g] = plane_stats(xs, n_norm)[0]
        outs = []
        for xin in ([x, filled(x, pad, PAD)] if sizes else [x]):
            y, st = nan((G, C, N, N)), nan((G, C, 2))
            gwd = gw.to(DEV) if affine else None
            gbd = gb.to(DEV) if affine else None
            xd, npg = xin.to(DEV), i32(sizes)
            ok(lib().fgnn_graphnorm_fwd_f32(L.ptr(xd), L.ptr(y), L.ptr(st), L.ptr(gwd), L.ptr(gbd), EPS, int(constant_n),
                                            G, C, N, L.ptr(npg), stream()), "fgnn_graphnorm_fwd_f32")
            outs.append((y.cpu(), st.cpu()))
        y, st = outs[0]
        assert_zero(y, pad, "y")
        for y2, st2 in outs[1:]:
            assert torch.equal(y2, y) and torch.equal(st2, st)
        e = max(rel_fro(y, ry), rel_fro(st, rs))
        worst = max(worst, e)
        assert e < TOL_GN, (constant_n, e)
    print(f"PARITY graphnorm affine={affine} {layout}: {worst:.2e}")


# --------------------------------------------------------------------------------------------------------------------
# fgnn_matmul_fwd_f32 / fgnn_matmul_bwd_f32
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [1, 15, 63, 64, 65, 127, 128, 129, 300])
def test_matmul_matches_fp64(N):
    """out = a @ b and its backward (da = dout b^T, db = a^T dout, each alone and both at once) past the first 64-tile;
    in the ragged batch one graph's n_g <= 64 < N leaves whole tiles in the padding."""
    gen = torch.Generator().manual_seed(N)
    C = 2
    worst = 0.0
    for sizes in (None, [N, 40 if N > 64 else max(1, N // 2), 1]):
        G = 3 if sizes else 2
        pad = planes_outside(G, N, sizes)
        a, b, dout = (filled(torch.randn((G, C, N, N), generator=gen), pad, 0.0) for _ in range(3))
        ro, rda, rdb = (torch.zeros((G, C, N, N), dtype=torch.float64) for _ in range(3))
        for g in range(G):
            n = sizes[g] if sizes else N
            A, B, D = (t[g, :, :n, :n].double() for t in (a, b, dout))
            ro[g, :, :n, :n] = A @ B
            rda[g, :, :n, :n] = D @ B.transpose(-1, -2)
            rdb[g, :, :n, :n] = A.transpose(-1, -2) @ D
        results = []
        for fill in ((0.0, PAD) if sizes else (0.0,)):
            ad, bd, dd = (filled(t, pad, fill).to(DEV) for t in (a, b, dout))
            npg = i32(sizes)
            out = nan((G, C, N, N))
            ok(lib().fgnn_matmul_fwd_f32(L.ptr(ad), L.ptr(bd), L.ptr(out), G, C, N, L.ptr(npg), stream()), "matmul fwd")
            grads = []
            for want_a, want_b in ((True, True), (True, False), (False, True)):
                da = nan((G, C, N, N)) if want_a else None
                db = nan((G, C, N, N)) if want_b else None
                ok(lib().fgnn_matmul_bwd_f32(L.ptr(ad), L.ptr(bd), L.ptr(dd), L.ptr(da), L.ptr(db), G, C, N, L.ptr(npg),
                                             stream()), "matmul bwd")
                grads.append((None if da is None else da.cpu(), None if db is None else db.cpu()))
            assert torch.equal(grads[1][0], grads[0][0]) and torch.equal(grads[2][1], grads[0][1])
            results.append((out.cpu(), *grads[0]))
        for t in results[0]:
            assert_zero(t, pad, "matmul")
        for other in results[1:]:
            assert all(torch.equal(u, v) for u, v in zip(other, results[0]))
        e = max(rel_fro(results[0][0], ro), rel_fro(results[0][1], rda), rel_fro(results[0][2], rdb))
        worst = max(worst, e)
        assert e < TOL_MM, (sizes, e)
    print(f"PARITY matmul N={N}: {worst:.2e}")


# --------------------------------------------------------------------------------------------------------------------
# fgnn_colmax_fwd_f32 / fgnn_colmax_bwd_f32
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["dense", "ragged"])
@pytest.mark.parametrize("N", [1, 33, 100])
def test_colmax_exact(N, layout):
    """Max values, arg-max and the backward are exact.  Ties go to the lowest maximal column, across lanes (columns 2
    and 5) and within one lane (3 and 35); channel 1 is negative everywhere."""
    G, C = 2, 3
    sizes = [N, max(1, N // 3)] if layout == "ragged" else None
    gen = torch.Generator().manual_seed(N + 5)
    x = torch.randn((G, C, N, N), generator=gen)
    x[:, 1] = -x[:, 1].abs() - 1
    for (i, j1, j2) in ((0, 2, 5), (1, 3, 35), (2, 5, 2)):
        if max(i, j1, j2) < (min(sizes) if sizes else N):
            for g in range(G):
                for c in range(C):
                    x[g, c, i, j1] = x[g, c, i, j2] = x[g, c, i].max() + 1
    pad = planes_outside(G, N, sizes)
    x = filled(x, pad, 0.0)
    rows_pad = vec_outside(G, N, sizes).expand(G, C, N)
    ref_val = torch.zeros((G, C, N))
    ref_arg = torch.zeros((G, C, N), dtype=torch.int64)
    for g in range(G):
        n = sizes[g] if sizes else N
        v = x[g, :, :n, :n].numpy()
        ref_arg[g, :, :n] = torch.from_numpy(np.argmax(v, axis=-1))           # numpy: the first maximal column
        ref_val[g, :, :n] = torch.from_numpy(v.max(axis=-1))
    dout = torch.randn((G, C, N), generator=gen)
    ref_dx = torch.zeros((G, C, N, N))
    valid = ~rows_pad
    gi, ci, ri = valid.nonzero(as_tuple=True)
    ref_dx[gi, ci, ri, ref_arg[gi, ci, ri]] = dout[gi, ci, ri]
    outs = []
    for fill in ((0.0, PAD) if sizes else (0.0,)):
        xd, npg, dd = filled(x, pad, fill).to(DEV), i32(sizes), dout.to(DEV)
        out, arg = nan((G, C, N)), torch.full((G, C, N), -7, dtype=torch.int32, device=DEV)
        ok(lib().fgnn_colmax_fwd_f32(L.ptr(xd), L.ptr(out), L.ptr(arg), G, C, N, L.ptr(npg), stream()), "colmax fwd")
        dx = nan((G, C, N, N))
        ok(lib().fgnn_colmax_bwd_f32(L.ptr(dd), L.ptr(arg), L.ptr(dx), G, C, N, L.ptr(npg), stream()), "colmax bwd")
        outs.append((out.cpu(), arg.cpu(), dx.cpu()))
    out, arg, dx = outs[0]
    assert torch.equal(out, ref_val)                                           # padded rows: exact zeros
    assert torch.equal(arg[valid].long(), ref_arg[valid])
    assert torch.equal(dx, ref_dx)
    for other in outs[1:]:
        assert all(torch.equal(u, v) for u, v in zip(other, outs[0]))


# --------------------------------------------------------------------------------------------------------------------
# fgnn_scores_pair_fwd_f32 / fgnn_scores_pair_bwd_f32
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N1,N2", [(15, 17), (17, 15), (127, 129), (129, 127)])
@pytest.mark.parametrize("C", [1, 17, 100, 128])
def test_scores_match_fp64(C, N1, N2):
    """scores = e1^T e2 and its backward with N1 != N2 on both sides of the 16- and 128-wide tiles, dense and ragged."""
    gen = torch.Generator().manual_seed(C * 1000 + N1)
    G = 2
    worst = 0.0
    for n1, n2 in ((None, None), ([N1, N1 // 2 + 1], [N2 - 3, N2])):
        sp = outside(G, N1, N2, n1, n2)
        p1, p2 = vec_outside(G, N1, n1), vec_outside(G, N2, n2)
        e1 = filled(torch.randn((G, C, N1), generator=gen), p1, 0.0)
        e2 = filled(torch.randn((G, C, N2), generator=gen), p2, 0.0)
        ds = filled(torch.randn((G, N1, N2), generator=gen), sp, 0.0)
        rs = torch.zeros((G, N1, N2), dtype=torch.float64)
        rd1 = torch.zeros((G, C, N1), dtype=torch.float64)
        rd2 = torch.zeros((G, C, N2), dtype=torch.float64)
        for g in range(G):
            a = n1[g] if n1 else N1
            b = n2[g] if n2 else N2
            x1 = e1[g:g + 1, :, :a].double().requires_grad_(True)
            x2 = e2[g:g + 1, :, :b].double().requires_grad_(True)
            s = O.siamese_scores(x1, x2)
            (s * ds[g:g + 1, :a, :b].double()).sum().backward()
            rs[g, :a, :b], rd1[g, :, :a], rd2[g, :, :b] = s[0].detach(), x1.grad[0], x2.grad[0]
        outs = []
        for fill in ((0.0, PAD) if n1 else (0.0,)):
            d1, d2, dd = filled(e1, p1, fill).to(DEV), filled(e2, p2, fill).to(DEV), filled(ds, sp, fill).to(DEV)
            s, g1, g2 = nan((G, N1, N2)), nan((G, C, N1)), nan((G, C, N2))
            s1, s2 = i32(n1), i32(n2)
            ok(lib().fgnn_scores_pair_fwd_f32(L.ptr(d1), L.ptr(d2), L.ptr(s), G, C, N1, N2, L.ptr(s1), L.ptr(s2),
                                              stream()), "scores fwd")
            ok(lib().fgnn_scores_pair_bwd_f32(L.ptr(d1), L.ptr(d2), L.ptr(dd), L.ptr(g1), L.ptr(g2), G, C, N1, N2,
                                              L.ptr(s1), L.ptr(s2), stream()), "scores bwd")
            outs.append((s.cpu(), g1.cpu(), g2.cpu()))
        s, g1, g2 = outs[0]
        assert_zero(s, sp, "scores")
        assert_zero(g1, p1, "de1")
        assert_zero(g2, p2, "de2")
        for other in outs[1:]:
            assert all(torch.equal(u, v) for u, v in zip(other, outs[0]))
        e = max(rel_fro(s, rs), rel_fro(g1, rd1), rel_fro(g2, rd2))
        worst = max(worst, e)
        assert e < TOL_SCORES, (n1, e)
    print(f"PARITY scores C={C} N1={N1} N2={N2}: {worst:.2e}")


# --------------------------------------------------------------------------------------------------------------------
# fgnn_ce_pair_argmax_fwd_f32 / fgnn_ce_pair_bwd_f32
# --------------------------------------------------------------------------------------------------------------------
def margin_scores(n1, n2, gen):
    """(n1, n2) scores with |s| <= 80 (exp overflows fp32 without the max shift) and a unique row maximum at least 1
    above the rest: the even rows' maximum on the diagonal, the odd rows' elsewhere.  Row 0 has an exact tie between
    columns 2 and 5 when n2 > 5 (the lowest wins)."""
    s = (torch.randn((n1, n2), generator=gen) * 25).clamp(-78, 78)
    for i in range(n1):
        top = float(s[i].max())
        if i % 2 == 0 and i < n2:
            s[i, i] = top + 1
        else:
            s[i, int(s[i].argmax())] = top + 1
    s[0, 0] = 80.0 if n2 > 1 else s[0, 0]
    if n2 > 5:
        s[0, 2] = s[0, 5] = 80.0
        s[0, 0] = 70.0
    return s


@pytest.mark.parametrize("N2", [1, 31, 33, 4096])
def test_ce_matches_fp64(N2):
    """Row-softmax cross-entropy against the identity matching: ce_sum, row_lse and the gradient (per-graph coef) against
    fp64; correct and row_argmax exact; rows i >= n2 carry no target (no loss, zero gradient)."""
    N1 = N2 + 3 if N2 < 4096 else 50
    G = 3
    gen = torch.Generator().manual_seed(N2)
    coef = torch.tensor([0.5, 1.25, 2.0])
    worst = 0.0
    for n1, n2 in ((None, None), ([N1, max(1, N1 // 2), 1], [N2, max(1, N2 - 2), 1])):
        sp = outside(G, N1, N2, n1, n2)
        s = torch.zeros((G, N1, N2))
        for g in range(G):
            a, b = (n1[g] if n1 else N1), (n2[g] if n2 else N2)
            s[g, :a, :b] = margin_scores(a, b, gen)
        rce = torch.zeros(G, dtype=torch.float64)
        rlse = torch.zeros((G, N1), dtype=torch.float64)
        rarg = torch.full((G, N1), -1, dtype=torch.int64)
        rds = torch.zeros((G, N1, N2), dtype=torch.float64)
        rcorrect = []
        for g in range(G):
            a, b = (n1[g] if n1 else N1), (n2[g] if n2 else N2)
            S = s[g, :a, :b].double().requires_grad_(True)
            m = min(a, b)
            ce = O.ce_sum_identity(S[:m])
            (coef[g].double() * ce).backward()
            rce[g], rds[g, :a, :b] = ce.detach(), S.grad
            rlse[g, :a] = torch.logsumexp(S.detach(), -1)
            rarg[g, :a] = torch.from_numpy(np.argmax(s[g, :a, :b].numpy(), axis=-1))
            rcorrect.append(int((rarg[g, :m] == torch.arange(m)).sum()))
        outs = []
        for fill in ((0.0, PAD) if n1 else (0.0,)):
            sd = filled(s, sp, fill).to(DEV)
            ce, correct = nan((G,)), torch.full((G,), -7, dtype=torch.int32, device=DEV)
            lse, arg = nan((G, N1)), torch.full((G, N1), -7, dtype=torch.int32, device=DEV)
            ws = scratch(lib().fgnn_ce_workspace_bytes(G, N1))
            s1, s2, cd = i32(n1), i32(n2), coef.to(DEV)
            ok(lib().fgnn_ce_pair_argmax_fwd_f32(L.ptr(sd), L.ptr(ce), L.ptr(correct), L.ptr(lse), L.ptr(arg), G, N1, N2,
                                                 L.ptr(s1), L.ptr(s2), L.ptr(ws), ws.numel(), stream()), "ce fwd")
            ds = nan((G, N1, N2))
            ok(lib().fgnn_ce_pair_bwd_f32(L.ptr(sd), L.ptr(lse), L.ptr(cd), L.ptr(ds), G, N1, N2, L.ptr(s1), L.ptr(s2),
                                          stream()), "ce bwd")
            outs.append((ce.cpu(), correct.cpu(), lse.cpu(), arg.cpu(), ds.cpu()))
        ce, correct, lse, arg, ds = outs[0]
        for other in outs[1:]:
            assert all(torch.equal(u, v) for u, v in zip(other, outs[0]))
        assert correct.tolist() == rcorrect
        assert torch.equal(arg.long(), rarg)
        if N2 > 5:
            assert int(arg[0, 0]) == 2                                        # the tie: lowest column
        assert_zero(ds, sp, "dscores")
        lse_pad = vec_outside(G, N1, n1)[:, 0]
        assert_zero(lse, lse_pad, "row_lse")
        for g in range(G):                                                    # rows without a target: zero gradient
            a, b = (n1[g] if n1 else N1), (n2[g] if n2 else N2)
            assert not ds[g, b:a].any()
        e = max(rel_fro(ce, rce), rel_fro(lse, rlse), rel_fro(ds, rds))
        worst = max(worst, e)
        assert e < TOL_CE, (n1, e)
    print(f"PARITY ce N2={N2}: {worst:.2e}")


# --------------------------------------------------------------------------------------------------------------------
# fgnn_adam_step_f32
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 400_001])
def test_adam_matches_torch_adam_in_fp64(n):
    """50 steps against torch.optim.Adam on float64 copies (weight_decay > 0; the gradient divisor alternates between 3
    and 0.5, which the kernel clamps to 1).  400 001 entries pass the grid-stride loop's first 1184 x 256 threads.  A
    step with skip_flag set changes nothing, bit for bit.  The reference takes the hyperparameters the kernel receives,
    rounded to float32 by the C ABI (as torch's own fp32 Adam rounds them): beta2 = 0.999 becomes 0.99900001287, which
    moves 1 - beta2, and with it exp_avg_sq, by 1.3e-5."""
    lr, b1, b2, eps, wd = (float(np.float32(v)) for v in (1e-3, 0.9, 0.999, 1e-8, 0.01))
    betas = (b1, b2)
    gen = torch.Generator().manual_seed(n)
    p0 = torch.randn(n, generator=gen) * 1e-2
    ref = p0.double().clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=lr, betas=betas, eps=eps, weight_decay=wd)
    p, m, v = p0.to(DEV), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    skip = torch.ones(1, device=DEV)
    for t in range(1, 51):
        g = torch.randn(n, generator=gen)
        div = 3.0 if t % 2 else 0.5
        gd, divd = g.to(DEV), torch.tensor([div], device=DEV)
        if t == 25:
            before = [u.clone() for u in (p, m, v)]
            ok(lib().fgnn_adam_step_f32(L.ptr(p), L.ptr(gd), L.ptr(m), L.ptr(v), n, lr, betas[0], betas[1], eps, wd, t,
                                        L.ptr(divd), L.ptr(skip), stream()), "adam (skipped)")
            assert all(torch.equal(u, w) for u, w in zip((p, m, v), before))
        ok(lib().fgnn_adam_step_f32(L.ptr(p), L.ptr(gd), L.ptr(m), L.ptr(v), n, lr, betas[0], betas[1], eps, wd, t,
                                    L.ptr(divd), None, stream()), "adam")
        ref.grad = g.double() / max(div, 1.0)
        opt.step()
    st = opt.state[ref]
    e = max(rel_fro(p.cpu().double() - p0.double(), ref.detach() - p0.double()),
            rel_fro(m.cpu(), st["exp_avg"]), rel_fro(v.cpu(), st["exp_avg_sq"]))
    print(f"PARITY adam n={n}: {e:.2e}")
    assert e < TOL_ADAM


# --------------------------------------------------------------------------------------------------------------------
# the fp32 mode end to end at widths the 16-bit path refuses
# --------------------------------------------------------------------------------------------------------------------
WIDE_SIZES = [17, 40, 33]


def wide_model(in_f, out_f, nb, cst, seed=3):
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=nb,
                    in_features=in_f, out_features=out_f, depth_of_mlp=2, constant_n_vertices=cst)
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    sd = O.xavier_state_dict(2, in_f, nb, 2, torch.Generator().manual_seed(seed), c_out=out_f, randomize_gn=True)
    model.load_state_dict(sd)
    return model.to(DEV).set_precision("fp32"), sd


def wide_batch(seed=9):
    gen = torch.Generator().manual_seed(seed)
    pairs = [O.synthetic_pair(s, 0.3, 0.1, gen) for s in WIDE_SIZES]
    return [p[0] for p in pairs], [p[1] for p in pairs]


def oracle_loss_and_grads(sd, g1, g2, n, dtype=torch.float64):
    """The oracle's siamese loss ('mean') over graph pairs run one at a time, its embeddings of g1, d loss / d parameter by
    autograd, and for every parameter gradient the magnitude of its summands, as in ref_mlp: every conv1x1 and
    graph_norm call of the oracle is recorded with its input and its output's gradient."""
    conv, gn, calls = O.conv1x1, O.graph_norm, []

    def conv_rec(x, w, b):
        out = conv(x, w, b)
        out.retain_grad()
        calls.append((w, b, x.detach(), out))
        return out

    def gn_rec(y, weight, bias, n=None, eps=1e-5):
        out = gn(y, weight, bias, n, eps)
        out.retain_grad()
        calls.append((weight, bias, O.normalize(y.detach(), n, eps), out))
        return out

    params = {k: v.detach().to(dtype).clone().requires_grad_(True) for k, v in sd.items()}
    O.conv1x1, O.graph_norm = conv_rec, gn_rec
    try:
        e1, scores = [], []
        for a, b in zip(g1, g2):
            r1 = O.node_embedding(a[None].to(dtype), params, n)[0]
            r2 = O.node_embedding(b[None].to(dtype), params, n)[0]
            e1.append(r1.detach())
            scores.append(r1.t() @ r2)
        loss = O.triplet_loss(scores)
    finally:
        O.conv1x1, O.graph_norm = conv, gn
    loss.backward()
    name = {id(v): k for k, v in params.items()}
    mags = {k: torch.zeros_like(v) for k, v in params.items()}
    with torch.no_grad():
        for w, b, inp, out in calls:
            d = out.grad.abs()[0].flatten(1)
            if name[id(w)].endswith("gn.weight"):                      # graph_norm: inp is normalize(y)
                mags[name[id(w)]] += (d * inp.abs()[0].flatten(1)).sum(1).reshape(w.shape)
            else:                                                       # conv1x1
                mags[name[id(w)]] += (d @ inp.abs()[0].flatten(1).t()).reshape(w.shape)
            mags[name[id(b)]] += d.sum(1).reshape(b.shape)
    return loss.detach(), e1, {k: v.grad for k, v in params.items()}, mags


@pytest.mark.parametrize("cst", [False, True])
@pytest.mark.parametrize("in_f,out_f,nb", [(96, 96, 2), (128, 128, 2), (64, 65, 3), (128, 32, 2)])
def test_wide_fp32_model_matches_fp64(in_f, out_f, nb, cst):
    """Siamese_Node_Exp in fp32 with an MLP input wider than 128 channels (every block's mlp3 reads in + out channels):
    embeddings, loss and every parameter gradient of a ragged batch against the fp64 oracle's autograd.  Each gradient
    is bounded against the magnitude of its summands, as in test_mlp_matches_fp64: some are pixel sums that cancel to a
    small fraction of their terms (the first conv bias of block 2's mlp2 at in = out = 96), and there even the oracle
    itself, run in fp32 on the CPU, is 1.1e-3 of the result away from fp64, 1.6e-4 over the whole gradient."""
    model, sd = wide_model(in_f, out_f, nb, cst)
    g1, g2 = wide_batch()
    N = max(WIDE_SIZES)
    x1 = mt.from_list(g1, dims=(1, 2)).to(DEV)
    x2 = mt.from_list(g2, dims=(1, 2)).to(DEV)
    e1 = model.embed({"input": x1})
    scores = model({"input": x1}, {"input": x2})
    loss = pkg.toolbox.losses.triplet_loss("mean")(scores)
    loss.backward()
    ref_loss, ref_e1, ref_grads, mags = oracle_loss_and_grads(sd, g1, g2, N if cst else None)
    plain = e1.tensor.rename(None).detach().cpu()
    e_emb = max(rel_fro(plain[i, :, :n], r) for i, (n, r) in enumerate(zip(WIDE_SIZES, ref_e1)))
    assert e_emb < TOL_WIDE_FWD, e_emb
    assert abs(float(loss.detach()) - float(ref_loss)) < TOL_WIDE_FWD * abs(float(ref_loss))
    fp32_grads = oracle_loss_and_grads(sd, g1, g2, N if cst else None, torch.float32)[2]
    worst, worst_k, floor = 0.0, None, 0.0
    for k, p in model.named_parameters():
        e = float((p.grad.cpu().double() - ref_grads[k]).norm() / mags[k].norm())
        floor = max(floor, float((fp32_grads[k].double() - ref_grads[k]).norm() / mags[k].norm()))
        if e > worst:
            worst, worst_k = e, k
    print(f"PARITY wide fp32 model in={in_f} out={out_f} blocks={nb} constant_n={cst}: embeddings {e_emb:.2e} "
          f"gradients {worst:.2e} ({worst_k}); the oracle in fp32 on the CPU: {floor:.2e}")
    assert worst < TOL_WIDE_GRAD, (worst_k, worst)


def test_wide_fp32_model_trains():
    """Six train_step_flat steps of a width-96 model (mlp3 reads 192 channels) lower the loss."""
    from graph_neural_net_b200.training import train_step_flat, FlatAdam
    model, _ = wide_model(96, 96, 2, False)
    g1, g2 = wide_batch()
    x1 = mt.from_list(g1, dims=(1, 2)).to(DEV)
    x2 = mt.from_list(g2, dims=(1, 2)).to(DEV)
    opt = FlatAdam(model.parameters(), lr=model.lr)
    losses = [train_step_flat(model, opt, {"input": x1}, {"input": x2})[0] for _ in range(6)]
    print("fp32 train_step_flat in=96 out=96 losses", [round(v, 4) for v in losses])
    assert all(math.isfinite(v) for v in losses) and losses[-1] < losses[0]


def test_fp32_width_limits_are_stated():
    """A c_out of 129 and a c_in of 513 are refused as invalid arguments naming the limit, before any launch."""
    from graph_neural_net_b200.models.layers import MlpBlock_Real
    x = torch.zeros((1, 2, 8, 8), device=DEV)
    with pytest.raises(L.FgnnError, match=r"status 1\).*c_out 129 unsupported \(max 128\)"):
        MlpBlock_Real(2, 129, 2).to(DEV)(x)
    with pytest.raises(L.FgnnError, match=r"status 1\).*c_in 513 unsupported \(max 512\)"):
        MlpBlock_Real(513, 8, 2).to(DEV)(torch.zeros((1, 513, 8, 8), device=DEV))
    model, _ = wide_model(129, 129, 2, False)
    with torch.no_grad(), pytest.raises(L.FgnnError, match=r"status 1\).*max 128"):
        model.node_embedder.forward_fused(torch.zeros((1, 2, 8, 8), device=DEV), "fp32")
    torch.cuda.synchronize()


# --------------------------------------------------------------------------------------------------------------------
# batches of more than 65 535 (graph, channel) planes
# --------------------------------------------------------------------------------------------------------------------
PG, PC, PN = 2049, 32, 5            # 65 568 planes


def test_many_planes_mlp_matmul_normalize():
    """MlpFunction (forward and backward), Matmul (forward and backward) and normalize on 2 049 graphs x 32 channels:
    more planes than one grid dimension holds."""
    from graph_neural_net_b200.models.layers import MlpBlock_Real, Matmul, normalize
    gen = torch.Generator().manual_seed(2049)
    mlp = MlpBlock_Real(4, PC, 2).to(DEV)
    sd = {f"m.{k}": v.detach().cpu().double().requires_grad_(True) for k, v in mlp.state_dict().items()}
    x = torch.randn((PG, 4, PN, PN), generator=gen)
    dy = torch.randn((PG, PC, PN, PN), generator=gen)
    xd = x.to(DEV).requires_grad_(True)
    y = mlp(xd)
    (y * dy.to(DEV)).sum().backward()
    xr = x.double().requires_grad_(True)
    ry = O.mlp_block(xr, sd, "m", 2, None, EPS)
    (ry * dy.double()).sum().backward()
    e = [rel_fro(y.detach().cpu(), ry.detach()), rel_fro(xd.grad.cpu(), xr.grad)]
    for k, p in mlp.named_parameters():
        if k != "convs.1.bias":
            e.append(rel_fro(p.grad.cpu(), sd["m." + k].grad))
    a, b, dout = (torch.randn((PG, PC, PN, PN), generator=gen) for _ in range(3))
    ad, bd = a.to(DEV).requires_grad_(True), b.to(DEV).requires_grad_(True)
    out = Matmul()(ad, bd)
    out.backward(dout.to(DEV))
    A, B, D = a.double(), b.double(), dout.double()
    e += [rel_fro(out.detach().cpu(), A @ B), rel_fro(ad.grad.cpu(), D @ B.transpose(-1, -2)),
          rel_fro(bd.grad.cpu(), A.transpose(-1, -2) @ D)]
    e.append(rel_fro(normalize(a.to(DEV)).cpu(), O.normalize(A, None, EPS)))
    print(f"PARITY {PG * PC} planes (mlp, matmul, normalize): {max(e):.2e}")
    assert max(e) < TOL_PLANES and max(e[-4:]) < TOL_MM, e


def test_many_planes_fused_fp32_embedder():
    """forward_fused(x, 'fp32') on 2 049 graphs of a width-32 model: one pass of 65 568 planes."""
    model, sd = wide_model(32, 32, 2, True)
    x = torch.stack([O.synthetic_pair(PN, 0.4, 0.1, torch.Generator().manual_seed(s))[0] for s in range(PG)])
    with torch.no_grad():
        e = model.node_embedder.forward_fused(x.to(DEV), "fp32").cpu()
    r = O.node_embedding(x.double(), {k: v.double() for k, v in sd.items()})
    err = rel_fro(e, r)
    print(f"PARITY fused fp32 embedder, {PG} graphs: {err:.2e}")
    assert err < TOL_FUSED
