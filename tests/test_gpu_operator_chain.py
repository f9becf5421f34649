"""The per-layer operator chain block by block: ``mobo_layer_precompute`` (opchain_kernel) and
``mobo_layer_precompute_bwd`` through the C ABI, against plain high-precision references of the same operations.

- Forward: every block of the operator buffer (P, L, W, H, their transposes, LQ, the four fragment-order copies, beta,
  the KL pieces) against a longdouble covariance reference and a longdouble factor of the device's own P, plus the
  exact structure (transposes, triangles, identity / zero padding) the row kernels rely on.
- The psd_safe_cholesky retries with the first bad pivot in the first, a middle and the last diagonal block, a failure
  after three retries followed by a reuse of the same buffer, and a fused step whose layers need different retry counts
  inside one cooperative launch.
- Backward: d theta, d zf, d m and d L_q against torch fp64 autograd of the loss whose whitened gradient statistics
  the gradient buffer carries, one upstream term at a time so that no term hides another.
- Caller memory: every entry point that takes caller scratch, run once on zeroed and once on NaN-filled buffers, must
  give bit-identical results (the library never assumes caller memory is zeroed).

The GPU tests are marked one by one; the table-coverage and layout tests run on the CPU."""
import math

import numpy as np
import pytest
import torch

from mobocmf_b200 import _lib
from mobocmf_b200 import functional as F
from oracle import ld_autodiff as LDA
from oracle import mfdgp_oracle as O

DEV = "cuda:0"
EPS = 2.220446049250313e-16
LD = np.longdouble
F64 = torch.float64
# A quiet NaN whose two 32-bit halves are both 0x7FF80000, a large positive int: a flag or counter nobody reset reads
# as "ready" / "failed" (wrong numbers, never a wait that cannot end: the flags are waited on with flag >= want).
G_BITS = 0x7FF800007FF80000
G = torch.tensor(G_BITS).view(F64)
COND_MAX = 1e5

# ---- case tables ------------------------------------------------------------------------------------------------
# forward: (kind, M, d, lengthscale, jitter).  Every block count nb = MP / 32 = 1 .. 8 for both kinds, M mod 32 in
# {0, 1, 31} and others, M = 1 and 2, every d for both kinds, one larger jitter.  Each lengthscale keeps
# cond(K_zz + jitter I) <= COND_MAX (asserted), with the largest value that does.
FWD_CASES = [
    (0, 1, 1, 0.5, 1e-6), (0, 32, 2, 0.15, 1e-6), (0, 33, 3, 0.34, 1e-6), (0, 95, 4, 0.37, 1e-6),
    (0, 128, 5, 0.45, 1e-6), (0, 150, 6, 0.56, 1e-6), (0, 161, 7, 0.66, 1e-6), (0, 193, 8, 0.69, 1e-6),
    (0, 256, 8, 0.63, 1e-6), (0, 2, 1, 0.5, 1e-6), (0, 70, 3, 0.3, 1e-4),
    (1, 1, 2, 0.5, 1e-6), (1, 2, 1, 0.5, 1e-6), (1, 31, 1, 0.07, 1e-6), (1, 64, 2, 0.24, 1e-6),
    (1, 65, 3, 0.42, 1e-6), (1, 97, 4, 0.52, 1e-6), (1, 160, 5, 0.58, 1e-6), (1, 191, 6, 0.72, 1e-6),
    (1, 224, 7, 0.71, 1e-6), (1, 255, 8, 0.86, 1e-6),
]
# retries: (M, d, lengthscale, diagonal block of the first non-positive pivot, jitter, expected retries)
RETRY_CASES = [(256, 4, 0.2, blk, jit, r) for blk in (0, 3, 7) for jit, r in ((-5e-9, 1), (-5e-8, 2), (-5e-7, 3))] + \
              [(200, 4, 0.2, 6, jit, r) for jit, r in ((-5e-9, 1), (-5e-8, 2), (-5e-7, 3))]
# backward: (kind, M, d, lengthscale)
BWD_CASES = [(0, 1, 1, 0.5), (0, 33, 3, 0.33), (0, 96, 5, 0.54), (0, 200, 7, 0.71), (0, 256, 6, 0.42),
             (1, 1, 2, 0.5), (1, 33, 4, 1.4), (1, 96, 6, 0.99), (1, 200, 8, 0.98), (1, 256, 3, 0.2)]


def test_case_tables_cover_the_kernel_edges():
    nbs = {k: {(M + 31) // 32 for kk, M, _, _, _ in FWD_CASES if kk == k} for k in (0, 1)}
    assert nbs[0] == nbs[1] == set(range(1, 9))
    res = {M % 32 for _, M, _, _, _ in FWD_CASES}
    assert {0, 1, 31} <= res and res - {0, 1, 31}
    assert {1, 2} <= {M for _, M, _, _, _ in FWD_CASES}
    for k in (0, 1):
        assert {d for kk, _, d, _, _ in FWD_CASES if kk == k} == set(range(1, 9))
    assert any(j == 1e-4 for *_, j in FWD_CASES) and all(j in (1e-6, 1e-4) for *_, j in FWD_CASES)
    assert {(blk, r) for M, _, _, blk, _, r in RETRY_CASES if M == 256} == {(b, r) for b in (0, 3, 7) for r in (1, 2, 3)}
    assert any(M % 32 and blk == (M - 1) // 32 for M, _, _, blk, _, _ in RETRY_CASES)
    for k in (0, 1):
        assert {M for kk, M, _, _ in BWD_CASES if kk == k} == {1, 33, 96, 200, 256}
    assert {d for _, _, d, _ in BWD_CASES} == set(range(1, 9))


def test_ops_layout_mirrors_the_library():
    lib = _lib.load()
    for M in range(1, 257):
        lay = F.ops_layout(M)
        MP = lay["MP"]
        assert lay["size"] == lib.mobo_ops_doubles(M) and MP == lib.mobo_padded_m(M)
        blocks = ["L", "W", "WT", "H", "HT", "P", "LQ", "WF", "HTF", "HF", "WTF"]
        assert [lay[b] for b in blocks] == [i * MP * MP for i in range(11)]
        assert lay["alpha"] - lay["beta"] == MP and lay["rowstat"] - lay["scal"] == 16
        assert lay["flags"] - lay["rowstat"] == 4 * MP and lay["size"] - lay["flags"] == 128


# ---- inputs and references ----------------------------------------------------------------------------------------
def case_inputs(kind, M, d, ls, seed):
    """Zx, zf (kind 1), constrained theta, m and a raw L_q: random lower triangle with some negative diagonal entries
    (the raw parameter is unconstrained) and garbage in the strict upper triangle (tril is applied inside)."""
    g = torch.Generator().manual_seed(seed)
    Zx = torch.rand(M, d, generator=g, dtype=F64)
    spread = lambda n: 0.85 + 0.3 * torch.rand(n, generator=g, dtype=F64)
    if kind == 0:
        theta = torch.cat([torch.tensor([1.3], dtype=F64), ls * spread(d)])
        zf = None
    else:
        theta = torch.cat([torch.tensor([1.1, 0.7, 0.9, 1.2, 0.15], dtype=F64), ls * spread(d), 1.5 * ls * spread(d)])
        zf = torch.randn(M, generator=g, dtype=F64)
    m = torch.randn(M, generator=g, dtype=F64)
    Lq = torch.tril(torch.randn(M, M, generator=g, dtype=F64), -1) * 0.05 / math.sqrt(M)
    dg = 0.05 + 0.1 * torch.rand(M, generator=g, dtype=F64)
    dg[::3] = -dg[::3]
    Lq = Lq + torch.diag(dg) + torch.triu(torch.randn(M, M, generator=g, dtype=F64), 1)
    return Zx, zf, theta, m, Lq


def cov_ref(kind, theta, A, B, fa=None, fb=None):
    """k(A, B) in longdouble with explicit coordinate differences (common.cuh, oc_kernel_entry)."""
    th = theta.numpy().astype(LD)
    A, B = A.numpy().astype(LD), B.numpy().astype(LD)
    d = A.shape[1]
    D2 = (A[:, None, :] - B[None, :, :]) ** 2
    if kind == 0:
        return th[0] * np.exp(-0.5 * (D2 / th[1:1 + d] ** 2).sum(-1))
    a1, v, af, lf, a2 = th[:5]
    fa, fb = fa.numpy().astype(LD), fb.numpy().astype(LD)
    E1 = np.exp(-0.5 * (D2 / th[5:5 + d] ** 2).sum(-1))
    E2 = np.exp(-0.5 * (D2 / th[5 + d:5 + 2 * d] ** 2).sum(-1))
    dff = fa[:, None] - fb[None, :]
    return a1 * E1 * (v * np.outer(fa, fb) + af * np.exp(-0.5 * dff * dff / (lf * lf))) + a2 * E2


def cov_torch(kind, theta, A, B, fa=None, fb=None):
    """The same covariance in torch (differentiable in theta and the f columns)."""
    d = A.shape[1]
    D2 = (A[:, None, :] - B[None, :, :]) ** 2
    if kind == 0:
        return theta[0] * torch.exp(-0.5 * (D2 / theta[1:1 + d] ** 2).sum(-1))
    a1, v, af, lf, a2 = theta[0], theta[1], theta[2], theta[3], theta[4]
    E1 = torch.exp(-0.5 * (D2 / theta[5:5 + d] ** 2).sum(-1))
    E2 = torch.exp(-0.5 * (D2 / theta[5 + d:5 + 2 * d] ** 2).sum(-1))
    dff = fa[:, None] - fb[None, :]
    return a1 * E1 * (v * torch.outer(fa, fb) + af * torch.exp(-0.5 * dff * dff / (lf * lf))) + a2 * E2


def p_ref(kind, theta, Zx, zf, jitter):
    return cov_ref(kind, theta, Zx, Zx, zf, zf) + LD(jitter) * np.eye(Zx.shape[0], dtype=LD)


def cond_of(P):
    return float(np.linalg.cond(np.asarray(P, dtype=np.float64)))


def frag_index(MP, i, k):
    """common.cuh frag_offset, vectorised."""
    return ((i >> 4) * (MP >> 2) + (k >> 2)) * 64 + 2 * (4 * (i & 7) + (k & 3)) + ((i >> 3) & 1)


def block_masks(MP):
    i, k = np.meshgrid(np.arange(MP), np.arange(MP), indexing="ij")
    return i, k, (i // 32) >= (k // 32), (i // 32) <= (k // 32)


def written_mask(M):
    """Doubles of an operator buffer that mobo_layer_precompute writes: the seven row-major blocks, the populated block
    triangles of the fragment copies, beta, scal[0..5, 7], the per-CTA KL partials and the flags."""
    lay = F.ops_layout(M)
    MP = lay["MP"]
    mask = torch.zeros(lay["size"], dtype=torch.bool)
    mask[:7 * MP * MP] = True
    i, k, lower, upper = block_masks(MP)
    fo = frag_index(MP, i, k)
    for name, tri in (("WF", lower), ("HF", lower), ("HTF", upper), ("WTF", upper)):
        mask[torch.from_numpy(lay[name] + fo[tri])] = True
    mask[lay["beta"]:lay["beta"] + MP] = True
    mask[lay["scal"]:lay["scal"] + 6] = True
    mask[lay["scal"] + 7] = True
    nb = MP // 32
    mask[lay["rowstat"]:lay["rowstat"] + 4 * (nb * (nb + 1) // 2)] = True
    mask[lay["flags"]:] = True
    return mask


def fill(t, garbage):
    if garbage:
        t.view(torch.int64).fill_(G_BITS)
    else:
        t.zero_()
    return t


def bits(t):
    return t.detach().contiguous().view(torch.int64).cpu()


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


def dev(t):
    return None if t is None else t.to(DEV).contiguous()


def precompute(kind, Zx, zf, theta, m, Lq, jitter, ops):
    lib = _lib.load()
    M, d = Zx.shape
    _lib.check(lib.mobo_layer_precompute(kind, d, M, _lib.ptr(Zx), _lib.ptr(zf), _lib.ptr(theta), _lib.ptr(m),
                                         _lib.ptr(Lq), float(jitter), _lib.ptr(ops), _lib.stream_ptr()),
               "mobo_layer_precompute")
    return ops


def new_ops(M, garbage=True):
    return fill(torch.empty(_lib.load().mobo_ops_doubles(M), dtype=F64, device=DEV), garbage)


def unpack(ops, M):
    lay = F.ops_layout(M)
    MP = lay["MP"]
    o = ops.detach().cpu()
    out = {n: o[lay[n]:lay[n] + MP * MP].view(MP, MP) for n in ("L", "W", "WT", "H", "HT", "P", "LQ")}
    out.update({n: o[lay[n]:lay[n] + MP * MP] for n in ("WF", "HTF", "HF", "WTF")})
    out["beta"] = o[lay["beta"]:lay["beta"] + MP]
    out["scal"] = o[lay["scal"]:lay["scal"] + 16]
    return out


def err_rel(a, ref):
    """max |a - ref| / max |ref| in longdouble."""
    a = np.asarray(a.numpy() if torch.is_tensor(a) else a, dtype=LD)
    ref = np.asarray(ref, dtype=LD)
    return float(np.max(np.abs(a - ref)) / np.max(np.abs(ref)))


RATIOS = {}


def report(family, value, bar):
    """Keeps the worst measured ratio to its bar per check family (printed with -s)."""
    r = value / bar
    if r > RATIOS.get(family, -1.0):
        RATIOS[family] = r
    print("ratio %-12s %.3e (value %.3e, bar %.3e)" % (family, r, value, bar))
    assert value <= bar, (family, value, bar)


def check_structure(o, M, kind, theta, jitter, retries=0):
    """The exact structure the row kernels and the backward rely on, compared by value (-0 == 0)."""
    MP = o["P"].shape[0]
    eye = torch.eye(MP, dtype=F64)
    assert torch.equal(o["WT"], o["W"].T) and torch.equal(o["HT"], o["H"].T)
    i, k, lower, upper = block_masks(MP)
    fo = torch.from_numpy(frag_index(MP, i, k))
    for name, src, tri in (("WF", "W", lower), ("HF", "H", lower), ("HTF", "HT", upper), ("WTF", "WT", upper)):
        t = torch.from_numpy(tri)
        assert torch.equal(o[name][fo[t]], o[src][t]), name
    for name in ("L", "W", "H", "LQ"):
        assert torch.equal(torch.triu(o[name], 1), torch.zeros(MP, MP, dtype=F64)), name
    for name in ("P", "L", "W"):
        assert torch.equal(o[name][M:], eye[M:]) and torch.equal(o[name][:, M:], eye[:, M:]), name
    assert not bool(o["H"][M:].any()) and not bool(o["H"][:, M:].any()) and not bool(o["beta"][M:].any())
    if kind == 0:
        v, prev, p10 = float(theta[0]) + jitter, 0.0, 1.0
        for _ in range(retries):
            jn = 1e-8 * p10
            v += jn - prev
            prev = jn
            p10 *= 10.0
        want = torch.full((M,), v, dtype=F64)
        assert same_bits(o["P"].diagonal()[:M].contiguous(), want), "diag P != a + jitter (+ retries) bit for bit"
    assert float(o["scal"][F.SC_STATUS]) == 0.0 and int(o["scal"][7]) == retries, o["scal"]


def check_lq(o, M, Lq):
    MP = o["P"].shape[0]
    LQ = torch.zeros(MP, MP, dtype=F64)
    LQ[:M, :M] = torch.tril(Lq)
    assert torch.equal(o["LQ"], LQ)


def factor_truth(P):
    """Longdouble factor, inverse, of a matrix (oracle/ld_autodiff)."""
    Lt = LDA._chol(P)
    Wt = LDA._solve_lower(Lt, np.eye(P.shape[0], dtype=LD))
    return Lt, Wt


# ---- 1. forward, block by block ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind,M,d,ls,jitter", FWD_CASES)
def test_forward_block_by_block(kind, M, d, ls, jitter):
    Zx, zf, theta, m, Lq = case_inputs(kind, M, d, ls, seed=1000 * kind + 10 * M + d)
    Pr = p_ref(kind, theta, Zx, zf, jitter)
    cond = cond_of(Pr)
    assert cond <= COND_MAX, cond
    tol = max(1e-10, 20 * EPS * cond)
    ins = [dev(t) for t in (Zx, zf, theta, m, Lq)]
    ops = precompute(kind, *ins, jitter, new_ops(M, garbage=True))
    o = unpack(ops, M)
    check_structure(o, M, kind, theta, jitter)
    check_lq(o, M, Lq)

    P = o["P"][:M, :M].numpy().astype(LD)
    report("P", err_rel(P, Pr), 1e-14)
    Lt, Wt = factor_truth(P)
    Lc = o["L"][:M, :M].numpy().astype(LD)
    report("L", err_rel(Lc, Lt), tol)
    report("L-residual", float(np.max(np.abs(Lc @ Lc.T - P)) / np.max(np.abs(P))), 4 * (M + 1) * EPS)
    LqT = np.tril(Lq.numpy().astype(LD))
    Ht, bt = Wt @ LqT, Wt @ m.numpy().astype(LD)
    report("W", err_rel(o["W"][:M, :M], Wt), tol)
    report("H", err_rel(o["H"][:M, :M], Ht), tol)
    report("beta", err_rel(o["beta"][:M], bt), tol)

    ldp = 2 * np.sum(np.log(np.diagonal(Lt)))
    ldq = np.sum(np.log(np.diagonal(LqT) ** 2))
    b2, h2 = np.sum(bt * bt), np.sum(Ht * Ht)
    kl = 0.5 * (ldp - ldq + b2 + h2 - M)
    for slot, name, val in ((1, "logdetP", ldp), (2, "logdetQ", ldq), (3, "beta2", b2), (4, "H2", h2), (0, "KL", kl)):
        report("KL-pieces", abs(float(o["scal"][slot]) - float(val)) / max(1.0, abs(float(val))), tol)

    # a second call into the same buffer, and a call into a zeroed buffer: bit-identical wherever the call writes
    mask = written_mask(M)
    again = precompute(kind, *ins, jitter, ops.clone())
    zero = precompute(kind, *ins, jitter, new_ops(M, garbage=False))
    first = bits(ops)[mask]
    assert torch.equal(bits(again)[mask], first)
    assert torch.equal(bits(zero)[mask], first)


# ---- 2. retries -------------------------------------------------------------------------------------------------
def retry_inputs(M, d, ls, blk):
    Zx, _, theta, m, Lq = case_inputs(0, M, d, ls, seed=77 + M + blk)
    j = min(32 * blk + 5, M - 1)
    Zx[j] = Zx[j - 3]            # K gets an exactly-zero eigenvalue; the first bad pivot is row j
    return Zx, theta, m, Lq, j


def retry_sequence(P0, retries):
    """P0 (fp64) after each psd_safe_cholesky addition; asserts that exactly `retries` additions are needed."""
    P, prev, p10 = P0.clone(), 0.0, 1.0
    for a in range(4):
        ok = int(torch.linalg.cholesky_ex(P).info) == 0
        assert ok == (a == retries), (a, retries)
        if ok:
            return P
        if a == 3:
            return None
        jn = 1e-8 * p10
        P.diagonal().add_(jn - prev)
        prev, p10 = jn, p10 * 10.0


@pytest.mark.gpu
@pytest.mark.parametrize("M,d,ls,blk,jitter,retries", RETRY_CASES)
def test_retries_at_every_block_position(M, d, ls, blk, jitter, retries):
    Zx, theta, m, Lq, j = retry_inputs(M, d, ls, blk)
    Pl = p_ref(0, theta, Zx, None, jitter)
    P0 = torch.from_numpy(np.asarray(Pl, dtype=np.float64))
    P0.diagonal().copy_(torch.full((M,), float(theta[0]) + jitter, dtype=F64))
    assert int(torch.linalg.cholesky_ex(P0).info) - 1 == j and j // 32 == blk
    assert retry_sequence(P0, retries) is not None
    ops = precompute(0, *[dev(t) for t in (Zx, None, theta, m, Lq)], jitter, new_ops(M))
    o = unpack(ops, M)
    check_structure(o, M, 0, theta, jitter, retries)
    check_lq(o, M, Lq)
    L_o = O.psd_safe_cholesky(P0)
    Lc = o["L"][:M, :M]
    assert err_rel(Lc, L_o.numpy()) < 1e-6
    P = o["P"][:M, :M].numpy().astype(LD)
    Lcl = Lc.numpy().astype(LD)
    report("L-residual", float(np.max(np.abs(Lcl @ Lcl.T - P)) / np.max(np.abs(P))), 4 * (M + 1) * EPS)
    _, Wt = factor_truth(P)
    bar = 20 * EPS * cond_of(P)
    report("retry-W", err_rel(o["W"][:M, :M], Wt), bar)
    report("retry-beta", err_rel(o["beta"][:M], Wt @ m.numpy().astype(LD)), bar)


@pytest.mark.gpu
def test_failed_retries_leave_nothing_behind():
    M, d, ls, blk = 256, 4, 0.2, 3
    Zx, theta, m, Lq, _ = retry_inputs(M, d, ls, blk)
    ins = [dev(t) for t in (Zx, None, theta, m, Lq)]
    ops = precompute(0, *ins, -1e-3, new_ops(M))
    scal = unpack(ops, M)["scal"]
    assert float(scal[F.SC_STATUS]) == 1.0 and int(scal[7]) == 3, scal
    precompute(0, *ins, 1e-6, ops)
    fresh = precompute(0, *ins, 1e-6, new_ops(M))
    check_structure(unpack(fresh, M), M, 0, theta, 1e-6)
    mask = written_mask(M)
    assert torch.equal(bits(ops)[mask], bits(fresh)[mask])


def layer_thetas(sd, L):
    out = []
    for l in range(L):
        h = O.layer_hypers(sd, l)
        if l == 0:
            out.append(torch.cat([h["a"].reshape(1), h["ls"].reshape(-1)]))
        else:
            out.append(torch.cat([h["a1"].reshape(1), h["vlin"].reshape(1), h["af"].reshape(1), h["lsf"].reshape(1),
                                  h["a2"].reshape(1), h["ls1"].reshape(-1), h["ls2"].reshape(-1)]))
    return [t.detach() for t in out]


@pytest.mark.gpu
def test_fused_step_with_different_retries_per_layer():
    """Layer 0 needs two retries and layer 1 none, inside one cooperative launch of the fused step."""
    from mobocmf_b200.fused import FusedELBOStep
    from mobocmf_b200.gp import settings
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    from tests.helpers import model_from_state, random_state, relerr
    M, d, L, S, B, jitter = 40, 2, 2, 2, 24, -5e-8
    sd, noise_upper = random_state(M, d, L, seed=4, ls=0.12)
    Zk = "hidden_layer_0.variational_strategy.inducing_points"
    mk = "hidden_layer_0.variational_strategy._variational_distribution.variational_mean"
    sd[Zk][9] = sd[Zk][4]
    sd[Zk][30] = sd[Zk][17]
    sd[mk][9] = sd[mk][4] + 1.0
    sd[mk][30] = sd[mk][17] - 1.0
    sd["hidden_layer_1.variational_strategy.inducing_points"][:, :d] = sd[Zk]
    th = layer_thetas(sd, L)
    Zx, m0 = sd[Zk], sd[mk]
    conds = []
    for l, want in ((0, 2), (1, 0)):
        zf = None if l == 0 else m0
        P = torch.from_numpy(np.asarray(p_ref(l, th[l], Zx, zf, jitter), dtype=np.float64))
        Pr = retry_sequence(P, want)
        assert Pr is not None
        conds.append(cond_of(Pr))
    tol = max(1e-10, 20 * EPS * max(conds))

    model = model_from_state(sd, noise_upper, L)
    for l in range(L):
        getattr(model, "hidden_layer_%d" % l).variational_strategy.jitter_val = jitter
    N = 60
    elbo = VariationalELBOMF(model, N, L)
    g = torch.Generator().manual_seed(5)
    xb = torch.rand(B, d, generator=g, dtype=F64).to(DEV)
    yb = torch.randn(B, 1, generator=g, dtype=F64).to(DEV)
    fb = torch.randint(0, L, (B, 1), generator=g).double().to(DEV)
    eps = [None] + [torch.randn(B * S, generator=g, dtype=F64).to(DEV) for _ in range(1, L)]
    step = FusedELBOStep(model, elbo)
    loss, kl = step(xb, yb, fb, eps=eps, num_samples=S)
    assert step.retries() == 2
    step.check()
    loss, kl = loss.clone(), kl.clone()
    g_fused = {n: p.grad.clone() for n, p in model.named_parameters() if p.requires_grad}
    for p in model.parameters():
        p.grad = None
    with settings.num_likelihood_samples(1):
        out = model(xb, eps=eps, num_samples=S)
        res = elbo(out, yb.T, fb)
    (-res[0]).backward()
    F.check_status()
    assert relerr(loss, -res[0]) < 1e-12 and relerr(kl, res[1]) < 1e-12, (relerr(loss, -res[0]), relerr(kl, res[1]))
    for n, p in model.named_parameters():
        if not p.requires_grad:
            continue
        gf, gc = g_fused[n], p.grad
        if "chol_variational_covar" in n:
            gf, gc = torch.tril(gf), torch.tril(gc)
        assert relerr(gf, gc) < max(1e-9, 30 * tol), (n, relerr(gf, gc), tol)


# ---- 3. backward against autograd ----------------------------------------------------------------------------------
def bwd_fixture(kind, M, d, ls):
    Zx, zf, theta, m, Lq = case_inputs(kind, M, d, ls, seed=500 + 1000 * kind + 10 * M + d)
    g = torch.Generator().manual_seed(M + d)
    R = 3 * M + 2
    X = torch.rand(R, d, generator=g, dtype=F64)
    fX = torch.randn(R, generator=g, dtype=F64) if kind == 1 else None
    Kr = cov_torch(kind, theta, X, Zx, fX, zf)
    dmu = torch.randn(R, generator=g, dtype=F64)
    dvar = torch.randn(R, generator=g, dtype=F64)
    clamped = torch.rand(R, generator=g) < 0.3
    return Zx, zf, theta, m, Lq, Kr, dmu, dvar, clamped


def bwd_reference(kind, Zx, zf, theta, m, Lq, jitter, Kr, dmu, dvar, clamped, g):
    """torch fp64 autograd of  sum dmu_r k_r^T P^-1 m + sum dvar_r (-[r not clamped] k_r^T P^-1 k_r
    + |tril(L_q)^T P^-1 k_r|^2) + g KL  with the rows k_r fixed."""
    theta = theta.clone().requires_grad_(True)
    zf = zf.clone().requires_grad_(True) if kind == 1 else None
    m = m.clone().requires_grad_(True)
    Lq = Lq.clone().requires_grad_(True)
    M = Zx.shape[0]
    P = cov_torch(kind, theta, Zx, Zx, zf, zf) + jitter * torch.eye(M, dtype=F64)
    Lc = torch.linalg.cholesky(P)
    T = torch.linalg.solve_triangular(Lc, Kr.T, upper=False)
    beta = torch.linalg.solve_triangular(Lc, m[:, None], upper=False)[:, 0]
    Lt = torch.tril(Lq)
    H = torch.linalg.solve_triangular(Lc, Lt, upper=False)
    mu = T.T @ beta
    var = -(T ** 2).sum(0) * (~clamped) + ((H.T @ T) ** 2).sum(0)
    kl = 0.5 * (torch.log(Lc.diagonal() ** 2).sum() - torch.log(Lt.diagonal() ** 2).sum() + (beta ** 2).sum() +
                (H ** 2).sum() - M)
    loss = (dmu * mu).sum() + (dvar * var).sum() + g * kl
    wrt = [theta, m, Lq] + ([zf] if kind == 1 else [])
    gr = torch.autograd.grad(loss, wrt)
    out = {"dtheta": gr[0], "dm": gr[1], "dLq": torch.tril(gr[2])}
    if kind == 1:
        out["dzf"] = gr[3]
    return out


def make_gops(M, T, dmu, dvar, clamped, g, garbage):
    """Gradient buffer: the convention slots (A2, Ac, b, g, clamped-row count; padded entries 0), everything else
    zero or garbage."""
    lay = F.ops_layout(M)
    MP = lay["MP"]
    gops = fill(torch.empty(lay["size"], dtype=F64), garbage)
    A2 = torch.zeros(MP, MP, dtype=F64)
    A2[:M, :M] = (T * dvar) @ T.T
    gops[lay["W"]:lay["W"] + MP * MP] = A2.reshape(-1)
    nclamp = int(clamped.sum())
    if nclamp:
        Ac = torch.zeros(MP, MP, dtype=F64)
        Ac[:M, :M] = (T * (dvar * clamped)) @ T.T
        gops[lay["H"]:lay["H"] + MP * MP] = Ac.reshape(-1)
    b = torch.zeros(MP, dtype=F64)
    b[:M] = T @ dmu
    gops[lay["alpha"]:lay["alpha"] + MP] = b
    gops[lay["scal"] + F.SC_KL] = g
    gops[lay["scal"] + 6] = float(nclamp)
    return gops.to(DEV)


def precompute_bwd(kind, ins, ops, gops, garbage):
    """mobo_layer_precompute_bwd with work and the four outputs zeroed or garbage-filled."""
    lib = _lib.load()
    Zx, zf, theta, m, Lq = ins
    M, d = Zx.shape
    work = fill(torch.empty(lib.mobo_precompute_bwd_work_doubles(M), dtype=F64, device=DEV), garbage)
    out = {"dtheta": fill(torch.empty_like(theta), garbage), "dm": fill(torch.empty_like(m), garbage),
           "dLq": fill(torch.empty_like(Lq), garbage)}
    if kind == 1:
        out["dzf"] = fill(torch.empty_like(zf), garbage)
    _lib.check(lib.mobo_layer_precompute_bwd(kind, d, M, _lib.ptr(Zx), _lib.ptr(zf), _lib.ptr(theta), _lib.ptr(m),
                                             _lib.ptr(Lq), _lib.ptr(ops), _lib.ptr(gops), _lib.ptr(work),
                                             _lib.ptr(out["dtheta"]), _lib.ptr(out.get("dzf")), _lib.ptr(out["dm"]),
                                             _lib.ptr(out["dLq"]), _lib.stream_ptr()), "mobo_layer_precompute_bwd")
    torch.cuda.synchronize()
    return out


# (name, dmu on, dvar on, clamped rows on, g on, outputs that are exactly zero)
BWD_RUNS = [("g", False, False, False, True, ()), ("b", True, False, False, False, ("dLq",)),
            ("A2", False, True, False, False, ("dm",)), ("A2+Ac", False, True, True, False, ("dm",)),
            ("all", True, True, True, True, ())]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,M,d,ls", BWD_CASES)
def test_backward_matches_autograd(kind, M, d, ls):
    jitter = 1e-6
    Zx, zf, theta, m, Lq, Kr, dmu, dvar, clamped = bwd_fixture(kind, M, d, ls)
    P = cov_torch(kind, theta, Zx, Zx, zf, zf) + jitter * torch.eye(M, dtype=F64)
    cond = float(torch.linalg.cond(P))
    assert cond <= COND_MAX, cond
    tol = max(1e-10, 20 * EPS * cond)
    T = torch.linalg.solve_triangular(torch.linalg.cholesky(P), Kr.T, upper=False)     # t_r = W k_r
    ins = [dev(t) for t in (Zx, zf, theta, m, Lq)]
    ops = precompute(kind, *ins, jitter, new_ops(M))
    none = torch.zeros_like(clamped)
    for name, on_mu, on_var, on_clamp, on_g, zeros in BWD_RUNS:
        dmu_r = dmu if on_mu else torch.zeros_like(dmu)
        dvar_r = dvar if on_var else torch.zeros_like(dvar)
        cl = clamped if on_clamp else none
        g = 0.7 if on_g else 0.0
        ref = bwd_reference(kind, Zx, zf, theta, m, Lq, jitter, Kr, dmu_r, dvar_r, cl, g)
        outs = [precompute_bwd(kind, ins, ops, make_gops(M, T, dmu_r, dvar_r, cl, g, gb), gb) for gb in (False, True)]
        for k in outs[0]:
            assert same_bits(outs[0][k], outs[1][k]), (name, k, "garbage in caller memory changed the result")
        got = {k: v.cpu() for k, v in outs[0].items()}
        assert torch.equal(torch.triu(got["dLq"], 1), torch.zeros(M, M, dtype=F64)), name
        for k, r in ref.items():
            c = got[k]
            if k in zeros:
                assert not bool(r.any()) and not bool(c.any()), (name, k)
                continue
            scale = float(r.abs().max())
            assert scale > 0.0, (name, k, "reference gradient is trivial")
            report("bwd-" + k, float((c - r).abs().max()) / scale, 100 * tol)


# ---- 4. caller memory holding NaN ----------------------------------------------------------------------------------
def rows_call(kind, ins, ops, x, xrep, mu_prev, var_prev, prep, eps, eps_mod, R, dmu, dvar, garbage):
    """mobo_layer_rows_fwd then mobo_layer_rows_bwd with Tsave / Usave / work / gops zeroed or garbage-filled."""
    lib = _lib.load()
    Zx, zf, theta, _, _ = ins
    M, d = Zx.shape
    nsave = lib.mobo_rows_save_doubles(M, R)
    Ts = fill(torch.empty(nsave, dtype=F64, device=DEV), garbage)
    Us = fill(torch.empty(nsave, dtype=F64, device=DEV), garbage)
    mu = torch.zeros(R, dtype=F64, device=DEV)
    var = torch.zeros(R, dtype=F64, device=DEV)
    craw = torch.zeros(R, dtype=F64, device=DEV)
    cnt = torch.zeros(1, dtype=torch.int32, device=DEV)
    common = (kind, d, M, _lib.ptr(Zx), _lib.ptr(zf), _lib.ptr(theta), _lib.ptr(ops), _lib.ptr(x), xrep,
              _lib.ptr(mu_prev), _lib.ptr(var_prev), prep, _lib.ptr(eps), eps_mod, None, R, 1)
    _lib.check(lib.mobo_layer_rows_fwd(*common, _lib.ptr(mu), _lib.ptr(var), _lib.ptr(craw), _lib.ptr(cnt),
                                       _lib.ptr(Ts), _lib.ptr(Us), _lib.stream_ptr()), "mobo_layer_rows_fwd")
    gops = fill(torch.empty(lib.mobo_ops_doubles(M), dtype=F64, device=DEV), garbage)
    work = fill(torch.empty(lib.mobo_rows_bwd_work_doubles(M, R), dtype=F64, device=DEV), garbage)
    df = torch.zeros(R, dtype=F64, device=DEV)
    dxrow = torch.zeros(R, d, dtype=F64, device=DEV)
    dtheta = torch.zeros_like(theta)
    dzf = torch.zeros(M, dtype=F64, device=DEV)
    _lib.check(lib.mobo_layer_rows_bwd(*common, _lib.ptr(dmu), _lib.ptr(dvar), _lib.ptr(craw), _lib.ptr(cnt),
                                       _lib.ptr(Ts), _lib.ptr(Us), 1, _lib.ptr(df), _lib.ptr(dxrow), _lib.ptr(dtheta),
                                       _lib.ptr(dzf), _lib.ptr(gops), _lib.ptr(work), _lib.stream_ptr()),
               "mobo_layer_rows_bwd")
    MP = F.ops_layout(M)["MP"]
    return {"mu": mu, "var": var, "craw": craw, "cnt": cnt.double(), "Ts": Ts[:R * MP], "Us": Us[:R * MP], "df": df,
            "dxrow": dxrow, "dtheta": dtheta, "dzf": dzf}, gops


@pytest.mark.gpu
@pytest.mark.parametrize("xrep", [1, 12])
def test_row_pass_ignores_caller_memory(xrep):
    """Generic forward (xrep = 1) and the sample-shared forward (xrep >= 11) of a kind-1 layer, and their backward."""
    kind, M, d = 1, 65, 3
    Zx, zf, theta, m, Lq = case_inputs(kind, M, d, 0.2, seed=4)
    ins = [dev(t) for t in (Zx, zf, theta, m, Lq)]
    ops = precompute(kind, *ins, 1e-6, new_ops(M))
    g = torch.Generator().manual_seed(xrep)
    n = 70 if xrep == 1 else 9
    R = n * xrep
    x = torch.rand(n, d, generator=g, dtype=F64).to(DEV)
    mu_prev = torch.randn(n, generator=g, dtype=F64).to(DEV)
    var_prev = (0.05 + 0.1 * torch.rand(n, generator=g, dtype=F64)).to(DEV)
    eps = torch.randn(xrep if xrep > 1 else R, generator=g, dtype=F64).to(DEV)
    dmu = torch.randn(R, generator=g, dtype=F64).to(DEV)
    dvar = torch.randn(R, generator=g, dtype=F64).to(DEV)
    args = (kind, ins, ops, x, xrep, mu_prev, var_prev, xrep, eps, eps.numel(), R, dmu, dvar)
    (a, ga), (b, gb) = rows_call(*args, garbage=False), rows_call(*args, garbage=True)
    for k in a:
        assert same_bits(a[k], b[k]), k
    lay = F.ops_layout(M)
    MP = lay["MP"]
    conv = torch.zeros(lay["size"], dtype=torch.bool)
    conv[lay["W"]:lay["W"] + MP * MP] = True
    conv[lay["H"]:lay["H"] + MP * MP] = True
    conv[lay["alpha"]:lay["alpha"] + MP] = True
    conv[lay["scal"] + 6] = True
    assert torch.equal(bits(ga)[conv], bits(gb)[conv])
    assert bool((bits(gb)[~conv] == G_BITS).all()), "mobo_layer_rows_bwd wrote outside the gradient-buffer convention"
    assert bool(a["dtheta"].abs().max() > 0) and bool(a["Ts"].abs().max() > 0)


def acq_chain(M, d, fidelity, S, seed):
    chain = []
    Zx = None
    zf = None
    for l in range(fidelity + 1):
        kind = 0 if l == 0 else 1
        Z, _, theta, m, Lq = case_inputs(kind, M, d, 0.25, seed=seed + l)
        Zx = Z if Zx is None else Zx
        ins = [dev(t) for t in (Zx, zf, theta, m, Lq)]
        chain.append((ins[1], ins[2], precompute(kind, *ins, 1e-6, new_ops(M))))
        zf = m
    g = torch.Generator().manual_seed(seed)
    samples = [None] + [torch.randn(S, generator=g, dtype=F64).to(DEV) for _ in range(fidelity)]
    return dev(Zx), chain, samples


@pytest.mark.gpu
@pytest.mark.parametrize("S", [3, 12])
def test_acquisition_chain_ignores_caller_memory(S):
    lib = _lib.load()
    M, d, fidelity, n = 48, 2, 2, 37
    Zx, chain, samples = acq_chain(M, d, fidelity, S, seed=21)
    zf = _lib.ptr_array([c[0] for c in chain])
    th = _lib.ptr_array([c[1] for c in chain])
    ops = _lib.ptr_array([c[2] for c in chain])
    sm = _lib.ptr_array(samples)
    g = torch.Generator().manual_seed(S)
    X = torch.rand(n, d, generator=g, dtype=F64).to(DEV)
    rn = torch.tensor([0.3], dtype=F64, device=DEV)
    d_mu = torch.randn(n, generator=g, dtype=F64).to(DEV)
    d_var = torch.randn(n, generator=g, dtype=F64).to(DEV)
    res = []
    for garbage in (False, True):
        scratch = fill(torch.empty(4 * n * S, dtype=F64, device=DEV), garbage)
        mu = torch.zeros(n, dtype=F64, device=DEV)
        var = torch.zeros(n, dtype=F64, device=DEV)
        _lib.check(lib.mobo_acq_moments(fidelity, d, M, S, n, _lib.ptr(Zx), zf, th, ops, sm, _lib.ptr(rn), 1e-6, 0.1,
                                        _lib.ptr(X), _lib.ptr(mu), _lib.ptr(var), _lib.ptr(scratch),
                                        _lib.stream_ptr()), "mobo_acq_moments")
        work = fill(torch.empty(lib.mobo_acq_bwd_work_doubles(fidelity, d, M, S, n), dtype=F64, device=DEV), garbage)
        dX = torch.zeros(n, d, dtype=F64, device=DEV)
        dn = torch.zeros(1, dtype=F64, device=DEV)
        _lib.check(lib.mobo_acq_moments_bwd(fidelity, d, M, S, n, _lib.ptr(Zx), zf, th, ops, sm, _lib.ptr(rn), 1e-6,
                                            0.1, _lib.ptr(X), _lib.ptr(d_mu), _lib.ptr(d_var), 0, _lib.ptr(dX),
                                            _lib.ptr(dn), _lib.ptr(work), _lib.stream_ptr()), "mobo_acq_moments_bwd")
        res.append((mu, var, dX, dn))
    for a, b in zip(*res):
        assert same_bits(a, b)
    assert bool(res[0][2].abs().max() > 0) and float(res[0][3]) != 0.0


@pytest.mark.gpu
def test_fused_step_ignores_its_workspace():
    """The step's workspace zeroed, NaN-filled, and as a step whose loss was not finite left it: same results."""
    from mobocmf_b200.errors import NanError
    from mobocmf_b200.fused import FusedELBOStep
    from mobocmf_b200.mlls.variational_elbo_mf import VariationalELBOMF
    from tests.helpers import model_from_state, random_state
    M, d, L, S, B = 75, 2, 3, 2, 50
    sd, noise_upper = random_state(M, d, L, seed=8, ls=0.3)
    model = model_from_state(sd, noise_upper, L)
    step = FusedELBOStep(model, VariationalELBOMF(model, 200, L))
    g = torch.Generator().manual_seed(3)
    x = torch.rand(B, d, generator=g, dtype=F64).to(DEV)
    y = torch.randn(B, 1, generator=g, dtype=F64).to(DEV)
    fid = torch.randint(0, L, (B, 1), generator=g).double().to(DEV)
    eps = [None] + [torch.randn(B * S, generator=g, dtype=F64).to(DEV) for _ in range(1, L)]

    def run(y_):
        loss, kl = step(x, y_, fid, eps=eps, num_samples=S)
        torch.cuda.synchronize()
        return [loss.clone(), kl.clone(), step.out[0:8].clone()] + \
               [p.grad.clone() for p in model.parameters() if p.requires_grad]

    fill(step._workspace(B, S), False)
    ref = run(y)
    assert float(ref[2][3]) == 0.0 and float(ref[2][5]) == 0.0
    fill(step._workspace(B, S), True)
    for a, b in zip(ref, run(y)):
        assert same_bits(a, b)
    y_nan = y.clone()
    y_nan[7] = float("nan")
    bad = run(y_nan)
    assert float(bad[2][5]) != 0.0
    with pytest.raises(NanError):
        step.check()
    for a, b in zip(ref, run(y)):
        assert same_bits(a, b)
