"""GPU: egom2p_sample_rows against an fp64 inverse CDF. The reference is oracle/sampling_oracle.py (`kept_mask` for the
filtered set) and the fp64 softmax of the kept logits, summed in ascending token order. Checked:
  * a probe at every step of the CDF between consecutive kept tokens: the float32 u nearest the step and two floats on
    either side, one row each -- the draws an inverse-CDF kernel gets wrong when its fp32 partial sums leave gaps;
  * a stratified sweep u_i = (i + 0.5) / R over vocabularies, filters, temperatures and kinds of logit rows: the token never
    decreases as u grows, is always kept, and the empirical CDF of the draws follows the fp64 CDF;
  * the filter contract (exact counts for top-k, tie groups kept whole), the returned probability, u at both ends, greedy
    and near-greedy temperatures with tied maxima in different chunks, the vocabulary limit;
  * GenerationSampler.sample_from_hidden with a fractional top_k over a row count that is not a multiple of its chunk.

The filtered set of the kernel is the n_kept largest logits, tie groups whole (include/egom2p_b200.h), so the reference
distribution of a draw is built from the n_kept the kernel reports for that row; the filter is checked against the oracle
separately. A draw is correct when the fp64 interval [CDF(tok) - p(tok), CDF(tok)) of the returned token lies within 1e-5
of u: the kernel sums fp32 weights from __expf."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import sampling_oracle as so  # noqa: E402

TOL_U = 1e-5          # fp32 partial sums and __expf, as a distance in u
PROB_RTOL = 5e-5      # |arg| <= 87 of __expf times a few fp32 roundings of the argument
PROB_ATOL = 1e-38     # below FLT_MIN a weight is subnormal (or flushed) in fp32
R = 65536             # draws per sweep configuration
CHUNK = 4096          # tokens per chunk of the kernel's draw (1024 threads x 4)


@pytest.fixture(scope="module")
def ops():
    from egom2p_b200 import ops as o
    return o


def _normal(V, sigma, seed):
    return (np.random.default_rng(seed).standard_normal(V) * sigma).astype(np.float32)


def _kernel_keep(x, n):
    """The n largest logits of x. The kernel keeps a value prefix and never splits a group of equal logits."""
    keep = x >= np.sort(x)[::-1][n - 1]
    assert keep.sum() == n, f"n_kept = {n} splits the tie group at {np.sort(x)[::-1][n - 1]} ({int(keep.sum())} >= it)"
    return keep


def _check_filter(x, top_k, top_p, n):
    """n_kept against the oracle: exact with no filter or top-k only (the count search is exact); with top-p, either
    a superset of the oracle's stable-sort set that adds only members of the tie group straddling top_p, or, without
    such a group, +-1 (the mass threshold is compared in fp32). Returns the kernel's filtered set."""
    want = so.kept_mask(x[None], top_k, top_p)[0]
    keep = _kernel_keep(x, n)
    if top_p == 0.0:
        assert n == int(want.sum()), (n, int(want.sum()))
        return keep
    group = x == x[want].min()
    if want[group].sum() < group.sum():
        assert not (want & ~keep).any(), "a token the oracle keeps was removed"
        assert group[keep & ~want].all(), "tokens outside the straddling tie group were added"
    else:
        assert abs(n - int(want.sum())) <= 1, (n, int(want.sum()))
    return keep


class _Ref:
    """fp64 reference for the filtered sets a launch reported. Rows of one launch may report different n_kept for the
    same logits: the top-p mass sums use float atomics, and top_p * Z can sit within their rounding of a token's step.
    Every distinct n_kept is checked against the oracle and gets its own distribution."""

    def __init__(self, x, temp, top_k, top_p, n_kept):
        self.ns, self.gid = np.unique(n_kept, return_inverse=True)
        self.keep = np.stack([_check_filter(x, top_k, top_p, int(n)) for n in self.ns])
        z = np.where(self.keep, x.astype(np.float64)[None] / float(np.float32(temp)), -np.inf)
        e = np.exp(z - z.max(1, keepdims=True))
        self.p = e / e.sum(1, keepdims=True)
        self.cdf = np.cumsum(self.p, 1)

    def check_draws(self, u, tok, prob):
        """u float64 (rows,): every token kept, its fp64 interval within TOL_U of u, prob its fp64 probability."""
        g = self.gid
        assert self.keep[g, tok].all(), f"filtered-out tokens drawn: {np.unique(tok[~self.keep[g, tok]])[:10]}"
        hi = self.cdf[g, tok]
        lo = hi - self.p[g, tok]
        off = np.maximum(np.maximum(lo - u, u - hi), 0.0)
        bad = np.nonzero(off > TOL_U)[0]
        if bad.size:
            want = np.array([np.searchsorted(self.cdf[g[i]], u[i], side="right") for i in bad[:8]])
            last_in_chunk = [int(np.nonzero(self.keep[g[i], :(t // CHUNK + 1) * CHUNK])[0][-1]) == t for i, t in zip(bad, tok[bad])]
            raise AssertionError(f"{bad.size} of {u.size} draws land more than {TOL_U} from the returned token's CDF interval; "
                                 f"{sum(last_in_chunk)} of them returned the last kept token of a {CHUNK}-token chunk. First: "
                                 f"u {u[bad[:8]].tolist()}, token {tok[bad[:8]].tolist()}, fp64 inverse CDF {want.tolist()}, "
                                 f"off by {off[bad[:8]].tolist()}")
        np.testing.assert_allclose(prob, self.p[g, tok], rtol=PROB_RTOL, atol=PROB_ATOL)


def _draw(ops, row, temp, top_p, top_k, u):
    """One draw per uniform: the device row (1, V), row pitch 0, one kernel row per u."""
    ud = torch.from_numpy(np.asarray(u, np.float32)).cuda()
    tok, prob, kept = ops.sample_rows(row.expand(ud.numel(), row.shape[1]), temp, top_p, top_k, ud, want_kept=True)
    return tok.cpu().numpy(), prob.cpu().numpy(), kept.cpu().numpy()


# ----------------------------------------------------------------------------------------------- CDF step probe
@pytest.mark.parametrize("V, top_p", [(64000, 0.0), (256, 0.0), (4096, 0.0), (64000, 0.8)],
                         ids=["V64000", "V256", "V4096", "V64000-p0.8"])
def test_every_cdf_step_probed(ops, V, top_p):
    x = _normal(V, 2.0, 100 + V)
    row = torch.from_numpy(x).cuda()[None]
    ref = _Ref(x, 1.0, 0, top_p, _draw(ops, row, 1.0, top_p, 0, [0.5])[2])
    steps = ref.cdf[0][ref.keep[0]][:-1].astype(np.float32)
    probes = [steps]
    up, down = steps, steps
    for _ in range(2):
        up, down = np.nextafter(up, np.float32(1)), np.nextafter(down, np.float32(0))
        probes += [up, down]
    u = np.unique(np.concatenate(probes))
    u = u[(u >= 0) & (u < 1)]
    tok, prob, kept = _draw(ops, row, 1.0, top_p, 0, u)
    _Ref(x, 1.0, 0, top_p, kept).check_draws(u.astype(np.float64), tok, prob)


# ----------------------------------------------------------------------------------------------- stratified sweep
VOCABS = (8, 256, 4096, 4099, 64000, 65536)   # 4099: a column slice of a width-4100 buffer (scalar tail, 3-token chunk)
FILTERS = {"none": (0, 0.0), "k1": (1, 0.0), "k50": (50, 0.0), "kVm1": (None, 0.0),
           "p0.05": (0, 0.05), "p0.8": (0, 0.8), "p0.95": (0, 0.95), "k50-p0.8": (50, 0.8)}
TEMPS = (0.01, 0.7, 1.0, 3.0)
ROWS = ("normal0.5", "normal2", "normal4", "spike", "constant")
# every vocabulary with every filter; temperatures and row kinds rotate so that each vocabulary and each filter meets every
# temperature and every kind of row
SWEEP = [(V, f, TEMPS[(i + j) % len(TEMPS)], ROWS[(i + 2 * j) % len(ROWS)])
         for i, V in enumerate(VOCABS) for j, f in enumerate(FILTERS)]


def _row(kind, V, seed):
    if kind == "constant":
        return np.full(V, 0.25, np.float32)
    if kind == "spike":
        x = _normal(V, 1.0, seed)
        x[np.random.default_rng(seed + 1).integers(V)] += 30.0
        return x
    return _normal(V, float(kind[len("normal"):]), seed)


@pytest.mark.parametrize("V, filt, temp, kind", SWEEP, ids=[f"V{V}-{f}-T{t}-{k}" for V, f, t, k in SWEEP])
def test_stratified_sweep_is_the_inverse_cdf(ops, V, filt, temp, kind):
    top_k, top_p = FILTERS[filt]
    top_k = V - 1 if top_k is None else top_k
    x = _row(kind, V, SWEEP.index((V, filt, temp, kind)))
    if V == 4099:   # real pitch 4100; the column past the slice holds a logit that would win every draw if it were read
        buf = torch.from_numpy(np.append(x, np.float32(x.max() + 100))).cuda()[None].expand(R, V + 1).contiguous()
        lg = buf[:, :V]
    else:
        lg = torch.from_numpy(x).cuda()[None].expand(R, V)
    u = ((np.arange(R) + 0.5) / R).astype(np.float32)
    tok, prob, kept = ops.sample_rows(lg, temp, top_p, top_k, torch.from_numpy(u).cuda(), want_kept=True)
    tok, prob, kept = tok.cpu().numpy(), prob.cpu().numpy(), kept.cpu().numpy()
    ref = _Ref(x, temp, top_k, top_p, kept)
    assert (np.diff(tok) >= 0).all(), f"token decreases at u = {u[1:][np.diff(tok) < 0][:5]}"
    ref.check_draws(u.astype(np.float64), tok, prob)
    # empirical CDF of the draws against the fp64 CDF of the majority's filtered set; rows with another set (see _Ref)
    # move it by at most the largest gap between the two CDFs
    major = np.bincount(ref.gid).argmax()
    spread = np.abs(ref.cdf - ref.cdf[major]).max()
    emp = np.cumsum(np.bincount(tok, minlength=V)) / R
    assert np.abs(emp - ref.cdf[major]).max() <= 1.0 / R + TOL_U + spread


# ----------------------------------------------------------------------------------------------- filter contract
@pytest.mark.parametrize("k_in_group", [1, 500, 1000])
def test_top_k_keeps_the_whole_tie_group(ops, k_in_group):
    """1000 tokens share one logit (dead codebook rows do); k ends at the group's first, middle or last member."""
    V, c = 64000, np.float32(3.0)
    x = _normal(V, 1.0, 7)
    rng = np.random.default_rng(8)
    x[rng.choice(V, 1000, replace=False)] = c
    n_above = int((x > c).sum())
    row = torch.from_numpy(x).cuda()[None]
    for top_p in (0.0, 0.999):
        tok, prob, kept = _draw(ops, row, 1.0, top_p, n_above + k_in_group, [0.0, 0.5, 0.999])
        if top_p == 0.0:
            assert (kept == n_above + 1000).all(), kept
        assert (_kernel_keep(x, int(kept[0])) >= (x >= c)).all()
        _Ref(x, 1.0, n_above + k_in_group, top_p, kept).check_draws(np.array([0.0, 0.5, 0.999]), tok, prob)


def test_top_p_keeps_the_whole_straddling_tie_group(ops):
    """top_p lands in the middle of a group of 1000 equal logits: the oracle's stable sort keeps its lower-index part, the
    kernel keeps all of it and nothing below it."""
    V, c = 64000, np.float32(2.0)
    x = _normal(V, 1.0, 9)
    x[np.random.default_rng(10).choice(V, 1000, replace=False)] = c
    e = np.exp(x.astype(np.float64) - x.max())
    e /= e.sum()
    above, group = e[x > c].sum(), e[x == c].sum()
    top_p = float(np.float32(above + 0.5 * group))
    want = so.kept_mask(x[None], 0.0, top_p)[0]
    assert 0 < want[x == c].sum() < 1000
    u = np.linspace(0.0, 0.999, 64)
    tok, prob, kept = _draw(ops, torch.from_numpy(x).cuda()[None], 1.0, top_p, 0, u)
    assert (kept == int((x >= c).sum())).all(), kept
    ref = _Ref(x, 1.0, 0, top_p, kept)
    assert (ref.keep[0] == (x >= c)).all()
    ref.check_draws(u, tok, prob)


# ----------------------------------------------------------------------------------------------- ends of u, temperature
@pytest.mark.parametrize("V, sigma, temp, top_k, top_p, raise_to", [
    (64000, 2.0, 1.0, 0, 0.0, {63999: -1.0}),
    (64000, 1.0, 0.01, 0, 0.0, {777: 2.0, 63000: 2.0}),     # every other weight underflows to 0
    (64000, 1.0, 0.01, 50, 0.8, {777: 2.0, 63000: 2.0}),    # ... including kept ones
    (4099, 1.0, 0.7, 0, 0.95, {4098: -0.5}),                # the last token sits in a 3-token chunk
    (65536, 2.0, 3.0, 50, 0.0, {})])
def test_u_at_both_ends(ops, V, sigma, temp, top_k, top_p, raise_to):
    """u = 0 returns the first kept token with nonzero fp32 weight, u = nextafter(1, 0) the last one. The rows are built so
    that the last one holds more than 1e-5 of the mass (else the fp64 inverse CDF at 1 - 2^-24 is an earlier token) and no
    kept weight is near the underflow of __expf (argument between -105 and -86)."""
    x = _normal(V, sigma, 11 + V)
    top = x.max()
    for i, d in raise_to.items():
        x[i] = top + d
    u = np.array([0.0, np.nextafter(np.float32(1), np.float32(0))], np.float32)
    tok, prob, kept = _draw(ops, torch.from_numpy(x).cuda()[None], temp, top_p, top_k, u)
    ref = _Ref(x, temp, top_k, top_p, kept)
    arg = (x.astype(np.float64) - x.max()) / float(np.float32(temp))
    for i in range(2):
        keep = ref.keep[ref.gid[i]]
        assert not (keep & (arg > -105.0) & (arg <= -86.0)).any()
        weighted = np.nonzero(keep & (arg > -86.0))[0]
        assert ref.p[ref.gid[i], weighted[-1]] > 1e-5
        assert tok[i] == weighted[0 if i == 0 else -1], (u[i], tok[i], weighted[[0, -1]])
    ref.check_draws(u.astype(np.float64), tok, prob)


def _tied_maxima_row():
    x = _normal(64000, 3.0, 12)
    x[100] = x[60000] = x.max() + 1.0          # chunks 0 and 14
    return torch.from_numpy(x).cuda()[None]


@pytest.mark.parametrize("temp", [0.0, 1e-11])
def test_greedy_returns_the_first_of_tied_maxima(ops, temp):
    row = _tied_maxima_row()
    u = [0.0, 0.3, 0.7, 0.99]
    for top_k, top_p in ((0, 0.0), (50, 0.8)):
        tok, prob, kept = _draw(ops, row, temp, top_p, top_k, u)
        assert (tok == 100).all() and (prob == 1.0).all() and (kept == 1).all(), (tok, prob, kept)


def test_tiny_temperature_draws_between_tied_maxima(ops):
    """T = 1e-9 is above the greedy cut (1e-10): the two maxima have weight 1, everything else 0."""
    u = [0.0, 0.25, 0.4999, 0.5001, 0.75, float(np.nextafter(np.float32(1), np.float32(0)))]
    tok, prob, kept = _draw(ops, _tied_maxima_row(), 1e-9, 0.0, 0, u)
    assert tok.tolist() == [100, 100, 100, 60000, 60000, 60000]
    assert (prob == 0.5).all() and (kept == 64000).all()


def test_vocabulary_above_65536_is_rejected(ops):
    lg = torch.zeros(1, 65540, device="cuda")[:, :65537]     # ld % 4 == 0: only the vocabulary is out of range
    with pytest.raises(RuntimeError, match="vocabulary 65537 exceeds 65536"):
        ops.sample_rows(lg, 1.0)


# ----------------------------------------------------------------------------------------------- sampler glue
class _Head:
    """The one model method GenerationSampler.sample_from_hidden calls."""

    def __init__(self, wb):
        self.wb = wb

    def head_operand(self, mod):
        return self.wb


@pytest.mark.parametrize("temp, top_k, top_p", [(1.0, 0.1, 0.0), (0.7, 0.1, 0.8)])
def test_sample_from_hidden_fractional_top_k_over_ragged_chunks(temp, top_k, top_p):
    """top_k = 0.1 means int(0.1 * V) tokens; the rows span two full chunks and three more. Compared with the oracle on fp64
    head logits from the same bf16 operands: the fp32 GEMM moves the CDF steps, so draws within 1e-4 of a step are skipped.
    The logits have scale 3, where the other 90 % of the tokens hold about 4 % of the mass."""
    from egom2p_b200.generate import GenerationSampler
    V, D = 64000, 768
    g = torch.Generator().manual_seed(13)
    w = (torch.randn(V, D, generator=g) * (3.0 / D ** 0.5)).bfloat16().cuda()
    s = GenerationSampler(_Head(w))
    chunk = s.LOGIT_CHUNK_BYTES // (4 * V)
    rows = 2 * chunk + 3
    yb = torch.randn(rows, D, generator=g).bfloat16().cuda()
    torch.cuda.manual_seed(14)
    tok, prob = s.sample_from_hidden(yb, "tok_depth", temp, top_k, top_p)
    torch.cuda.manual_seed(14)
    u = torch.rand(rows, device="cuda", dtype=torch.float32).cpu().numpy().astype(np.float64)   # the sampler's uniforms
    lg = (yb.double() @ w.double().t()).cpu().numpy()
    want_tok, want_prob, margin = so.draw(lg, float(np.float32(temp)), u, top_k, top_p)
    tok, prob = tok.cpu().numpy(), prob.cpu().numpy()
    assert tok.shape == (rows,)
    solid = margin > 1e-4
    assert solid.mean() > 0.5
    assert np.array_equal(tok[solid], want_tok[solid]), np.nonzero(tok[solid] != want_tok[solid])[0][:10]
    np.testing.assert_allclose(prob[solid], want_prob[solid], rtol=1e-3)
