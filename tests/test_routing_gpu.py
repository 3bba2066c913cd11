"""GPU: the integer kernels that decide which token goes where, checked exactly against the oracle.

- egom2p_index_plan (csrc/plan.cu): slots, pads, modality ids, target ids and decoder key ranges under every decoder mask
  option, at lengths and budgets where the block scans run several times and the partition truncates a modality;
- egom2p_plan_rows (csrc/plan.cu): the row lists of the vocabulary heads;
- EgoM2P._pack_plan: the packed view of a plan (valid slots only, sample after sample);
- egom2p_embed_gather_fwd / _bwd (csrc/embed.cu), dense and packed: the forward bit for bit against torch fp32 in the kernel's
  operation order, the backward against fp64 index_add_ within the error bound of fp32 summation in any order;
- egom2p_gather_rows_bf16 / egom2p_scatter_rows_f32 (csrc/elementwise.cu) bit for bit against index_select / index_copy_;
- the input checks of their Python wrappers.

Everything except the backward sums is integer routing or a copy, so every comparison but those is exact."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import egom2p_oracle as orc  # noqa: E402
import synth  # noqa: E402

f64, bf16 = torch.float64, torch.bfloat16
# Concatenated lengths L > 2048 and not a multiple of 1024, so the 1024-thread block scans of the plan run three times;
# 8 modalities is EGOM2P_MAX_MODS.
LENS = {1: [2563], 4: [30, 1500, 7, 900], 8: [30, 517, 5, 1200, 64, 333, 1, 700]}
EGOB = ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"]
EGOB_DEC_ORDER = ["tok_rgb", "tok_gaze", "tok_depth", "tok_cam"]
DEV = "cuda"


@pytest.fixture(scope="module")
def ops():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from egom2p_b200 import ops as _ops
    return _ops


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


# ------------------------------------------------------------------------------------------------ batches
class Case:
    """One batch of n modalities in concatenation order: masks (True = not a token of this side), the reference's
    decoder_attention_mask (the modality's token count at its lowest token position), token ids."""

    def __init__(self, masks, vocabs, seed):
        rng = np.random.default_rng(seed)
        self.masks = masks
        self.B = masks[0].shape[0]
        self.lens = [m.shape[1] for m in masks]
        self.vocabs = vocabs
        self.mod_ids = [100 + 37 * i for i in range(len(masks))]
        self.off = np.concatenate([[0], np.cumsum(self.lens)])
        self.L = int(self.off[-1])
        self.cnts = []
        for m in masks:
            c = np.zeros(m.shape, np.int32)
            for b in range(self.B):
                w = np.flatnonzero(~m[b])
                if len(w):
                    c[b, w[0]] = len(w)
            self.cnts.append(c)
        self.ids = [rng.integers(0, v, size=m.shape, dtype=np.int64) for m, v in zip(masks, vocabs)]

    def names(self):
        return [f"m{i}" for i in range(len(self.masks))]

    def valid_counts(self):
        """(B, n) tokens of every modality in every sample."""
        return np.stack([(~m).sum(1) for m in self.masks], 1)


def _ragged_masks(lens, B, seed):
    """Sample 0 has no token, sample 1 has every position; in sample 2 modality 1 (or 0 when alone) is empty while the
    others are not; the rest draw a random density per modality."""
    rng = np.random.default_rng(seed)
    masks = []
    for i, L in enumerate(lens):
        m = np.ones((B, L), dtype=bool)
        m[1] = False
        for b in range(2, B):
            if b == 2 and i == min(1, len(lens) - 1):
                continue
            n = int(rng.integers(1, L + 1)) if b != 2 else max(1, L // 3)
            m[b, rng.permutation(L)[:n]] = False
        masks.append(m)
    return masks


def _budgets(case):
    """1; below sample 3's token count (its partition truncates inside a modality); exactly that count; between it and L; L."""
    n3 = int(case.valid_counts()[3].sum())
    assert 40 < n3 < case.L
    return [1, n3 - 37, n3, (n3 + case.L) // 2, case.L]


# ------------------------------------------------------------------------------------------------ 1. index plan
def _run_plan(ops, case, budget, decoder, causal=False, sep=True):
    B = case.B
    if not decoder:
        return ops.index_plan([_cuda(m) for m in case.masks], case.mod_ids, budget)
    return ops.index_plan([_cuda(m) for m in case.masks], case.mod_ids, budget, decoder=True,
                          attn_cnt=[_cuda(c) for c in case.cnts], ids=[_cuda(t.reshape(B, -1)) for t in case.ids],
                          causal=causal, sep=sep)


def _oracle_plan(case, budget, decoder, causal=False, sep=True):
    names = case.names()
    mids = dict(zip(names, case.mod_ids))
    if not decoder:
        return orc.plan_encoder(dict(zip(names, case.masks)), mids, budget)
    return orc.plan_decoder(dict(zip(names, case.masks)), dict(zip(names, case.cnts)), dict(zip(names, case.ids)), mids,
                            names, budget, causal=causal, sep=sep)


def _slot_mod_pos(case, ids_keep):
    """(modality, position inside it) of every slot, from the oracle's concatenated index."""
    m = np.searchsorted(case.off[1:], ids_keep, side="right")
    return m, ids_keep - case.off[m]


def _dense_ranges(attn, rows):
    """[lo, hi) of every row of a dense (B, M, M) mask (True = masked), -1 where the row is fully masked; asserts that the
    visible keys of every selected row are one contiguous range, which is what the kernel's (key_lo, key_hi) can express."""
    ok = ~attn
    M = ok.shape[2]
    some = ok.any(2)
    lo = np.where(some, ok.argmax(2), -1)
    hi = np.where(some, M - ok[:, :, ::-1].argmax(2), -1)
    sel = some & rows
    assert np.array_equal(ok.sum(2)[sel], (hi - lo)[sel]), "the oracle's mask is not one key range per row"
    return lo, hi, sel


def _check_plan(ops, case, budget, decoder, causal=False, sep=True):
    pl = _run_plan(ops, case, budget, decoder, causal, sep)
    o = _oracle_plan(case, budget, decoder, causal, sep)
    what = f"budget {budget} decoder={decoder} causal={causal} sep={sep}"
    keep = o["ids_keep"]
    assert np.array_equal(pl.keep_idx.cpu().numpy(), keep), what
    assert np.array_equal(pl.pad.cpu().numpy(), o["mask"]), what
    assert np.array_equal(pl.mod_mask.cpu().numpy(), o["mod_mask"]), what
    assert np.array_equal(pl.n_valid.cpu().numpy(), (~o["mask"]).sum(1)), what
    # the two outputs the embedding kernels read, on every slot (pass 3 also reads keep_mod on pad slots)
    m_ref, p_ref = _slot_mod_pos(case, keep)
    assert np.array_equal(pl.keep_mod.cpu().numpy(), m_ref), what
    assert np.array_equal(pl.keep_pos.cpu().numpy(), p_ref), what
    if not decoder:
        return pl, o
    assert np.array_equal(pl.target_ids.cpu().numpy(), o["target_ids"]), what
    lo, hi = pl.key_lo.cpu().numpy(), pl.key_hi.cpu().numpy()
    assert ((0 <= lo) & (lo <= hi) & (hi <= budget)).all(), what
    if causal and sep:
        # The reference lets a pad row of modality m also see the earlier pad columns of m (its mask compares modality ids
        # before pads become -1); the kernel gives a pad row the causal range cut to m's segment of valid slots, so no row
        # attends a pad key. No loss or logit of a valid row depends on a pad row (DESIGN.md section 3).
        pad = o["mask"]
        nv = case.valid_counts()
        seg_hi = np.minimum(np.cumsum(nv, 1), budget)
        seg_lo = np.concatenate([np.zeros((case.B, 1), nv.dtype), seg_hi[:, :-1]], 1)
        s = np.broadcast_to(np.arange(budget), lo.shape)
        p_lo = np.take_along_axis(seg_lo, m_ref, 1)
        p_hi = np.maximum(np.minimum(s + 1, np.take_along_axis(seg_hi, m_ref, 1)), p_lo)
        assert np.array_equal(lo[pad], p_lo[pad]) and np.array_equal(hi[pad], p_hi[pad]), what
        rows = ~pad
    else:
        rows = np.ones(lo.shape, dtype=bool)
    j = np.arange(budget)[None, None, :]
    dense = ~((j >= lo[:, :, None]) & (j < hi[:, :, None]))
    assert np.array_equal(dense[rows], o["attn_mask"][rows]), what
    # and the range itself, wherever it is not empty (an empty range may sit anywhere)
    r_lo, r_hi, nonempty = _dense_ranges(o["attn_mask"], rows)
    assert np.array_equal(lo[nonempty], r_lo[nonempty]) and np.array_equal(hi[nonempty], r_hi[nonempty]), what
    return pl, o


@pytest.mark.parametrize("n_mods", [1, 4, 8])
def test_index_plan_encoder_exact(ops, n_mods):
    case = Case(_ragged_masks(LENS[n_mods], 6, seed=n_mods), [97] * n_mods, seed=n_mods)
    for budget in _budgets(case):
        _check_plan(ops, case, budget, decoder=False)


@pytest.mark.parametrize("causal,sep", [(False, True), (False, False), (True, True), (True, False)])
@pytest.mark.parametrize("n_mods", [1, 4, 8])
def test_index_plan_decoder_exact(ops, n_mods, causal, sep):
    case = Case(_ragged_masks(LENS[n_mods], 6, seed=10 + n_mods), [97] * n_mods, seed=10 + n_mods)
    budgets = _budgets(case)
    assert max(budgets[1:4]) > 1024                 # pass 3's cumsum runs several block scans
    for budget in budgets:
        _check_plan(ops, case, budget, decoder=True, causal=causal, sep=sep)


def _egob_case(B, seed, dec):
    """ego-b geometry (lengths 30 / 5120 / 30 / 5120) with synth.make_batch masks: per sample and modality an input and a
    target count, some of them 0 and some the whole modality."""
    cfg = synth.make_cfg(12, 1, 0, 0, EGOB, video_vocab=64000)
    rng = np.random.default_rng(seed)
    n_in, n_tg = {}, {}
    for m, inf in cfg["mods"].items():
        L = inf["len"]
        n_in[m] = [int(x) for x in rng.integers(0, L // 3 + 1, B)]
        n_tg[m] = [int(x) for x in rng.integers(0, L - L // 3 + 1, B)]
        n_in[m][0] = n_tg[m][0] = 0
        n_in[m][1] = L // 3
        n_tg[m][1] = L - L // 3
    md = synth.make_batch(cfg, B=B, seed=seed, n_in=n_in, n_tgt=n_tg)
    order = EGOB_DEC_ORDER if dec else EGOB
    key = "target_mask" if dec else "input_mask"
    case = Case([md[m][key].numpy() for m in order], [cfg["mods"][m]["vocab"] for m in order], seed)
    case.mod_ids = [synth.MOD_IDS[m] for m in order]
    case.cnts = [md[m]["decoder_attention_mask"].numpy() for m in order]
    case.ids = [md[m]["tensor"].reshape(B, -1).numpy() for m in order]
    return case


def test_index_plan_egob_geometry(ops):
    enc = _egob_case(32, 5, dec=False)
    _check_plan(ops, enc, 2048, decoder=False)
    dec = _egob_case(32, 5, dec=True)
    assert (dec.valid_counts().sum(1) > 2048).any() and (dec.valid_counts().sum(1) < 2048).any()
    for causal in (False, True):
        for sep in (True, False):
            _check_plan(ops, dec, 2048, decoder=True, causal=causal, sep=sep)


# ------------------------------------------------------------------------------------------------ 2. head row lists
def _mod_mask(total, kind, ids, seed):
    rng = np.random.default_rng(seed)
    if kind == "all_pad":
        return np.full(total, -1, np.int16)
    if kind == "one_id":                            # ids[0] on every row
        return np.full(total, ids[0], np.int16)
    # every id but the last (absent: count 0), and pads; the first row holds ids[0]
    mm = rng.choice(np.array(list(ids[:-1]) + [-1], np.int16), size=total)
    mm[0] = ids[0]
    return mm


@pytest.mark.parametrize("kind", ["mixed", "all_pad", "one_id"])
@pytest.mark.parametrize("total", [1, 1023, 1025, 65536])
def test_plan_rows_exact(ops, total, kind):
    ids = [6323, 349, 26680, 7613, 5, 1200, 31000, 77]
    mm = _mod_mask(total, kind, ids, seed=total)
    rows, counts = ops.plan_rows(_cuda(mm).reshape(-1, 1 if total < 2048 else 2048), ids)
    rows, counts = rows.cpu().numpy(), counts.cpu().numpy()
    for m, i in enumerate(ids):
        ref = np.flatnonzero(mm == i)
        assert counts[m] == len(ref), (m, i)
        assert np.array_equal(rows[m, :counts[m]], ref), (m, i)
    if kind == "mixed":
        assert counts[-1] == 0 and (counts[:-1] > 0).sum() >= min(total, 2)


# ------------------------------------------------------------------------------------------------ 3. packed plans
def _pack(plan):
    from egom2p_b200.model import EgoM2P
    nv = plan.n_valid.tolist()
    return EgoM2P._pack_plan(plan, nv, plan.budget) + (nv,)


@pytest.mark.parametrize("decoder", [False, True])
def test_pack_plan_exact(ops, decoder):
    case = Case(_ragged_masks(LENS[4], 6, seed=3), [97] * 4, seed=3)
    pl = _run_plan(ops, case, 997, decoder, causal=True, sep=True)
    pp, off, lens, nv = _pack(pl)
    assert nv[0] == 0 and nv[1] == 997
    R, M, B = sum(nv), pl.budget, case.B
    assert pp.rows == R and pp.B == B and pp.budget == M
    assert lens.tolist() == nv and off.tolist() == list(np.cumsum([0] + nv[:-1]))
    rb = pp.row_batch.cpu().numpy()
    assert rb.dtype == np.int32 and (np.diff(rb) >= 0).all()
    assert np.array_equal(np.bincount(rb, minlength=B), nv)
    names = ["keep_mod", "keep_pos", "mod_mask"] + (["key_lo", "key_hi"] if decoder else [])
    dense = {k: getattr(pl, k).cpu().numpy() for k in names}
    packed = {k: getattr(pp, k).cpu().numpy() for k in names}
    for b in range(B):
        o = int(off[b])
        for k in names:
            assert np.array_equal(packed[k][o:o + nv[b]], dense[k][b, :nv[b]]), (k, b)
    assert not pp.pad.any()
    slot = pp.slot_index.cpu().numpy()
    assert np.array_equal(slot, np.concatenate([b * M + np.arange(n) for b, n in enumerate(nv)]))
    s2r = pp.slot_to_row.cpu().numpy()
    assert np.array_equal(s2r[slot], np.arange(R))
    rest = np.ones(B * M, dtype=bool)
    rest[slot] = False
    assert (s2r[rest] == -1).all()


# ------------------------------------------------------------------------------------------------ 4./5. embedding gather
class Tables:
    """Random fp32 tables of one side: token tables (vocab, D), positions (len, D), modality embeddings (D), mask token."""

    def __init__(self, case, D, seed):
        g = torch.Generator(device=DEV).manual_seed(seed)
        r = lambda *s: torch.randn(*s, device=DEV, generator=g)
        self.D = D
        self.tok = [r(v, D) for v in case.vocabs]
        self.pos = [r(L, D) for L in case.lens]
        self.mod = [r(D) for _ in case.lens]
        self.mask_token = r(D)
        self.ids = [_cuda(t) for t in case.ids]


def _slot_rows(case, o, pp=None):
    """Host description of every row of the dense layout, or of the packed plan `pp`: (valid, sample, modality, position),
    from the oracle's plan only."""
    B, M = o["ids_keep"].shape
    m, p = _slot_mod_pos(case, o["ids_keep"])
    valid = ~o["mask"].reshape(-1)
    b = np.repeat(np.arange(B), M)
    m, p = m.reshape(-1), p.reshape(-1)
    if pp is not None:
        s = pp.slot_index.cpu().numpy()
        valid, b, m, p = valid[s], b[s], m[s], p[s]
        assert valid.all()
    return valid, b, m, p


def _embed_ref(case, tabs, rows, decoder):
    """x0 / emb in fp32 in the kernel's (and the reference's) order: emb = pos + mod; x0 = tok + emb, or
    (0 + mask_token) + emb for the decoder; pad rows 0."""
    valid, b, m, p = rows
    D = tabs.D
    x0 = torch.zeros(len(valid), D, device=DEV)
    emb = torch.zeros_like(x0)
    for k in range(len(case.lens)):
        sel = np.flatnonzero(valid & (m == k))
        if not len(sel):
            continue
        sel_t, pk = _cuda(sel), _cuda(p[sel])
        e = tabs.pos[k][pk] + tabs.mod[k]
        if decoder:
            t = torch.zeros_like(e) + tabs.mask_token
        else:
            t = tabs.tok[k][tabs.ids[k][_cuda(b[sel]), pk]]
        x0[sel_t] = t + e
        emb[sel_t] = e
    return x0, emb


def _fwd(ops, case, tabs, plan, decoder, want_emb):
    D = tabs.D
    if decoder:
        return ops.embed_gather_fwd(plan, D, case.lens, case.vocabs, None, None, tabs.pos, tabs.mod,
                                    mask_token=tabs.mask_token, want_emb=want_emb)
    return ops.embed_gather_fwd(plan, D, case.lens, case.vocabs, tabs.ids, tabs.tok, tabs.pos, tabs.mod, want_emb=want_emb)


def _bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _check_fwd(ops, case, tabs, budget, decoder):
    pl = _run_plan(ops, case, budget, decoder)
    o = _oracle_plan(case, budget, decoder)
    D = tabs.D
    x_ref, e_ref = _embed_ref(case, tabs, _slot_rows(case, o), decoder)
    pp, _, _, _ = _pack(pl)
    for want_emb in (True, False):
        x0, emb = _fwd(ops, case, tabs, pl, decoder, want_emb)
        assert _bits_equal(x0.reshape(-1, D), x_ref), (decoder, want_emb)
        assert (emb is None) != want_emb
        if want_emb:
            assert _bits_equal(emb.reshape(-1, D), e_ref)
        xp, ep = _fwd(ops, case, tabs, pp, decoder, want_emb)
        slot = pp.slot_index
        assert xp.shape == (pp.rows, D) and _bits_equal(xp, x_ref[slot]), ("packed", decoder, want_emb)
        if want_emb:
            assert _bits_equal(ep, e_ref[slot])
    return pl, o


@pytest.mark.parametrize("D", [48, 384, 512, 768])
def test_embed_gather_fwd_bit_exact(ops, D):
    case = Case(_ragged_masks(LENS[4], 5, seed=D), [300, 1000, 17, 5000], seed=D)
    tabs = Tables(case, D, seed=D)
    for decoder in (False, True):
        _check_fwd(ops, case, tabs, 1213, decoder)


def test_embed_gather_fwd_egob_tables(ops):
    """Vocabulary 64 000 and 5 120 positions per video modality at D = 768, with the first and the last token id present."""
    case = _egob_case(6, 9, dec=False)
    for k, v in enumerate(case.vocabs):
        case.ids[k][:, ::7] = 0
        case.ids[k][:, 3::7] = v - 1
    tabs = Tables(case, 768, seed=1)
    pl, o = _check_fwd(ops, case, tabs, 2048, decoder=False)
    _, b, m, p = _slot_rows(case, o)
    valid = ~o["mask"].reshape(-1)
    kept = np.array([case.ids[mm][bb, pp] for bb, mm, pp in zip(b[valid], m[valid], p[valid])])
    big = np.array([case.vocabs[mm] for mm in m[valid]]) == 64000
    assert (kept[big] == 0).any() and (kept[big] == 63999).any()
    assert (p[valid][big] > 5000).any()
    dec = _egob_case(6, 9, dec=True)
    _check_fwd(ops, dec, Tables(dec, 768, seed=2), 2048, decoder=True)


def _bwd_ref(case, tabs, rows, dx0, demb, init, decoder):
    """{"tok" | "mod" | "mask": [(fp64 sum, bound) per buffer]}: the initial buffer plus index_add_ of the row gradients in
    fp64, and per element the bound n_terms * 2^-23 * sum|terms| (the initial value is a term) of an fp32 summation of the
    same terms in any order. A row adds dx0 to its token row or to the mask token, and dx0 + demb to its modality
    embedding: two fp32 terms, since the kernel rounds their sum before accumulating it."""
    valid, b, m, p = rows
    g = dx0.double()
    t_mod, a_mod, n_mod = (g, g.abs(), 1) if demb is None else (g + demb.double(), g.abs() + demb.double().abs(), 2)

    def total(base, dst, sel, terms, mags, n_per_row):
        s, a = base.double().clone(), base.double().abs()
        n = torch.ones(base.shape[0], 1, dtype=f64, device=DEV)
        if len(sel):
            r = _cuda(sel)
            s.index_add_(0, dst, terms[r])
            a.index_add_(0, dst, mags[r])
            n.index_add_(0, dst, torch.full((len(sel), 1), float(n_per_row), dtype=f64, device=DEV))
        return s, n * 2.0 ** -23 * a

    zeros = lambda k: torch.zeros(k, dtype=torch.int64, device=DEV)
    ref = {"tok": [], "mod": [], "mask": []}
    for k in range(len(case.lens)):
        sel = np.flatnonzero(valid & (m == k))
        ref["mod"].append(total(init["mod"][k].reshape(1, -1), zeros(len(sel)), sel, t_mod, a_mod, n_mod))
        if not decoder:
            tid = tabs.ids[k][_cuda(b[sel]), _cuda(p[sel])]
            ref["tok"].append(total(init["tok"][k], tid, sel, g, g.abs(), 1))
    sel = np.flatnonzero(valid)
    ref["mask"].append(total(init["mask"][0].reshape(1, -1), zeros(len(sel)), sel, g, g.abs(), 1))
    return ref


def _check_bwd(got, ref, what):
    got = got.double().reshape(ref[0].shape)
    err = (got - ref[0]).abs()
    worst = (err / ref[1]).nan_to_num(0.0, posinf=np.inf).max().item() if err.numel() else 0.0
    print(f"{what}: largest error {worst:.3f} of the bound")
    assert (err <= ref[1]).all(), f"{what}: error {worst:.3g} x the bound"


# Outputs passed as NULL: one token table, every token table, one modality embedding, every one of them, the mask token.
@pytest.mark.parametrize("decoder,null", [(False, "none"), (False, "tok"), (False, "all_tok"), (False, "mod"), (False, "all_mod"),
                                          (True, "none"), (True, "mask"), (True, "mod"), (True, "all_mod")])
@pytest.mark.parametrize("layout", ["dense", "packed"])
def test_embed_gather_bwd_fp64(ops, layout, decoder, null):
    D, budget = 384, 997                            # 6 x 997 rows: not a multiple of the kernel's 32-row CTAs
    case = Case(_ragged_masks(LENS[4], 6, seed=21), [300, 500, 17, 5000], seed=21)
    hot = case.ids[1]                               # one token id on ~80 % of modality 1: thousands of rows, many CTAs
    hot[np.random.default_rng(0).random(hot.shape) < 0.8] = 123
    tabs = Tables(case, D, seed=7)
    pl = _run_plan(ops, case, budget, decoder)
    o = _oracle_plan(case, budget, decoder)
    plan = pl if layout == "dense" else _pack(pl)[0]
    rows = _slot_rows(case, o, None if layout == "dense" else plan)
    if not decoder:
        valid, _, m, p = rows
        assert (hot[rows[1][valid & (m == 1)], p[valid & (m == 1)]] == 123).sum() > 2000
    R = len(rows[0])
    g = torch.Generator(device=DEV).manual_seed(R)
    dx0 = torch.randn(R, D, device=DEV, generator=g)
    demb = None if decoder else torch.randn(R, D, device=DEV, generator=g)
    init = {"tok": [torch.randn(v, D, device=DEV, generator=g) for v in case.vocabs],
            "mod": [torch.randn(D, device=DEV, generator=g) for _ in case.lens],
            "mask": [torch.randn(D, device=DEV, generator=g)]}
    buf = {k: [t.clone() for t in v] for k, v in init.items()}
    d_tabs = None if decoder else list(buf["tok"])
    d_mods = list(buf["mod"])
    d_mask = buf["mask"][0] if decoder else None
    if null == "tok":
        d_tabs[1] = None
    elif null == "all_tok":
        d_tabs = None
    elif null == "mod":
        d_mods[2] = None
    elif null == "all_mod":
        d_mods = None
    elif null == "mask":
        d_mask = None
    ops.embed_gather_bwd(plan, D, case.lens, case.vocabs, None if decoder else tabs.ids, tabs.pos, tabs.mod, dx0, demb,
                         d_tabs, d_mods, d_mask)
    ref = _bwd_ref(case, tabs, rows, dx0, demb, init, decoder)
    passed = {"tok": d_tabs or [None] * 4, "mod": d_mods or [None] * 4, "mask": [d_mask]}
    for name in (["mod", "mask"] if decoder else ["tok", "mod"]):
        for k, (b_, i_) in enumerate(zip(buf[name], init[name])):
            what = f"{name}[{k}] {layout} decoder={decoder}"
            if passed[name][k] is None:              # skipped output: its buffer is never written
                assert torch.equal(b_, i_), what
            else:
                _check_bwd(b_, ref[name][k], what)


# ------------------------------------------------------------------------------------------------ 6. head row gather / scatter
# (rows of src, n, cols); the second-to-last case has 65 536 x 96 16-byte vectors, far more than the grid's 1 184 CTAs x 256.
GATHER = [(5, 1, 8), (1000, 1, 768), (300, 777, 8), (2048, 4096, 768), (65536, 65536, 768), (70000, 40000, 8)]
# (rows of dst, n, cols); the first case scatters a permutation of all rows
SCATTER = [(1000, 1000, 8), (5, 1, 8), (1000, 1, 768), (300, 177, 8), (65536, 65536, 768), (70000, 40000, 768)]


@pytest.mark.parametrize("S,n,cols", GATHER)
def test_gather_rows_bf16_bit_exact(ops, S, n, cols):
    g = torch.Generator(device=DEV).manual_seed(S + n + cols)
    src = torch.randn(S, cols, device=DEV, generator=g).to(bf16)
    idx = torch.randint(0, S, (n,), device=DEV, generator=g)     # duplicates when n is not small against S
    idx[-1] = S - 1
    if n > 1:
        idx[0] = S - 1
    out = ops.gather_rows_bf16(src, idx)
    assert out.shape == (n, cols) and torch.equal(out.view(torch.int16), src.index_select(0, idx).view(torch.int16))


@pytest.mark.parametrize("S,n,cols", SCATTER)
def test_scatter_rows_f32_bit_exact(ops, S, n, cols):
    g = torch.Generator(device=DEV).manual_seed(S + n + cols)
    idx = torch.randperm(S, device=DEV, generator=g)[:n]
    if not (idx == S - 1).any():
        idx[0] = S - 1                                              # still no duplicate: the order of writes is fixed
    src = torch.randn(n, cols, device=DEV, generator=g)
    dst = torch.randn(S, cols, device=DEV, generator=g)
    ref = dst.clone().index_copy_(0, idx, src)                      # rows not in idx keep their values
    ops.scatter_rows_f32(src, idx, dst)
    assert _bits_equal(dst, ref)


# ------------------------------------------------------------------------------------------------ 7. wrapper checks, id clamping
def test_gather_rows_rejects_wrong_layout(ops):
    src = torch.randn(64, 16, device=DEV).to(bf16)
    idx = torch.arange(8, device=DEV)
    with pytest.raises(TypeError):
        ops.gather_rows_bf16(src, idx.int())
    with pytest.raises(TypeError):
        ops.gather_rows_bf16(src.float(), idx)
    with pytest.raises(ValueError):
        ops.gather_rows_bf16(torch.randn(64, 32, device=DEV).to(bf16)[:, :16], idx)   # row pitch 32, not 16
    with pytest.raises(ValueError):
        ops.gather_rows_bf16(src, torch.arange(16, device=DEV)[::2])
    with pytest.raises(RuntimeError):
        ops.gather_rows_bf16(src, idx.cpu())


def test_scatter_rows_rejects_wrong_layout(ops):
    src, dst = torch.randn(8, 16, device=DEV), torch.randn(64, 16, device=DEV)
    idx = torch.arange(8, device=DEV)
    with pytest.raises(TypeError):
        ops.scatter_rows_f32(src, idx.int(), dst)
    with pytest.raises(TypeError):
        ops.scatter_rows_f32(src.to(bf16), idx, dst)
    with pytest.raises(ValueError):
        ops.scatter_rows_f32(torch.randn(8, 32, device=DEV)[:, :16], idx, dst)
    with pytest.raises(ValueError):
        ops.scatter_rows_f32(src, idx, torch.randn(64, 32, device=DEV)[:, 16:])
    with pytest.raises(ValueError):
        ops.scatter_rows_f32(src, torch.arange(16, device=DEV)[::2], dst)
    assert torch.equal(ops.scatter_rows_f32(src, idx, dst.clone())[:8], src)


def _small_embed(ops):
    case = Case(_ragged_masks([30, 50], 4, seed=2), [40, 60], seed=2)
    return case, Tables(case, 64, seed=3), _run_plan(ops, case, 60, decoder=False)


def test_embed_gather_fwd_rejects_wrong_layout(ops):
    case, t, pl = _small_embed(ops)
    call = lambda **kw: ops.embed_gather_fwd(pl, 64, case.lens, case.vocabs, kw.get("ids", t.ids), kw.get("tok", t.tok),
                                             kw.get("pos", t.pos), kw.get("mod", t.mod))
    call()
    with pytest.raises(TypeError):
        call(ids=[i.int() for i in t.ids])
    with pytest.raises(ValueError):
        call(ids=[i.t().contiguous().t() for i in t.ids])                 # column-major (B, len)
    with pytest.raises(TypeError):
        call(tok=[x.to(bf16) for x in t.tok])
    with pytest.raises(ValueError):
        call(tok=[torch.randn(x.shape[0], 128, device=DEV)[:, :64] for x in t.tok])
    with pytest.raises(ValueError):
        call(pos=[x[:-1] for x in t.pos])
    with pytest.raises(TypeError):
        call(mod=[x.double() for x in t.mod])
    with pytest.raises(ValueError):
        ops.embed_gather_fwd(pl, 64, case.lens, case.vocabs, None, None, t.pos, t.mod,
                             mask_token=torch.randn(64, 2, device=DEV)[:, 0])


def test_embed_gather_bwd_rejects_wrong_layout(ops):
    case, t, pl = _small_embed(ops)
    R = pl.B * pl.budget
    dx0 = torch.randn(R, 64, device=DEV)
    d_tabs = [torch.zeros_like(x) for x in t.tok]
    call = lambda **kw: ops.embed_gather_bwd(pl, 64, case.lens, case.vocabs, kw.get("ids", t.ids), t.pos, t.mod,
                                             kw.get("dx0", dx0), None, kw.get("d_tabs", d_tabs), None, None)
    call()
    with pytest.raises(TypeError):
        call(ids=[i.int() for i in t.ids])
    with pytest.raises(ValueError):
        call(ids=[i.t().contiguous().t() for i in t.ids])
    with pytest.raises(TypeError):
        call(dx0=dx0.to(bf16))
    with pytest.raises(ValueError):
        call(d_tabs=[torch.zeros(x.shape[0], 128, device=DEV)[:, :64] for x in t.tok])


def test_embed_gather_clamps_out_of_range_ids(ops):
    """A token id below 0 reads (and its gradient lands in) row 0 of the table, one at or above the vocabulary row vocab - 1."""
    case, t, pl = _small_embed(ops)
    o = _oracle_plan(case, 60, False)
    valid, b, m, p = _slot_rows(case, o)
    rows = np.flatnonzero(valid & (m == 1))[:3]
    assert len(rows) == 3
    bad = [-5, case.vocabs[1], case.vocabs[1] + 1000]
    for r, v in zip(rows, bad):
        t.ids[1][b[r], p[r]] = v
    x0, _ = ops.embed_gather_fwd(pl, 64, case.lens, case.vocabs, t.ids, t.tok, t.pos, t.mod)
    x0 = x0.reshape(-1, 64)
    for r, row in zip(rows, [0, case.vocabs[1] - 1, case.vocabs[1] - 1]):
        assert _bits_equal(x0[r], t.tok[1][row] + (t.pos[1][p[r]] + t.mod[1]))
    dx0 = torch.zeros(pl.B * pl.budget, 64, device=DEV)
    dx0[_cuda(rows)] = torch.tensor([[1.0], [2.0], [4.0]], device=DEV)
    d_tabs = [torch.zeros_like(x) for x in t.tok]
    ops.embed_gather_bwd(pl, 64, case.lens, case.vocabs, t.ids, t.pos, t.mod, dx0, None, d_tabs, None, None)
    hit = d_tabs[1].abs().sum(1).nonzero().reshape(-1).tolist()
    assert hit == [0, case.vocabs[1] - 1]
    assert (d_tabs[1][0] == 1.0).all() and (d_tabs[1][-1] == 6.0).all()
