"""The fused CSC training step (csc_fused.cuh) across the shapes its selection rule admits, and on repetitive sequences.

Every case builds a default handle and its fused=False twin (the kernel-per-op tape) from the same parameters, asserts which path the
default handle ran, and checks it against the tape (same discrete results; loss 2e-6 relative; gradients 5e-6 of each block's largest
entry), against the PyTorch-CPU oracle (loss 1e-5 relative per group; gradient 2e-4 of its largest entry), for determinism (two calls,
same bits) and over three optimiser steps (parameters within 2e-6 per step of the tape's).

Which path ran is read from the kernel count of the step (ctx.last_timing()): the fully fused step is a fixed handful of kernels,
the tape is a few hundred, and a step the fused reverse pass flagged and re-ran on the tape is the sum of the two.
Run with -s to print one line per case: case, path, worst relative error against the oracle."""
import numpy as np
import pytest
import torch

import motifs_jl_b200 as mb
from motifs_jl_b200 import model as mdl, synth
from oracle import csc_oracle as co, scan_oracle as so

pytestmark = pytest.mark.gpu

_HP_FIELDS = ("filter_len", "M", "h", "K", "q", "batch_size", "num_pass_xyz", "num_pass_df", "magnifying_factor", "gamma")


def _ohp(hp):
    return co.Hyperparam(**{k: getattr(hp, k) for k in _HP_FIELDS})


def _kernels(ctx):
    return ctx.last_timing()[1]["csc"]


@pytest.fixture(scope="module")
def calib(ctx):
    """Kernel counts of one loss_grad on the default shape (batch 6, one group, Lb 100): fully fused, and on the tape."""
    hp = mdl.Hyperparam()
    a = synth.planted_gapped(12, 100, 1)
    seqs = ctx.seqs_from_ascii(a)
    flat = co.init_params(_ohp(hp), 1)
    out = {}
    for name, fused in (("fused", True), ("tape", False)):
        m = mb._lib.CscModel(ctx, hp, 100, fused=fused)
        m.set_params(flat)
        m.loss_grad(seqs, np.arange(6))
        out[name] = _kernels(ctx)
        m.free()
    seqs.free()
    assert 0 < out["fused"] <= 8 and out["tape"] > 5 * out["fused"], out
    return out


def _path(n, n_tape, calib):
    if n == calib["fused"]:
        return "fused"
    if n == n_tape:
        return "tape"
    if n == calib["fused"] + n_tape:
        return "fallback"                 # fused step flagged by its reverse pass, re-run on the tape
    return f"other({n})"


def _report(case, path, worst):
    print(f"\n[envelope] {case:<34} {path:<9} worst rel. error vs oracle {worst:.2e}", end="")


def _median_mask_ref(z, y, mf):
    """create_ZY_mask + cat_ZY, model.jl:194-210, per group in numpy (Statistics.median: middle(a,b) = a/2 + b/2)."""
    G = z.shape[0]
    zy = np.concatenate([z, y], axis=2)
    out = np.zeros_like(zy); med = np.zeros(G, np.float32)
    for g in range(G):
        pos = np.sort(zy[g][zy[g] > 0])
        if len(pos) == 0:
            med[g] = -np.inf
        elif len(pos) % 2:
            med[g] = pos[len(pos) // 2]
        else:
            med[g] = np.float32(pos[len(pos) // 2 - 1] * np.float32(0.5) + pos[len(pos) // 2] * np.float32(0.5))
        out[g] = np.where(zy[g] >= med[g], np.float32(mf) * zy[g], np.float32(0))
    return out, med


def _buffers(m, hp, Lb, G):
    B, c, l = hp.batch_size * G, Lb - hp.filter_len + 1, Lb - hp.filter_len + 1 - hp.h + 1
    return {name: m.get_buffer(name, n) for name, n in (("x", B * l * hp.K), ("z", B * c * hp.M), ("y", B * c * hp.M), ("zy", B * c * 2 * hp.M))}


def _assert_matches_tape(hp, lf, gf, bf, lt, gt, bt):
    assert np.allclose(lf, lt, rtol=2e-6, atol=0)
    for name in bf:
        assert np.array_equal(bf[name] != 0, bt[name] != 0), name
        assert np.allclose(bf[name], bt[name], rtol=1e-4, atol=1e-6), name
    o = 0
    for blk, n in co.param_sizes(_ohp(hp)).items():
        ref, new = gt[o:o + n], gf[o:o + n]
        assert np.abs(new - ref).max() <= 5e-6 * max(np.abs(ref).max(), 1e-9), blk
        o += n


# On repetitive rows the reference itself is ill-conditioned: run in float32 and in float64 on the batches of test_repetitive_sequences,
# the oracle keeps different top-q supports and median masks, and its loss moves by up to 1.6e-4 and its gradient by up to 1.7e-2 of
# the largest entry.  A group whose discrete results depend on rounding is held to this bar on the loss and its gradient is not compared.
_TIE_LOSS = 1e-3


def _same_support(a, b):
    return all(np.array_equal(a[n] != 0, np.asarray(b[n]).reshape(a[n].shape) != 0) for n in a)


def _oracle_worst(hp, flat, codes, idx, loss, g, groups=None, sup=None):
    """Per group: loss within 1e-5 relative; the mean gradient within 2e-4 of its largest entry.  `groups` maps group -> the
    representative group whose oracle result it shares (identical rows), so repeated batches are evaluated once.
    With `sup` (the handle's final x and zy, one block per group) the oracle also runs in float64.  A group whose top-q supports or median
    masks differ between the oracle's float32 and float64 runs, or between the handle and the oracle, sits on a tie that rounding breaks
    (an fp32 summation order decides between equal values): its loss is held to _TIE_LOSS and the gradient is not compared.
    Returns (worst relative error, number of such groups)."""
    ohp, B = _ohp(hp), hp.batch_size
    G = loss.shape[0]
    cache, og_sum, worst, ties = {}, np.zeros(g.size, np.float64), 0.0, 0
    for k in range(G):
        r = groups[k] if groups is not None else k
        if r not in cache:
            ol, og, aux = co.loss_and_grad(codes[idx[r * B:(r + 1) * B]], flat, ohp)
            osup = {n: aux[n].detach().numpy() for n in ("x", "zy")}
            ill = False
            if sup is not None:
                _, _, aux64 = co.loss_and_grad(codes[idx[r * B:(r + 1) * B]], flat, ohp, dtype=torch.float64)
                ill = not _same_support(osup, {n: aux64[n].detach().numpy() for n in osup})
            cache[r] = (float(ol), og[: g.size], osup, ill)
        ol, og, osup, ill = cache[r]
        rel = abs(float(loss[k, 0]) - ol) / abs(ol)
        if sup is not None and (ill or not _same_support({n: sup[n][k] for n in osup}, osup)):
            ties += 1
            assert rel <= _TIE_LOSS, (k, float(loss[k, 0]), ol)
        else:
            assert rel <= 1e-5, (k, float(loss[k, 0]), ol)
            worst = max(worst, rel)
        og_sum += og
    if ties == 0:
        og_mean = og_sum / G
        gerr = np.abs(g - og_mean).max() / np.abs(og_mean).max()
        assert gerr <= 2e-4, gerr
        worst = max(worst, gerr)
    return worst, ties


def _pair(ctx, hp, Lb, G, flat):
    mf = mb._lib.CscModel(ctx, hp, Lb, n_groups=G)
    mt = mb._lib.CscModel(ctx, hp, Lb, n_groups=G, fused=False)
    mf.set_params(flat); mt.set_params(flat)
    return mf, mt


def _run_pair(ctx, calib, mf, mt, seqs, idx):
    lt, gt = mt.loss_grad(seqs, idx)
    n_tape = _kernels(ctx)
    lf, gf = mf.loss_grad(seqs, idx)
    return _path(_kernels(ctx), n_tape, calib), (lf, gf), (lt, gt)


# (case id, hyper-parameters other than the defaults, Lb, groups, accepted paths)
_FUSED, _TAPE, _EITHER = ("fused",), ("tape",), ("fused", "tape")
_CASES = [
    ("Lb23", {}, 23, 1, _FUSED),                         # c = 16: one row per CTA
    ("Lb24", {}, 24, 1, _FUSED),                         # c = 17: CTAs 9-15 own no rows
    ("Lb27", {}, 27, 1, _FUSED),                         # c = 20
    ("Lb330", {}, 330, 1, _FUSED),                       # the largest Lb whose forward kernel fits the 227 KB opt-in shared memory
    ("Lb331", {}, 331, 1, _TAPE),                        # one byte over it
    ("batch2", dict(batch_size=2), 100, 1, _FUSED),      # the smallest batch with B x 16 >= K
    ("batch3", dict(batch_size=3), 100, 1, _FUSED),
    ("batch4", dict(batch_size=4), 100, 1, _FUSED),
    ("batch7", dict(batch_size=7), 100, 1, _EITHER),     # 7 and 8 clusters of 16 CTAs: whether they are co-resident depends on the part
    ("batch8", dict(batch_size=8), 100, 1, _EITHER),     # B x LIST_CAP = FZ_THREADS
    ("xyz1", dict(num_pass_xyz=1), 100, 1, _FUSED),
    ("xyz8", dict(num_pass_xyz=8), 100, 1, _FUSED),
    ("xyz9", dict(num_pass_xyz=9), 100, 1, _TAPE),
    ("df1", dict(num_pass_df=1), 100, 1, _FUSED),
    ("df4", dict(num_pass_df=4), 100, 1, _FUSED),
    ("df5", dict(num_pass_df=5), 100, 1, _TAPE),
    ("q1", dict(q=1), 100, 1, _FUSED),
    ("q64", dict(q=64), 100, 1, _FUSED),                 # q = LIST_CAP
    ("batch2x3groups", dict(batch_size=2), 100, 3, _FUSED),   # 6 clusters, as many as the default step
    ("batch3x2groups", dict(batch_size=3), 100, 2, _FUSED),
    ("batch6x2groups", {}, 100, 2, _TAPE),               # 12 clusters do not fit
    ("q65", dict(q=65), 100, 1, _TAPE),                  # q > LIST_CAP: the code lists overflow on every step, training keeps the tape
    ("q100", dict(q=100), 100, 1, _TAPE),
    ("q256", dict(q=256), 100, 1, _TAPE),
    ("q257", dict(q=257), 100, 1, _TAPE),                # also past FZ_KCAP, the fused reverse pass's kept-entry capacity
    ("q100x40groups", dict(q=100), 100, 40, _TAPE),      # the batched one-CTA-per-sequence kernels with overflowing code lists
]


@pytest.mark.parametrize("case,hpd,Lb,G,paths", _CASES, ids=[c[0] for c in _CASES])
def test_shape_envelope(ctx, calib, case, hpd, Lb, G, paths):
    hp = mdl.Hyperparam(**hpd)
    B = hp.batch_size
    N = B * G + 5
    a = synth.planted_gapped(N, Lb, 17)
    seqs = ctx.seqs_from_ascii(a)
    flat = co.init_params(_ohp(hp), 17)
    mf, mt = _pair(ctx, hp, Lb, G, flat)
    rng = np.random.default_rng(3)
    idx = rng.permutation(N)[: B * G]
    path, (lf, gf), (lt, gt) = _run_pair(ctx, calib, mf, mt, seqs, idx)
    assert path in paths, (case, path)
    _assert_matches_tape(hp, lf, gf, _buffers(mf, hp, Lb, G), lt, gt, _buffers(mt, hp, Lb, G))
    worst, _ = _oracle_worst(hp, flat, so.ascii_to_codes(a), idx, lf, gf)
    lf2, gf2 = mf.loss_grad(seqs, idx)
    assert np.array_equal(lf, lf2) and np.array_equal(gf, gf2)
    # three optimiser steps on the same batches: |update| <= eta = 1e-3 per entry, the two paths stay within 2e-6 per step
    for step in range(3):
        bi = rng.permutation(N)[: B * G]
        mf.step_begin(seqs, bi); mf.adabelief_step()
        mt.step_begin(seqs, bi); mt.adabelief_step()
        d = np.abs(mf.get_params() - mt.get_params())
        assert d.max() <= 2e-6 * (step + 1), (step, d.max(), int(d.argmax()))
    _report(case, path, worst)
    mf.free(); mt.free(); seqs.free()


def _code_records_match(got, exp):
    """The bars of test_code_retrieval_matches_oracle: same (position, fil, seq), magnitudes within 2 Float16 ulps for 99 %."""
    assert len(got) == len(exp)
    for f in ("position", "fil", "seq"):
        assert np.array_equal(got[f], exp[f]), f
    gm, em = got["mag_f16"].view(np.float16).astype(np.float32), exp["mag_f16"].view(np.float16).astype(np.float32)
    d = np.abs(gm - em)
    assert (d <= 2e-6).mean() >= 0.99, f"{(d > 2e-6).sum()} of {len(d)} magnitudes differ by more than 2 Float16 ulps"
    assert np.allclose(gm, em, rtol=2e-2, atol=4e-6)


@pytest.mark.parametrize("q,G", [(80, 1), (100, 1), (100, 40)])
def test_code_retrieval_past_the_list_capacity(ctx, q, G):
    """q > LIST_CAP on a forward-only handle: more than 64 codes in every sequence, more than CODE_SLOTS = 96 for q = 100, which
    code retrieval emits again with a wider stride."""
    hp = mdl.Hyperparam(q=q)
    a = synth.planted_gapped(30, 100, 7)
    seqs = ctx.seqs_from_ascii(a)
    flat = co.init_params(_ohp(hp), 7)
    m = mb._lib.CscModel(ctx, hp, 100, n_groups=G, forward_only=True)
    m.set_params(flat)
    got = m.codes(seqs)
    exp = co.code_retrieval(so.ascii_to_codes(a), flat, _ohp(hp))
    _code_records_match(got, exp)
    assert np.bincount(got["seq"]).max() > (96 if q > 96 else 64)
    _report(f"codes_q{q}x{G}groups", "tape", 0.0)
    m.free(); seqs.free()


# ---- repetitive sequences --------------------------------------------------------------------------------------------------
_KINDS = ("polyA", "AT", "CAG", "Arun60", "mixed")


def _rep_rows(kind, n, Lb, seed):
    rng = np.random.default_rng(seed)
    rand = synth.random_ascii(n, Lb, seed + 1000)
    if kind == "polyA":
        return np.full((n, Lb), ord("A"), np.uint8)
    if kind in ("AT", "CAG"):
        unit = np.frombuffer(kind.encode(), np.uint8)
        reps = Lb // len(unit) + 2
        return np.stack([np.tile(unit, reps)[p: p + Lb] for p in rng.integers(0, len(unit), n)])
    if kind == "Arun60":
        out = rand.copy()
        for r, p in enumerate(rng.integers(0, Lb - 60 + 1, n)):
            out[r, p: p + 60] = ord("A")
        return out
    # mixed: two rows of each repetitive kind in turn, the rest random
    out = synth.planted_gapped(n, Lb, seed + 2000)
    kinds = ("polyA", "AT", "CAG", "Arun60")
    for r in range(0, n, 3):
        out[r] = _rep_rows(kinds[(r // 3) % 4], 1, Lb, seed + r)[0]
    return out


_BATCHES = 4          # distinct 6-row batches per kind; a 40-group launch cycles through them


@pytest.mark.parametrize("Lb,G", [(100, 1), (200, 1), (100, 40), (200, 40)])
@pytest.mark.parametrize("kind", _KINDS)
def test_repetitive_sequences(ctx, calib, kind, Lb, G):
    """Poly-A, (AT)n, (CAG)n, a 60 bp A-run and a mix with random rows repeat the same windows along a sequence, so many code values tie:
    the kept set at the q-th value can exceed the fused reverse pass's list capacity, and the median's bin holds thousands of entries.
    The step must succeed (fused, or flagged and re-run on the tape); the batch median must equal the reference median of the z and y of
    the same run, bit for bit, on both paths; loss, gradient and code records must match the tape and the oracle wherever the two broke
    no tie differently (an fp32 summation order decides between equal values; such groups are counted and their loss held to _TIE_LOSS);
    the code records must be the handle's own x, and the oracle's records wherever those do not depend on rounding."""
    hp = mdl.Hyperparam()
    B = hp.batch_size
    a = np.concatenate([_rep_rows(kind, B, Lb, 11 * j + 1) for j in range(_BATCHES)])
    seqs = ctx.seqs_from_ascii(a)
    flat = co.init_params(_ohp(hp), 5)
    groups = [k % _BATCHES for k in range(G)]
    idx = np.concatenate([np.arange(B * g, B * g + B) for g in groups])
    mf, mt = _pair(ctx, hp, Lb, G, flat)
    path, (lf, gf), (lt, gt) = _run_pair(ctx, calib, mf, mt, seqs, idx)
    assert path in (("fused", "fallback") if G == 1 else ("tape",)), path
    bf, bt = _buffers(mf, hp, Lb, G), _buffers(mt, hp, Lb, G)
    note = ""
    if path != "fused":                    # both ran the tape: the same kernels in the same order
        assert np.array_equal(lf, lt) and np.array_equal(gf, gt)
    elif all(np.array_equal(bf[k] != 0, bt[k] != 0) for k in ("x", "zy")):
        _assert_matches_tape(hp, lf, gf, bf, lt, gt, bt)
    else:                                  # a tie at the q-th value or the median broken the other way by fp32 summation order
        assert np.allclose(lf, lt, rtol=_TIE_LOSS, atol=0)
        note = " (tie vs tape)"
    c, l = Lb - hp.filter_len + 1, Lb - hp.filter_len + 1 - hp.h + 1
    # the batch median of the z and y this run produced, recomputed in numpy: bit for bit, on both paths
    for b in (bf, bt):
        z, y = b["z"].reshape(G, B * c, hp.M), b["y"].reshape(G, B * c, hp.M)
        rzy, _ = _median_mask_ref(z, y, hp.magnifying_factor)
        assert np.array_equal(b["zy"].reshape(G, B * c, 2 * hp.M), rzy)
    worst, ties = _oracle_worst(hp, flat, so.ascii_to_codes(a), idx, lf, gf, groups=groups,
                                sup={"x": bf["x"].reshape(G, B, l, hp.K), "zy": bf["zy"].reshape(G, B, c, 2 * hp.M)})
    mf.free(); mt.free()
    fo = mb._lib.CscModel(ctx, hp, Lb, n_groups=G, forward_only=True)
    fo.set_params(flat)
    got = fo.codes(seqs)
    # the records are the positive entries of x, ordered by filter and position, as Float16: the last decoded batch is still in the handle
    NS = B * G
    s0 = (len(a) - 1) // NS * NS
    xl = fo.get_buffer("x", NS * l * hp.K).reshape(NS, l, hp.K)
    for i in range(len(a) - s0):
        xt = xl[i].T
        fil, pos = np.nonzero(xt > 0)
        gq = got[got["seq"] == s0 + i]
        assert np.array_equal(gq["fil"], fil) and np.array_equal(gq["position"], pos), s0 + i
        assert np.array_equal(gq["mag_f16"], xt[fil, pos].astype(np.float16).view(np.uint16)), s0 + i
    # against the oracle, per sequence, wherever its own float32 and float64 runs keep the same codes
    codes = so.ascii_to_codes(a)
    exp = co.code_retrieval(codes, flat, _ohp(hp))
    exp64 = co.code_retrieval(codes, flat, _ohp(hp), dtype=torch.float64)
    same = 0
    for q in range(len(a)):
        eq, e64 = exp[exp["seq"] == q], exp64[exp64["seq"] == q]
        if len(eq) == len(e64) and np.array_equal(eq["position"], e64["position"]) and np.array_equal(eq["fil"], e64["fil"]):
            _code_records_match(got[got["seq"] == q], eq)
            same += 1
    _report(f"{kind}_Lb{Lb}x{G}groups", path, worst)
    print(f" groups with a tie vs oracle {ties}/{G}{note}; sequences compared with the oracle's codes {same}/{len(a)}; codes/seq max "
          f"{np.bincount(got['seq']).max()}", end="")
    fo.free(); seqs.free()


def test_flagged_step_updates_from_the_tape_gradient(ctx, calib):
    """A step the fused reverse pass cannot represent (here the warm-up's top-q keeps every entry: omega_w = 0 makes all values tie at
    zero, more than FZ_KCAP kept entries) is re-run on the tape.  loss_grad returns the tape's result, one optimiser step applies the
    tape's gradient exactly once (parameters bit-identical to a tape handle's, step counter advanced once), and the next ordinary step
    runs fused again."""
    hp = mdl.Hyperparam()
    a = synth.planted_gapped(12, 100, 31)
    seqs = ctx.seqs_from_ascii(a)
    flat = co.init_params(_ohp(hp), 31)
    deg = flat.copy(); deg[-1] = 0.0                           # omega_stepsize_warmup (the last of the three warm-up scalars)
    idx = np.arange(6)
    mf, mt = _pair(ctx, hp, 100, 1, deg)
    path, (lf, gf), (lt, gt) = _run_pair(ctx, calib, mf, mt, seqs, idx)
    assert path == "fallback"
    assert np.array_equal(lf, lt) and np.array_equal(gf, gt)
    assert _oracle_worst(hp, deg, so.ascii_to_codes(a), idx, lf, gf)[1] == 0
    mf.free(); mt.free()
    mf, mt = _pair(ctx, hp, 100, 1, deg)                      # fresh optimiser state on both
    mf.step_begin(seqs, idx); l_f = mf.adabelief_step()
    mt.step_begin(seqs, idx); l_t = mt.adabelief_step()
    assert l_f == l_t
    pf, pt = mf.get_params(), mt.get_params()
    assert np.array_equal(pf, pt) and not np.array_equal(pf, deg)
    # back to ordinary parameters (the warm-up scalars are not trained): the step runs fused, and the second update is the tape's to
    # within summation order; had the flagged step advanced the step counter twice, the bias correction would differ by ~50 %
    pf[-1] = pt[-1] = flat[-1]
    mf.set_params(pf); mt.set_params(pt)
    idx2 = np.arange(6, 12)
    path, _, _ = _run_pair(ctx, calib, mf, mt, seqs, idx2)
    assert path == "fused"
    mf.step_begin(seqs, idx2); mf.adabelief_step()
    mt.step_begin(seqs, idx2); mt.adabelief_step()
    assert np.abs(mf.get_params() - mt.get_params()).max() <= 2e-6
    _report("flagged_step", "fallback", 0.0)
    mf.free(); mt.free(); seqs.free()


def test_training_with_repetitive_rows(ctx):
    """50 optimiser steps on the default handle, a third of the batches holding repetitive rows: every step completes and the loss of a
    fixed batch of ordinary rows goes down."""
    hp = mdl.Hyperparam()
    clean = synth.planted_gapped(120, 100, 9)
    rep = np.concatenate([_rep_rows(k, 6, 100, 40 + i) for i, k in enumerate(_KINDS)])
    a = np.concatenate([clean, rep])
    seqs = ctx.seqs_from_ascii(a)
    flat = co.init_params(_ohp(hp), 9)
    m = mb._lib.CscModel(ctx, hp, 100)
    m.set_params(flat)
    probe = np.arange(6)
    l0, _ = m.loss_grad(seqs, probe)
    rng = np.random.default_rng(4)
    for step in range(50):
        if step % 3 == 2:
            idx = np.concatenate([rng.choice(120, 3, replace=False), 120 + rng.choice(len(rep), 3, replace=False)])
        else:
            idx = rng.choice(120, 6, replace=False)
        m.step_begin(seqs, idx)
        loss, l1 = m.adabelief_step()
        assert np.isfinite(loss) and np.isfinite(l1), step
    l1_, _ = m.loss_grad(seqs, probe)
    assert l1_[0, 0] < l0[0, 0], (l0[0, 0], l1_[0, 0])
    m.free(); seqs.free()
