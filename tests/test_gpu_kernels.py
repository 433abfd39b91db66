"""GPU parity tests proper: every C-ABI kernel against the CPU oracle (and the reference fixtures) on the
same seeded inputs.  Tolerances: index selection bit-exact wherever the float64 ground truth can decide
it; weights/readout 1e-5; transformer tensors 2e-4 relative to O(10) activations; BASELINE.json's bar is
1e-3 max-abs on segmentation logits (tests/test_gpu_e2e.py)."""
import math
import os

import numpy as np
import pytest
import torch

from oracle import memory_math as mm
from oracle import transformer as otf
from tests.conftest import GOLDEN

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def K_():
    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB):
        ge.build()
    import cutie_b200.kernels as k
    k.lib()
    return k


def dev(t):
    return t.cuda()


def make_bank(B, N, K, CK=64, CV=256, seed=0, cuts=()):
    g = torch.Generator().manual_seed(seed)
    key = torch.randn(B, N, CK, generator=g)
    shr = 1 + torch.randn(B, N, generator=g) ** 2
    vals = [torch.randn(B, N, CV, generator=g) for _ in range(K)]
    return key, shr, vals


def segments_of(K_, key, shr, vals, cuts):
    """Split [B,N,..] tensors into physically separate (non-adjacent) runs like the arena does, each with the FP16 key
    image of its own buffer (so banks at or above the filter threshold take the image plan)."""
    segs, lo = [], 0
    for hi in list(cuts) + [key.shape[1]]:
        # embed each run in a larger buffer so batch strides differ from n*C
        pad = 3
        kb = torch.zeros(key.shape[0], hi - lo + pad, key.shape[2]).cuda()
        sb = torch.zeros(key.shape[0], hi - lo + pad).cuda()
        kb[:, :hi - lo] = key[:, lo:hi].cuda()
        sb[:, :hi - lo] = shr[:, lo:hi].cuda()
        vb = []
        for v in vals:
            t = torch.zeros(v.shape[0], hi - lo + pad, v.shape[2]).cuda()
            t[:, :hi - lo] = v[:, lo:hi].cuda()
            vb.append(t[:, :hi - lo])
        img = torch.zeros(key.shape[0], K_.key_image_tiles(hi - lo + pad), K_.KEY_IMAGE_FLOATS).cuda()
        K_.bank_key_image(kb, sb, 0, hi - lo, img)
        segs.append(K_.BankSegment(kb[:, :hi - lo], sb[:, :hi - lo], tuple(vb), img, 0))
        lo = hi
    return segs


def check_topk(K_, B, N, Q, K, top_k, cuts=(), seed=0, key_scale=1.0):
    key, shr, vals = make_bank(B, N, K, seed=seed)
    key = key * key_scale
    g = torch.Generator().manual_seed(seed + 1)
    qk = torch.randn(B, 64, Q, generator=g) * key_scale
    qe = torch.sigmoid(torch.randn(B, 64, Q, generator=g))
    segs = segments_of(K_, key, shr, vals, cuts)
    usage = torch.zeros(B, N, dtype=torch.int64).cuda()
    idx, w, sim = K_.affinity_topk(segs, qk.cuda(), qe.cuda(), top_k, usage_acc=usage, want_sim=True)
    out = K_.readout_gather(idx, w, segs)
    torch.cuda.synchronize()
    idx, w, sim, out, usage = idx.cpu(), w.cpu(), sim.cpu(), out.cpu(), usage.cpu()
    # ---- oracle ----
    truth = mm.similarity_direct(key.transpose(1, 2), shr.unsqueeze(1), qk, qe, dtype=torch.float64)
    kk = idx[:, :, :top_k].transpose(1, 2).long()                     # [B,k,Q]
    assert (idx[:, :, top_k:] == -1).all() and (w[:, :, top_k:] == 0).all()
    assert (kk >= 0).all() and (kk < N).all()
    # similarity of the winners is the true similarity (fp32 direct form: relative 1e-5)
    got_sim = sim[:, :, :top_k].transpose(1, 2).double()
    ref_sim = torch.gather(truth, 1, kk)
    assert torch.allclose(got_sim, ref_sim, rtol=2e-5, atol=1e-5)
    # index sets: identical on every query whose k-th/(k+1)-th gap the fp32 direct form can resolve
    n_dec, n_dec_eq, n_eq, n_all = mm.topk_set_agreement(kk, truth, top_k, 4e-6)
    assert n_dec_eq == n_dec, f'{n_dec - n_dec_eq} decidable queries picked a different top-{top_k} set'
    assert n_dec >= 0.95 * n_all
    # winners sorted by descending similarity
    assert (got_sim[:, :-1] >= got_sim[:, 1:]).all()
    # softmax weights over the winners
    ref_w = torch.softmax(ref_sim, dim=1).float()
    assert torch.allclose(w[:, :, :top_k].transpose(1, 2), ref_w, rtol=1e-4, atol=1e-6)
    assert torch.allclose(w.sum(-1), torch.ones(B, Q), atol=1e-5)
    # usage: fixed-point sum of weights per token
    aff = mm.scatter_affinity(kk, w[:, :, :top_k].transpose(1, 2).contiguous(), N)
    assert torch.allclose(usage.double() * 2.0 ** -40, aff.sum(2).double(), atol=1e-5)
    assert abs(float(usage.double().sum()) * 2.0 ** -40 - B * Q) < 1e-3 * B * Q
    # readout == dense V . A of the reference formulation
    vstack = torch.stack([v.transpose(1, 2) for v in vals], 1)          # [B,K,CV,N]
    ref_out = mm.readout(aff, vstack)
    assert torch.allclose(out, ref_out, rtol=1e-4, atol=2e-5)
    return idx, w


@pytest.mark.parametrize('B,N,Q,K,cuts', [
    (1, 333, 77, 3, ()),                 # ragged everything, single segment
    (2, 1000, 130, 2, (128, 500, 501)),  # four segments, one of length 1, batch 2 (flip_aug)
    (1, 30, 5, 1, ()),                   # N == top_k: every token wins
    (1, 4099, 1620, 3, (4000,)),         # 480p query count, two segments, many key splits
])
def test_affinity_topk_readout_vs_oracle(K_, B, N, Q, K, cuts):
    check_topk(K_, B, N, Q, K, 30, cuts)


def test_affinity_topk_k64_and_k1(K_):
    check_topk(K_, 1, 700, 100, 1, 64)
    check_topk(K_, 1, 700, 100, 1, 1)
    check_topk(K_, 1, 700, 100, 2, 33, cuts=(100,))


def test_affinity_topk_large_bank_property(K_):
    """Full-size bank (cfg 2 scale keys, fewer queries to keep the float64 oracle fast): invariants +
    agreement with the oracle on a query subset."""
    check_topk(K_, 1, 60000, 96, 1, 30, cuts=(1620, 30000))


def test_topk_too_few_tokens_raises(K_):
    key, shr, vals = make_bank(1, 10, 1)
    segs = segments_of(K_, key, shr, vals, ())
    with pytest.raises(K_.KernelError):
        K_.affinity_topk(segs, torch.randn(1, 64, 8).cuda(), torch.rand(1, 64, 8).cuda(), 30)


def test_memory_kat_against_reference_fixture(K_):
    """The reference's own get_similarity/do_softmax/_readout outputs (tests/golden/kat_memory.npz)."""
    g = np.load(os.path.join(GOLDEN, 'kat_memory.npz'))
    mk, ms = torch.from_numpy(g['mk']), torch.from_numpy(g['ms'])
    qk, qe, v = torch.from_numpy(g['qk']), torch.from_numpy(g['qe']), torch.from_numpy(g['v'])
    B, CK, N = mk.shape
    K = v.shape[1]
    segs = segments_of(K_, mk.transpose(1, 2).contiguous(), ms[:, 0], [v[:, k].transpose(1, 2).contiguous() for k in range(K)], (100,))
    usage = torch.zeros(B, N, dtype=torch.int64).cuda()
    idx, w, _ = K_.affinity_topk(segs, qk.cuda(), qe.cuda(), 30, usage_acc=usage)
    out = K_.readout_gather(idx, w, segs).cpu()
    idx, w = idx.cpu(), w.cpu()
    ref_idx = torch.from_numpy(g['topk_idx'])                               # [B,30,Q] from torch.topk
    assert (idx[:, :, :30].transpose(1, 2).long().sort(1)[0] == ref_idx.sort(1)[0]).all()
    aff = mm.scatter_affinity(idx[:, :, :30].transpose(1, 2).long(), w[:, :, :30].transpose(1, 2).contiguous(), N)
    assert torch.allclose(aff, torch.from_numpy(g['affinity']), atol=2e-6)
    assert torch.allclose(usage.cpu().double() * 2.0 ** -40, torch.from_numpy(g['usage']).double(), atol=1e-5)
    assert torch.allclose(out, torch.from_numpy(g['readout']), rtol=1e-4, atol=2e-5)


def test_tie_rule(K_):
    """Exact duplicate keys: values of the winners match the reference; ties resolve to the lower index."""
    g = np.load(os.path.join(GOLDEN, 'kat_memory.npz'))
    mk, ms = torch.from_numpy(g['tie_mk']), torch.from_numpy(g['tie_ms'])
    qk, qe = torch.from_numpy(g['qk'][:1]), torch.from_numpy(g['qe'][:1])
    N = mk.shape[-1]
    segs = segments_of(K_, mk.transpose(1, 2).contiguous(), ms[:, 0], [], ())
    idx, w, sim = K_.affinity_topk(segs, qk.cuda(), qe.cuda(), 30, want_sim=True)
    idx, w, sim = idx.cpu(), w.cpu(), sim.cpu()
    ref_aff = torch.from_numpy(g['tie_affinity'])
    # the multiset of winning weights is identical even though tied indices may differ
    ref_w = ref_aff.transpose(1, 2).sort(-1, descending=True)[0][:, :, :30]
    assert torch.allclose(w[:, :, :30].sort(-1, descending=True)[0], ref_w, atol=2e-6)
    half = N // 2
    # tokens n and n+half are identical: 30 winners = 15 duplicate pairs, in (lower, upper) order
    kk = idx[0, :, :30]
    assert (kk[:, 0::2] + half == kk[:, 1::2]).all()
    assert (sim[0, :, 0:30:2] == sim[0, :, 1:30:2]).all()


def test_usage_commit(K_):
    use = torch.rand(2, 50).cuda()
    life = torch.rand(2, 50).cuda()
    acc = (torch.rand(2, 80) * 2 ** 40).to(torch.int64).cuda()
    u0, l0 = use.clone(), life.clone()
    K_.usage_commit(use[:, 5:45], life[:, 5:45], acc, 7)
    exp = u0.clone()
    exp[:, 5:45] += (acc[:, 7:47].double() * 2.0 ** -40).float()
    assert torch.allclose(use, exp, atol=1e-6)
    assert torch.allclose(life[:, 5:45], l0[:, 5:45] + 1) and torch.equal(life[:, :5], l0[:, :5])


def test_bank_append_export_gather(K_):
    g = torch.Generator().manual_seed(3)
    src = torch.randn(2, 64, 77, generator=g).cuda()
    arena = torch.zeros(2, 200, 64).cuda()
    K_.bank_append(src, arena[:, 10:87])
    assert torch.equal(arena[:, 10:87], src.transpose(1, 2))
    assert arena[:, :10].abs().sum() == 0 and arena[:, 87:].abs().sum() == 0
    back = torch.empty(2, 64, 77).cuda()
    K_.bank_export(arena[:, 10:87], back)
    assert torch.equal(back, src)
    v = torch.randn(2, 256, 33, generator=g).cuda()
    va = torch.zeros(2, 40, 256).cuda()
    K_.bank_append(v, va[:, 3:36])
    assert torch.equal(va[:, 3:36], v.transpose(1, 2))
    idx = torch.stack([torch.randperm(110, generator=g)[:20] for _ in range(2)]).cuda()
    dst = torch.zeros(2, 25, 64).cuda()
    K_.bank_gather([arena[:, 10:87], arena[:, 100:133]], idx, dst[:, 2:22])
    cat = torch.cat([arena[:, 10:87], arena[:, 100:133]], 1)
    for b in range(2):
        assert torch.equal(dst[b, 2:22], cat[b][idx[b]])
    # width-1 rows (shrinkage / usage counters)
    s = torch.randn(2, 110).cuda()
    d1 = torch.zeros(2, 20).cuda()
    K_.bank_gather([s.unsqueeze(-1)], idx, d1.unsqueeze(-1))
    assert torch.equal(d1, torch.gather(s, 1, idx))


def test_consolidate_vs_reference_fixture(K_):
    g = np.load(os.path.join(GOLDEN, 'kat_memory.npz'))
    ck, cs, ce = (torch.from_numpy(g[k]) for k in ('cons_key', 'cons_shrinkage', 'cons_selection'))
    v1, v5, cu = torch.from_numpy(g['cons_v1']), torch.from_numpy(g['cons_v5']), torch.from_numpy(g['cons_usage'])
    B, CK, Nc = ck.shape
    P = g['cons_pk'].shape[-1]
    pidx = torch.stack([torch.topk(cu[b], k=P, sorted=True)[1] for b in range(B)])
    segs = segments_of(K_, ck.transpose(1, 2).contiguous(), cs[:, 0],
                       [v1.transpose(1, 2).contiguous(), v5.transpose(1, 2).contiguous()], (77,))
    pk = torch.zeros(B, P, CK).cuda()
    pe = torch.zeros(B, P, CK).cuda()
    K_.bank_gather([s.key for s in segs], pidx.cuda(), pk)
    ce_rows = ce.transpose(1, 2).contiguous().cuda()
    K_.bank_gather([ce_rows], pidx.cuda(), pe)
    assert torch.equal(pk.cpu().transpose(1, 2), torch.from_numpy(g['cons_pk']))
    ov = [torch.zeros(B, P, 256).cuda() for _ in range(2)]
    osr = torch.zeros(B, P).cuda()
    K_.consolidate(segs, pk, pe, ov, osr)
    assert torch.allclose(ov[0].cpu().transpose(1, 2), torch.from_numpy(g['cons_pv1']), rtol=1e-4, atol=2e-5)
    assert torch.allclose(ov[1].cpu().transpose(1, 2), torch.from_numpy(g['cons_pv5']), rtol=1e-4, atol=2e-5)
    assert torch.allclose(osr.cpu().unsqueeze(1), torch.from_numpy(g['cons_ps']), rtol=1e-4, atol=2e-5)
    # cutie_consolidate_partial: two shards of the candidates, each normalised by its own (returned) softmax statistics,
    # combined the way inference/sharded.combine_partial_softmax does -> the whole-bank result
    parts = []
    for lo, hi in ((0, 100), (100, Nc)):
        sh = segments_of(K_, ck[:, :, lo:hi].transpose(1, 2).contiguous(), cs[:, 0, lo:hi],
                         [v1[:, :, lo:hi].transpose(1, 2).contiguous(), v5[:, :, lo:hi].transpose(1, 2).contiguous()], ())
        pv = [torch.zeros(B, P, 256).cuda() for _ in range(2)]
        ps, mx, se = torch.zeros(B, P).cuda(), torch.zeros(B, P).cuda(), torch.zeros(B, P).cuda()
        K_.consolidate(sh, pk, pe, pv, ps, stats=(mx, se))
        parts.append((torch.cat(pv + [ps.unsqueeze(-1)], -1), mx, se))
    big = torch.maximum(parts[0][1], parts[1][1])
    wgt = [se * torch.exp(mx - big) for _, mx, se in parts]
    comb = sum(w.unsqueeze(-1) * part for w, (part, _, _) in zip(wgt, parts)) / (wgt[0] + wgt[1]).unsqueeze(-1)
    whole = torch.cat(ov + [osr.unsqueeze(-1)], -1)
    assert torch.allclose(comb, whole, rtol=1e-5, atol=1e-6), float((comb - whole).abs().max())


# ---------------------------------------------------------------------------------------------
# object transformer kernels vs tests/cpu_kernels.py contracts (which are pinned through the
# reference fixture in the not-gpu suite) and vs the reference fixture directly
# ---------------------------------------------------------------------------------------------
def test_qt_linear_variants(K_):
    from tests import cpu_kernels as ck
    g = torch.Generator().manual_seed(5)
    for M in (16, 48, 160):
        x = torch.randn(M, 256, generator=g) * 3
        W = torch.randn(768, 256, generator=g) / 16
        b = torch.randn(768, generator=g)
        lw, lb = 1 + 0.1 * torch.randn(256, generator=g), 0.1 * torch.randn(256, generator=g)
        pe = torch.randn(M, 256, generator=g)
        res = torch.randn(M, 256, generator=g)
        # LN + pe + bias, xhat side output, weight row-slice view
        xh_c, xh_g = torch.empty(M, 256), torch.empty(M, 256).cuda()
        yc = ck.qt_linear(x, W[256:512], b[256:512], ln=(lw, lb), pe=pe, xhat_out=xh_c)
        Wg, bg = W.cuda(), b.cuda()
        yg = K_.qt_linear(x.cuda(), Wg[256:512], bg[256:512], ln=(lw.cuda(), lb.cuda()), pe=pe.cuda(), xhat_out=xh_g)
        assert torch.allclose(yg.cpu(), yc, rtol=1e-4, atol=1e-4)
        assert torch.allclose(xh_g.cpu(), xh_c, rtol=1e-5, atol=1e-5)
        # residual, no LN
        yc = ck.qt_linear(x, W[:256], b[:256], residual=res)
        yg = K_.qt_linear(x.cuda(), Wg[:256], bg[:256], residual=res.cuda())
        assert torch.allclose(yg.cpu(), yc, rtol=1e-4, atol=1e-4)
        # FFN shapes: 256 -> 2048 relu with LN; 2048 -> 256 with residual
        W1 = torch.randn(2048, 256, generator=g) / 16
        b1 = torch.randn(2048, generator=g)
        W2 = torch.randn(256, 2048, generator=g) / 45
        hc = ck.qt_linear(x, W1, b1, ln=(lw, lb), relu=True)
        hg = K_.qt_linear(x.cuda(), W1.cuda(), b1.cuda(), ln=(lw.cuda(), lb.cuda()), relu=True)
        assert torch.allclose(hg.cpu(), hc, rtol=1e-4, atol=1e-4)
        yc = ck.qt_linear(hc, W2, b[:256], residual=x)
        yg = K_.qt_linear(hg, W2.cuda(), bg[:256], residual=x.cuda())
        assert torch.allclose(yg.cpu(), yc, rtol=1e-4, atol=2e-4)
        # summary normalisation + embedding residual broadcast over objects
        summ = torch.randn(M, 257, generator=g)
        summ[:, -1] = summ[:, -1].abs() + 0.5
        emb = torch.randn(16, 256, generator=g)
        yc = ck.qt_linear(summ, W[:256], b[:256], summary_norm=True, residual=emb, residual_mod=16)
        yg = K_.qt_linear(summ.cuda(), Wg[:256], bg[:256], summary_norm=True, residual=emb.cuda(), residual_mod=16)
        assert torch.allclose(yg.cpu(), yc, rtol=1e-4, atol=1e-4)


def test_qt_head_fold_and_self_attention(K_):
    from tests import cpu_kernels as ck
    g = torch.Generator().manual_seed(6)
    M = 48
    a = torch.randn(M, 256, generator=g)
    W = torch.randn(768, 256, generator=g) / 16
    bias = torch.randn(256, generator=g)
    for tr in (False, True):
        oc, dc = ck.qt_head_fold(a, W[256:512], transpose_w=tr, scale=0.37, bias_vec=bias)
        og, dg = K_.qt_head_fold(a.cuda(), W.cuda()[256:512], transpose_w=tr, scale=0.37, bias_vec=bias.cuda())
        assert torch.allclose(og.cpu(), oc, rtol=1e-4, atol=1e-5)
        assert torch.allclose(dg.cpu(), dc, rtol=1e-4, atol=1e-5)
    qk = torch.randn(M, 512, generator=g) * 2
    v = torch.randn(M, 256, generator=g)
    assert torch.allclose(K_.qt_self_attention(qk.cuda(), v.cuda(), 16).cpu(), ck.qt_self_attention(qk, v, 16),
                          rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize('B,K,HW', [(1, 3, 1620), (2, 2, 60), (1, 1, 33)])
def test_qt_aux_mask(K_, B, K, HW):
    from tests import cpu_kernels as ck
    g = torch.Generator().manual_seed(7)
    pix = torch.randn(B * K, 256, HW, generator=g) * 2
    w = torch.randn(256, generator=g) / 8
    b = torch.randn(1, generator=g)
    lc, fc, cc = ck.qt_aux_mask(pix, w, b, B, K)
    lg, fg, cg = K_.qt_aux_mask(pix.cuda(), w.cuda(), b.cuda(), B, K)
    assert torch.allclose(lg.cpu(), lc, rtol=1e-4, atol=1e-4)
    # the foreground bit may legitimately differ only where two log-odds are within rounding of each other
    diff = (fg.cpu() != fc)
    if diff.any():
        p = lc.sigmoid()
        allp = torch.cat([torch.prod(1 - p, 1, keepdim=True), p], 1).clamp(1e-7, 1 - 1e-7)
        lo = torch.log(allp / (1 - allp))
        top2 = lo.topk(2, dim=1)[0]
        near = (top2[:, 0] - top2[:, 1]).abs() < 1e-4
        assert (diff.any(1) <= near).all()
    assert (cg.cpu() == fg.cpu().reshape(B * K, HW).sum(1).int()).all()


@pytest.mark.parametrize('BK,HW,case', [(3, 1620, 'mixed'), (2, 60, 'mixed'), (2, 77, 'nofg'), (1, 40, 'allfg'), (2, 77, 'mixed'),
                                        (5, 3600, 'mixed'), (1, 129, 'mixed'), (1, 64, 'allfg')])
def test_qt_cross_attention_kernels(K_, BK, HW, case):
    from tests import cpu_kernels as ck
    g = torch.Generator().manual_seed(8)
    M = BK * 16
    qfold = torch.randn(M, 8, 256, generator=g) / 8
    pix = torch.randn(BK, 256, HW, generator=g) * 2
    pe = torch.randn(BK, 256, HW, generator=g)
    if case == 'mixed':
        fg = (torch.rand(BK, HW, generator=g) > 0.6).to(torch.uint8)
    elif case == 'nofg':
        fg = torch.zeros(BK, HW, dtype=torch.uint8)
    else:
        fg = torch.ones(BK, HW, dtype=torch.uint8)
    if case == 'mixed' and BK > 1:
        fg[1] = 0                                    # one object without any foreground pixel
    cnt = fg.sum(1).int()
    W = torch.randn(768, 256, generator=g) / 16
    b = torch.randn(768, generator=g)
    ac = ck.qt_pixel_to_query(qfold, pix, pe, fg.view(1, BK, HW), cnt, W[512:], b[512:], 16)
    ag = K_.qt_pixel_to_query(qfold.cuda(), pix.cuda(), pe.cuda(), fg.cuda().view(1, BK, HW), cnt.cuda(),
                              W.cuda()[512:], b.cuda()[512:], 16)
    assert torch.allclose(ag.cpu(), ac, rtol=2e-4, atol=2e-4)
    kfold = torch.randn(M, 8, 256, generator=g) / 8
    kdots = torch.randn(M, 8, generator=g)
    vfold = torch.randn(M, 8, 256, generator=g) / 4
    ob = torch.randn(256, generator=g)
    oc = ck.qt_query_to_pixel(kfold, kdots, vfold, ob, pix, pe, 16)
    og = K_.qt_query_to_pixel(kfold.cuda(), kdots.cuda(), vfold.cuda(), ob.cuda(), pix.cuda(), pe.cuda(), 16)
    assert torch.allclose(og.cpu(), oc, rtol=2e-4, atol=2e-4)


def test_query_transformer_vs_reference_fixture(K_):
    """Whole QueryTransformer.forward on the GPU kernels vs the reference's recorded outputs."""
    from cutie_b200.config import default_config
    from cutie_b200.model.cutie import CUTIE
    from oracle.synth import synthetic_state_dict
    g = np.load(os.path.join(GOLDEN, 'qt_module.npz'))
    cfg = default_config()
    net = CUTIE(cfg).eval()
    net.load_state_dict(synthetic_state_dict(net.state_dict(), 0))
    qt = net.object_transformer.cuda()
    torch.backends.cudnn.allow_tf32 = False      # the 1x1 / 3x3 convs inside the transformer stay cuDNN
    with torch.inference_mode():
        out, aux = qt(torch.from_numpy(g['pixel']).cuda(), torch.from_numpy(g['obj_summaries']).cuda())
    ref = torch.from_numpy(g['out'])
    err = float((out.cpu() - ref).abs().max())
    assert err < 5e-4 * max(1.0, float(ref.abs().max())), err
    for i in range(4):
        assert torch.allclose(aux['logits'][i].cpu(), torch.from_numpy(g[f'aux_logits_{i}']), atol=1e-3)


@pytest.mark.timeout(300)
@pytest.mark.parametrize('K,h,w', [(3, 30, 54), (1, 7, 5), (5, 45, 80)])
def test_query_chain_is_bit_identical_to_the_separate_launches(K_, K, h, w):
    """cutie_qt_chain (persistent grid, grid barriers between phases) runs the stand-alone kernels' bodies: the whole
    QueryTransformer.forward must come out bit-identical with the chain on and off, repeatedly (the barrier counters must
    return to zero after every launch), and inside a CUDA graph replay."""
    import cutie_b200.model.object_transformer as ot
    from cutie_b200.config import default_config
    from cutie_b200.model.cutie import CUTIE
    from oracle.synth import synthetic_state_dict
    cfg = default_config()
    net = CUTIE(cfg).eval()
    net.load_state_dict(synthetic_state_dict(net.state_dict(), 0))
    qt = net.object_transformer.cuda()
    torch.backends.cudnn.allow_tf32 = False
    g = torch.Generator().manual_seed(K)
    pixel = torch.randn(1, K, 256, h, w, generator=g).cuda()
    summ = (torch.rand(1, K, 1, 16, 257, generator=g) + 0.1).cuda()
    old = ot.QT_CHAIN
    try:
        with torch.inference_mode():
            ot.QT_CHAIN = False
            want, aux_w = qt(pixel, summ)
            ot.QT_CHAIN = True
            before = K_.LAUNCH_COUNT
            got, aux_g = qt(pixel, summ)
            chained_launches = K_.LAUNCH_COUNT - before
            for _ in range(3):
                again, _ = qt(pixel, summ)
                assert torch.equal(again, got)
            torch.cuda.synchronize()
            assert torch.equal(got, want), float((got - want).abs().max())
            for a, b in zip(aux_g['logits'], aux_w['logits']):
                assert torch.equal(a, b)
            assert torch.equal(K_._QT_SYNC[pixel.device.index].cpu(), torch.zeros(4, dtype=torch.int32))
            # 4 chain launches + 3 x (p2q tiles, q2p) + 4 aux masks + the convolutions' own kernels
            assert chained_launches < 41
            graph = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                qt(pixel, summ)
            torch.cuda.current_stream().wait_stream(side)
            with torch.cuda.graph(graph):
                cap, _ = qt(pixel, summ)
            for _ in range(3):
                graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(cap, want)
    finally:
        ot.QT_CHAIN = old


@pytest.mark.parametrize('B,K,C,h,w', [(1, 3, 256, 30, 54), (2, 2, 16, 7, 5), (1, 1, 8, 1, 1), (1, 3, 256, 60, 108)])
def test_upsample2x_add_matches_aten(K_, B, K, C, h, w):
    """Mask decoder UpsampleBlock input (modules.py:15-19): bilinear x2 (align_corners=False) + skip broadcast."""
    g_ = torch.Generator().manual_seed(1)
    g = torch.randn(B, K, C, h, w, generator=g_).cuda()
    skip = torch.randn(B, C, 2 * h, 2 * w, generator=g_).cuda()
    out = K_.upsample2x_add(g, skip)
    up = torch.nn.functional.interpolate(g.flatten(0, 1), scale_factor=2, mode='bilinear', align_corners=False)
    want = up.reshape(B, K, C, 2 * h, 2 * w) + skip.unsqueeze(1)
    assert out.shape == want.shape
    torch.testing.assert_close(out, want, rtol=0, atol=2e-6)


def test_prob_to_mask_matches_argmax_and_lut(K_):
    """InferenceCore.output_prob_to_mask (inference_core.py:377-385, object_manager.py:99-104) as one kernel,
    on a strided (un-padded) view, with exact ties (first maximum wins like torch.argmax)."""
    g_ = torch.Generator().manual_seed(3)
    full = torch.rand(4, 480, 864, generator=g_).cuda()
    full[1, 10:20] = full[2, 10:20]                       # exact ties between channels 1 and 2
    full[0, 30:40] = 2.0
    full[3, 30:40] = 2.0                                  # tie between first and last channel
    prob = full[:, :, 5:859]                              # [4, 480, 854] view: row stride 864
    lut = torch.tensor([0, 7, 3, 11], dtype=torch.int64).cuda()
    out = K_.prob_to_mask(prob, lut)
    want = lut[torch.argmax(prob, dim=0)]
    assert out.dtype == torch.int64 and torch.equal(out, want)
