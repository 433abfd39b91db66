"""tcgen05 FP16 candidate filter over the bank's key operand image + exact re-rank: the image layout, and bit-identity of
the filtered path with the exact fp32 scan."""
import pytest
import torch

from oracle import memory_math as mm
from tests.test_gpu_kernels import K_, check_topk, segments_of  # noqa: F401

pytestmark = pytest.mark.gpu


@pytest.fixture
def tc_everywhere(K_):
    K_.set_tc_min_tokens(256)
    yield
    K_.set_tc_min_tokens(-1)


@pytest.mark.parametrize('B,N,Q,K,top_k,cuts', [
    (1, 333, 77, 2, 30, ()),                   # three image tiles
    (2, 1000, 130, 2, 30, (128, 500, 501)),    # four segments, batch 2
    (1, 4099, 1620, 3, 30, (4000,)),           # 480p query count
    (1, 5000, 300, 1, 64, (100,)),             # kpad 64
    (1, 70001, 96, 1, 30, (1620, 30000)),      # three segments
])
def test_fp16_filter_matches_oracle_and_exact_scan(K_, tc_everywhere, B, N, Q, K, top_k, cuts):
    assert K_.affinity_plan(N, top_k) == 1
    before = K_.image_level_launches()
    idx_tc, w_tc = check_topk(K_, B, N, Q, K, top_k, cuts)          # all oracle assertions on the filtered path
    assert K_.image_level_launches() == before + 1, 'the FP16 image plan did not run'
    K_.set_tc_min_tokens(1 << 40)                                   # same inputs through the exact scan only
    assert K_.affinity_plan(N, top_k) == 0
    idx_ex, w_ex = check_topk(K_, B, N, Q, K, top_k, cuts)
    assert torch.equal(idx_tc, idx_ex), 'filtered selection differs from the exact scan'
    assert torch.equal(w_tc, w_ex), 'weights are not bit-identical'


def test_filter_keeps_duplicates_and_near_duplicates(K_, tc_everywhere):
    """Near-duplicate frames (the hard case of SURVEY.md Appendix B): many tokens within FP16 noise of each other."""
    g = torch.Generator().manual_seed(2)
    base = torch.randn(1, 500, 64, generator=g) * 4
    key = torch.cat([base + 1e-3 * torch.randn(1, 500, 64, generator=g) for _ in range(8)], 1)   # 4000 tokens
    shr = 1 + torch.randn(1, 4000, generator=g) ** 2
    vals = [torch.randn(1, 4000, 256, generator=g)]
    qk = base[:, :200].transpose(1, 2).contiguous() + 1e-3 * torch.randn(1, 64, 200, generator=g)
    qe = torch.sigmoid(torch.randn(1, 64, 200, generator=g))
    segs = segments_of(K_, key, shr, vals, (1500,))
    assert K_.affinity_plan(4000, 30) == 1
    before = K_.image_level_launches()
    idx, w, sim = K_.affinity_topk(segs, qk.cuda(), qe.cuda(), 30, want_sim=True)
    assert K_.image_level_launches() == before + 1, 'the FP16 image plan did not run'
    K_.set_tc_min_tokens(1 << 40)
    idx2, w2, sim2 = K_.affinity_topk(segs, qk.cuda(), qe.cuda(), 30, want_sim=True)
    assert torch.equal(idx, idx2) and torch.equal(w, w2) and torch.equal(sim, sim2)


# ---------------------------------------------------------------------------------------------------------
# key image layout and the image plan's edge cases
# ---------------------------------------------------------------------------------------------------------
def _image_offsets(row, elem):
    """Byte offset of FP16 operand element `elem` (0..143) of token row `row` inside a 36864-byte tile
    (csrc/tc_operand_f16.cuh: 2 SWIZZLE_128B K-blocks of 64 f16 + one un-swizzled 16-element tail block)."""
    if elem < 128:
        blk, w = elem >> 6, elem & 63
        return blk * 16384 + row * 128 + (((w >> 3) ^ (row & 7)) << 4) + (w & 7) * 2
    e = elem - 128
    return 2 * 16384 + (e >> 3) * 2048 + (row >> 3) * 128 + (row & 7) * 16 + (e & 7) * 2


def test_key_image_layout_and_values(K_):
    g = torch.Generator().manual_seed(3)
    B, cap = 2, 1000
    key = (torch.randn(B, cap, 64, generator=g) * 2).cuda()
    shr = (1 + torch.randn(B, cap, generator=g) ** 2).cuda()
    key[0, 100] *= 200.0                               # shr k^2 beyond the f16 range: a flagged ("always candidate") row
    tiles = K_.key_image_tiles(cap)
    img = torch.full((B, tiles, K_.KEY_IMAGE_FLOATS), 7.0, device='cuda')
    p0, n = 77, 600                                   # unaligned range: rows outside it must stay untouched
    K_.bank_key_image(key, shr, p0, n, img)
    untouched = torch.full((1,), 7.0).view(torch.float16)            # the two f16 halves of the fill pattern
    key, shr = key.cpu(), shr.cpu()
    flat = img.cpu().view(torch.float16).reshape(B, tiles, -1)       # [B, tiles, 18432] f16 elements
    rows = torch.arange(cap)
    t, r = rows // 128, rows % 128
    eps = 1.05e-3
    for b in range(B):
        inside = (rows >= p0) & (rows < p0 + n)
        ln = shr[b][:, None] * key[b]                                         # shr k    (fp32, same op order)
        sq = ln * key[b]                                                      # shr k^2
        sat = (torch.maximum(sq.abs().amax(1), ln.abs().amax(1)) > 60000.0)
        assert bool(sat[100]) == (b == 0)
        live = inside & ~sat
        for c in (0, 1, 7, 8, 31, 32, 63):
            for which, want in ((0, sq[:, c]), (64, ln[:, c])):
                off = torch.tensor([_image_offsets(int(x), which + c) // 2 for x in r])
                got = flat[b, t, off]
                assert torch.equal(got[live], want[live].half()), f'element {which + c}'          # round to nearest f16
                assert (got[inside & sat] == 0).all()
                assert (got[~inside] == untouched[off[~inside] % 2]).all(), 'rows outside the range were written'
        n2, n1 = key[b].double().pow(2).sum(1), key[b].double().abs().sum(1)
        P2 = shr[b].double() * n2
        tail = {0: shr[b].half().float(), 1: shr[b].half().float(), 6: torch.ones(cap), 7: torch.zeros(cap)}
        for e, want in tail.items():
            off = torch.tensor([_image_offsets(int(x), 128 + e) // 2 for x in r])
            assert torch.equal(flat[b, t, off][live].float(), want[live]), e
        for e in range(8, 16):
            off = torch.tensor([_image_offsets(int(x), 128 + e) // 2 for x in r])
            assert (flat[b, t, off][inside] == 0).all()
        # the error-bound factors are rounded AWAY from zero: never smaller than the exact ones, never more than 1 % larger
        bounds = {2: eps * P2, 3: 2 * eps * (P2 * shr[b].double()).sqrt(), 4: eps * shr[b].double(),
                  5: 2.0 ** -25 * (P2 + shr[b].double() * n1)}
        for e, exact in bounds.items():
            off = torch.tensor([_image_offsets(int(x), 128 + e) // 2 for x in r])
            got = -flat[b, t, off].double()
            assert (got[live] >= exact[live]).all(), e
            if e != 5:
                assert (got[live] <= exact[live] * 1.012 + 1e-7).all(), e
        # a flagged row: no energy terms, flag = -60000 (the filter sees D < any threshold; the sampler sees +60000)
        offF = torch.tensor([_image_offsets(int(x), 128 + 7) // 2 for x in r])
        assert (flat[b, t, offF][inside & sat].float() == -60000.0).all()


def _arena_bank(K_, B, layout, seed, centred=False):
    """layout: list of (capacity, phys_begin, n) -- one arena per entry, the segment is rows [phys, phys+n).
    centred: keys sit on a large common mean and the images are built around a key centre (as the runtime does)."""
    g = torch.Generator().manual_seed(seed)
    segs, keys, shrs = [], [], []
    offset = (torch.randn(B, 1, 64, generator=g) * 4).cuda() if centred else 0.0
    mu = (offset[:, 0] + 0.1).contiguous() if centred else None          # any vector is valid; a good one is near the mean
    for cap, p0, n in layout:
        key = (torch.randn(B, cap, 64, generator=g) * 1.5).cuda() + offset
        shr = (1 + torch.randn(B, cap, generator=g) ** 2).cuda()
        img = torch.full((B, K_.key_image_tiles(cap), K_.KEY_IMAGE_FLOATS), float('nan'), device='cuda')
        K_.bank_key_image(key, shr, p0, n, img, mu)    # everything outside the segment stays NaN on purpose
        segs.append(K_.BankSegment(key[:, p0:p0 + n], shr[:, p0:p0 + n], (), img, p0, mu))
        keys.append(key[:, p0:p0 + n]), shrs.append(shr[:, p0:p0 + n])
    return segs, torch.cat(keys, 1), torch.cat(shrs, 1)


@pytest.mark.parametrize('B,Q,top_k,layout', [
    (1, 300, 30, [(9000, 0, 9000)]),                                        # aligned, one arena
    (1, 260, 30, [(3000, 1, 2999), (20000, 12345, 7000), (20000, 0, 5001)]),    # ring wrap: tail run + head run
    (2, 130, 30, [(700, 130, 500), (8000, 127, 7000), (8000, 7999, 1), (6000, 128, 3000)]),   # 4 runs, batch 2
    (1, 96, 64, [(80000, 3, 70001)]),                                       # unaligned start, kpad 64
    (1, 1620, 30, [(420000, 1000, 413100)]),                                # BASELINE cfg 2 bank size
])
@pytest.mark.parametrize('centred', [False, True])
def test_image_plan_is_bit_identical_to_exact_scan(K_, tc_everywhere, B, Q, top_k, layout, centred):
    segs, key, shr = _arena_bank(K_, B, layout, seed=11, centred=centred)
    N = key.shape[1]
    assert K_.affinity_plan(N, top_k) == 1
    g = torch.Generator().manual_seed(5)
    qk = (torch.randn(B, 64, Q, generator=g) * 1.5).cuda() + (segs[0].key_mu[:, :, None] if centred else 0.0)
    qe = torch.sigmoid(torch.randn(B, 64, Q, generator=g)).cuda()
    before = K_.image_level_launches()
    acc = torch.zeros(B, N, dtype=torch.int64, device='cuda')
    idx, w, sim = K_.affinity_topk(segs, qk, qe, top_k, usage_acc=acc, want_sim=True)
    assert K_.image_level_launches() == before + 1, 'the FP16 image plan did not run'
    plain = [K_.BankSegment(s.key, s.shrinkage, ()) for s in segs]          # same bank without images: exact scan
    idx_p, w_p, sim_p = K_.affinity_topk(plain, qk, qe, top_k, want_sim=True)
    assert K_.image_level_launches() == before + 1
    K_.set_tc_min_tokens(1 << 40)                                           # exact fp32 scan only
    acc_x = torch.zeros(B, N, dtype=torch.int64, device='cuda')
    idx_x, w_x, sim_x = K_.affinity_topk(plain, qk, qe, top_k, usage_acc=acc_x, want_sim=True)
    for a, b_ in ((idx, idx_x), (w, w_x), (sim, sim_x), (idx_p, idx_x), (w_p, w_x), (acc, acc_x)):
        assert torch.equal(a, b_)
    # and against float64 truth: the selected set is the true top-k up to fp32 near-ties
    truth = None if N * Q > 3e8 else mm.similarity_direct(key.cpu().transpose(1, 2), shr.cpu().unsqueeze(1), qk.cpu(), qe.cpu(),
                                                         dtype=torch.float64)
    if N * Q <= 3e8:
        n_dec, n_dec_eq, _, _ = mm.topk_set_agreement(idx[:, :, :top_k].cpu().long().transpose(1, 2), truth, top_k,
                                                      rel_noise=1e-5)
        assert n_dec > 0 and n_dec_eq == n_dec


@pytest.mark.parametrize('key_scale,q_scale,note', [
    (1e-3, 1.0, 'tiny keys: shr k^2 ~ 1e-6 is an f16 subnormal (absolute error term)'),
    (40.0, 1.0, 'huge keys: some rows exceed the f16 range and are flagged always-candidate'),
    (1.0, 40.0, 'huge queries: b^2 > 3e4 does not fit f16 => those queries are re-ranked exhaustively'),
    (300.0, 1.0, 'every row flagged: the filter passes everything, the exact re-rank decides'),
])
def test_image_path_outside_the_f16_range(K_, tc_everywhere, key_scale, q_scale, note):
    g = torch.Generator().manual_seed(21)
    B, cap, Q, top_k = 1, 6000, 200, 30
    key = (torch.randn(B, cap, 64, generator=g) * key_scale).cuda()
    if key_scale == 40.0:
        key[:, ::3] /= 40.0                               # a mix of representable and flagged rows
    shr = (1 + torch.randn(B, cap, generator=g) ** 2).cuda()
    img = torch.zeros(B, K_.key_image_tiles(cap), K_.KEY_IMAGE_FLOATS, device='cuda')
    K_.bank_key_image(key, shr, 0, cap, img)
    qk = (torch.randn(B, 64, Q, generator=g) * q_scale).cuda()
    if q_scale == 40.0:
        qk[:, :, ::2] /= 40.0                             # half of the queries stay filterable
    qe = torch.sigmoid(torch.randn(B, 64, Q, generator=g)).cuda()
    seg = [K_.BankSegment(key, shr, (), img, 0)]
    idx, w, sim = K_.affinity_topk(seg, qk, qe, top_k, want_sim=True)
    K_.set_tc_min_tokens(1 << 40)
    idx_x, w_x, sim_x = K_.affinity_topk([K_.BankSegment(key, shr, ())], qk, qe, top_k, want_sim=True)
    assert torch.equal(idx, idx_x) and torch.equal(w, w_x) and torch.equal(sim, sim_x), note


@pytest.mark.parametrize('runs', [[(20000, 12345, 7000), (20000, 0, 5001)],          # 12 001 tokens
                                  [(20000, 2345, 14000), (20000, 0, 9001)]])          # 23 001 tokens
def test_threshold_seeds_never_change_the_result(K_, tc_everywhere, runs):
    """seed_idx only tightens the filter threshold: the previous winners (the runtime's use), random distinct tokens,
    partly invalid lists and the true answer itself all give the bit-identical selection (the threshold is the smaller of
    the tile-sampled bound and the seed bound; an unusable list leaves the sampled bound)."""
    segs, key, shr = _arena_bank(K_, 1, runs, seed=4, centred=True)
    N, Q, top_k = key.shape[1], 260, 30
    g = torch.Generator().manual_seed(6)
    qk = (torch.randn(1, 64, Q, generator=g) * 1.5).cuda() + segs[0].key_mu[:, :, None]
    qe = torch.sigmoid(torch.randn(1, 64, Q, generator=g)).cuda()
    idx0, w0, s0 = K_.affinity_topk(segs, qk, qe, top_k, want_sim=True)
    K_.KEEP_LAST_WORKSPACE = True
    try:
        rand = torch.stack([torch.randperm(N, generator=g)[:32] for _ in range(Q)])[None].int().cuda()
        rand[:, :, 30:] = -1
        partly = rand.clone()
        partly[:, ::3, 5] = -1                                            # every third query has an invalid seed
        partly[:, 1::3, 7] = N + 5
        counts = {}
        for name, seed in (('true winners', idx0), ('random distinct', rand), ('partly invalid', partly)):
            idx, w, s = K_.affinity_topk(segs, qk, qe, top_k, want_sim=True, seed_idx=seed.contiguous())
            assert torch.equal(idx, idx0) and torch.equal(w, w0) and torch.equal(s, s0), name
            counts[name] = float(K_.last_candidate_counts().float().mean())
        idx, _, _ = K_.affinity_topk(segs, qk, qe, top_k)
        counts['no seeds'] = float(K_.last_candidate_counts().float().mean())
    finally:
        K_.KEEP_LAST_WORKSPACE = False
    print('candidates per query:', counts)
    # the true winners give the tightest possible threshold; what is left is the FP16 error band around the k-th energy
    assert counts['true winners'] <= counts['no seeds'] and counts['true winners'] <= counts['random distinct']
