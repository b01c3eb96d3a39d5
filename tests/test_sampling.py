"""Per-segment sampling (SURVEY.md §8 f2: sparse_sample / NAG.get_sampling / SampleSubNodes /
SampleSegments).  Deterministic parts are held bit-exactly to vectors produced by the
reference's own files (tests/golden/sampling.pt, oracle/make_golden_select.py); the random
draw is held to the sampling law (the reference's random stream cannot be reproduced)."""
import os

import pytest
import torch

from oracle import sampling as OS
from superpoint_transformer_b200 import ops
from superpoint_transformer_b200.transforms import (SampleSubNodes, SampleSegments, SampleEdges,
                                                   NAGRestrictSize, RestrictSize,
                                                   SampleRadiusSubgraphs, SampleKHopSubgraphs)

from test_select import (assert_level_equal, levels_of, to_product, oracle_primitives,  # noqa
                         GOLDEN as SELECT_GOLDEN)

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden', 'sampling.pt')


@pytest.fixture(scope='module')
def gold():
    return torch.load(GOLDEN, weights_only=False)


@pytest.fixture(scope='module')
def nags():
    return torch.load(SELECT_GOLDEN, weights_only=False)['nags']


def check_draw(case, samples, ptr):
    """what every valid draw satisfies: the reference's counts, distinct elements of the right
    segment, inside the mask, segments ascending"""
    idx, mask = case['idx'], case['mask']
    assert torch.equal(ptr, case['ptr_samples'])
    assert samples.shape == case['idx_samples'].shape
    assert samples.unique().numel() == samples.numel()
    sizes = ptr[1:] - ptr[:-1]
    seg = torch.arange(sizes.shape[0]).repeat_interleave(sizes)
    assert torch.equal(idx[samples], seg)
    if mask is not None:
        allowed = torch.zeros(idx.shape[0], dtype=torch.bool)
        allowed[mask] = True
        assert allowed[samples].all()


# ----------------------------------------------------------------------------- CPU
def test_oracle_sparse_sample_counts_match_reference(gold):
    g = torch.Generator().manual_seed(0)
    for case in gold['sparse']:
        check_draw(case, case['idx_samples'], case['ptr_samples'])      # the reference itself
        samples, ptr = OS.sparse_sample(case['idx'], case['n_max'], case['n_min'], case['mask'],
                                        generator=g)
        check_draw(case, samples, ptr)


def test_product_sampling_counts_match_reference(gold):
    """ops.sampling_counts (the fp32 tanh heuristic, plain tensor ops) gives the reference's
    number of samples per segment on the unmasked cases."""
    for case in gold['sparse']:
        if case['mask'] is not None:
            continue
        size = case['idx'].bincount()
        n = ops.sampling_counts(size, case['n_max'], case['n_min'])
        assert torch.equal(n, case['ptr_samples'][1:] - case['ptr_samples'][:-1])


def test_host_logic_sample_segments_matches_reference(gold, nags, oracle_primitives):
    """Same torch seed, CPU tensors, device primitives stood in by the oracle: the weights must
    be the reference's to the bit for torch.multinomial to keep the same nodes."""
    for case in gold['segments']:
        spec = nags[case['nag']]
        nag = to_product(spec['levels'], spec['start'])
        torch.manual_seed(case['seed'])
        res = SampleSegments(ratio=case['ratio'], by_size=case['by_size'],
                             by_class=case['by_class'])(nag)
        for j, (a, b) in enumerate(zip(levels_of(res), case['out'])):
            # attributes the reference lost across levels (DESIGN.md §3.8) are not compared
            a = {k: v for k, v in a.items() if k in b}
            assert_level_equal(a, b, f"{case['nag']} ratio={case['ratio']} level {j}",
                               canonical_sub=True)


def test_host_logic_restrict_size_matches_reference(gold, nags, oracle_primitives):
    for case in gold['restrict']:
        spec = nags[case['nag']]
        nag = to_product(spec['levels'], spec['start'])
        torch.manual_seed(case['seed'])
        res = NAGRestrictSize(level=case['level'], num_nodes=case['num_nodes'],
                              num_edges=case['num_edges'])(nag)
        for j, (a, b) in enumerate(zip(levels_of(res), case['out'])):
            a = {k: v for k, v in a.items() if k in b}
            assert_level_equal(a, b, f"{case['nag']} level={case['level']} level {j}",
                               canonical_sub=True)
    # Data-level variant: node and edge budgets are met, edges stay inside the selection
    spec = nags['full4']
    torch.manual_seed(0)
    d = RestrictSize(num_nodes=20, num_edges=15)(to_product(spec['levels'], 0)[1])
    assert d.num_nodes == 20 and d.num_edges <= 15 and int(d.edge_index.max()) < 20
    assert d.edge_attr.shape[0] == d.num_edges


def check_sample_edges(gold, nags, device):
    for case in gold['edges']:
        spec = nags[case['nag']]
        nag = to_product(spec['levels'], spec['start'], device)
        before = [None if nag[i].edge_index is None else
                  (nag[i].edge_index.clone(), nag[i].edge_attr.clone()) for i in nag.level_range]
        res = SampleEdges(level=case['level'], n_min=case['n_min'], n_max=case['n_max'],
                          seed=3)(nag)
        assert res is nag                                    # in place, like the reference
        for j, want in enumerate(case['degree']):
            d = res[j + spec['start']]
            if want is None:
                assert d.edge_index is None
                continue
            got = torch.bincount(d.edge_index[0], minlength=d.num_nodes).cpu()
            assert torch.equal(got, want)                    # the reference's count per node
            # every kept edge is an input edge and carries its own attributes
            ei, ea = before[j]
            n = d.num_nodes
            key_in = (ei[0] * n + ei[1]).cpu()
            key_out = (d.edge_index[0] * n + d.edge_index[1]).cpu()
            assert torch.isin(key_out, key_in).all()
            rows = {(int(k), tuple(r.tolist())) for k, r in zip(key_in, ea.cpu())}
            assert all((int(k), tuple(r.tolist())) in rows
                       for k, r in zip(key_out, d.edge_attr.cpu()))


def test_host_logic_sample_edges_degrees_match_reference(gold, nags, oracle_primitives):
    check_sample_edges(gold, nags, 'cpu')
    with pytest.raises(NotImplementedError):
        SampleEdges(n_min=[1, 2], n_max=4)


def subgraph_case(case, nags, device, seeds=None):
    """Run the product transform of a golden subgraph case; `seeds`: use these seed nodes
    instead of drawing (GPU runs reuse the CPU draw: torch's CUDA generator is another stream)."""
    spec = nags[case['nag']]
    nag = to_product(spec['levels'], spec['start'], device)
    if case['batches'] is not None:
        for i, b in enumerate(case['batches']):
            nag[i].batch = b.to(device)
    cls = SampleKHopSubgraphs if case['kind'] == 'khop' else SampleRadiusSubgraphs
    t = cls(disjoint=False, **case['kw'])
    drawn = []
    draw = t.seeds
    t.seeds = (lambda n, i: (drawn.append(draw(n, i)) or drawn[-1])) if seeds is None \
        else (lambda n, i: seeds.to(device))
    torch.manual_seed(case['seed'])
    res = t(nag)
    return res, (drawn[0] if drawn else seeds)


def check_subgraph(case, res):
    want = case['out']
    got = levels_of(res)
    if case['batches'] is not None:
        assert all('batch' in a for a in got)
    for j, (a, b) in enumerate(zip(got, want)):
        a = {k: v for k, v in a.items() if k in b}
        assert_level_equal(a, b, f"{case['nag']} {case['kind']} {case['kw']} level {j}",
                           canonical_sub=True)


def test_host_logic_subgraph_sampling_matches_reference(gold, nags, oracle_primitives):
    assert len(gold['subgraphs']) >= 10
    for case in gold['subgraphs']:
        res, _ = subgraph_case(case, nags, 'cpu')
        check_subgraph(case, res)
    # disjoint: a NAGBatch with one item per seed, each equal to the single-seed selection
    case = gold['subgraphs'][1]
    spec = nags[case['nag']]
    nag = to_product(spec['levels'], spec['start'])
    torch.manual_seed(3)
    t = SampleRadiusSubgraphs(r=0.3, i_level=1, k=3, disjoint=True)
    res = t(nag)
    assert res[1].batch is not None and int(res[1].batch.max()) == 2
    torch.manual_seed(3)
    seeds = t.seeds(nag, 1)
    sizes = [nag.select(1, OS.radius_nodes(nag[1].pos, s.view(1), 0.3))[1].num_nodes
             for s in seeds]
    assert torch.bincount(res[1].batch).tolist() == sizes
    # r <= 0 / hops < 0: untouched
    assert levels_of(SampleRadiusSubgraphs(r=0, disjoint=False)(nag))[1].keys() == \
        levels_of(nag)[1].keys()
    with pytest.raises(ValueError):
        SampleKHopSubgraphs(i_level=7)(nag)


def test_sampling_without_label_histograms(nags, oracle_primitives):
    """Levels without `y` (the synthetic benchmark partitions): by_class has nothing to use and
    the weights stay uniform (+ size term), as with the reference's `Data.y is None`."""
    spec = nags['full4']
    levels = [{k: v for k, v in lv.items() if k != 'y'} for lv in spec['levels']]
    nag = to_product(levels, spec['start'])
    for by_class in (False, True):
        t = SampleSegments(0.25, by_size=True, by_class=by_class)
        want = OS.segment_weights(None, nag.get_sub_size(2, low=0), True, by_class)
        assert torch.equal(t.weights(nag, 2), want)
        torch.manual_seed(0)
        out = t(nag)
        assert out[3].num_nodes == 3 and 'y' not in out[1]
        torch.manual_seed(0)
        sub = SampleRadiusSubgraphs(r=0.3, i_level=1, k=2, by_class=by_class,
                                    disjoint=False)(nag)
        assert 0 < sub[1].num_nodes <= nag[1].num_nodes


def test_segment_weights_match_oracle(nags, oracle_primitives):
    spec = nags['full4']
    nag = to_product(spec['levels'], spec['start'])
    for by_size in (False, True):
        for by_class in (False, True):
            t = SampleSegments(0.2, by_size=by_size, by_class=by_class)
            for i_level in (1, 2, 3):
                want = OS.segment_weights(nag[i_level].y, nag.get_sub_size(i_level, low=0),
                                          by_size, by_class)
                assert torch.equal(t.weights(nag, i_level), want)


def test_sample_sub_nodes_identity_and_cpu_refusal(nags):
    spec = nags['two']
    nag = to_product(spec['levels'], spec['start'])
    assert SampleSubNodes(high=1, low=1)(nag) is nag
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        SampleSubNodes(high=1, low=0)(nag)


# ----------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_gpu_sparse_sample_counts_and_validity(gold):
    for case in gold['sparse']:
        mask = None if case['mask'] is None else case['mask'].cuda()
        samples, ptr = ops.sparse_sample(case['idx'].cuda(), case['n_max'], case['n_min'], mask,
                                         return_pointers=True, seed=7)
        check_draw(case, samples.cpu(), ptr.cpu())
        again = ops.sparse_sample(case['idx'].cuda(), case['n_max'], case['n_min'], mask, seed=7)
        assert torch.equal(again, samples)                       # (seed, input) -> output
        if samples.numel() < case['idx'].numel() // 2 and samples.numel() > 8:
            other = ops.sparse_sample(case['idx'].cuda(), case['n_max'], case['n_min'], mask,
                                      seed=8)
            assert not torch.equal(other, samples)
        # candidate order inside a segment (the documented difference from the reference)
        s, p = samples.cpu(), ptr.cpu()
        for g in range(min(p.numel() - 1, 50)):
            seg = s[p[g]:p[g + 1]]
            assert torch.equal(seg, seg.sort().values) or case['mask'] is not None


@pytest.mark.gpu
def test_gpu_sample_edges_and_restrict_size(gold, nags):
    check_sample_edges(gold, nags, 'cuda')
    spec = nags['full4']
    res = NAGRestrictSize(level='1+', num_nodes=30, num_edges=50)(
        to_product(spec['levels'], 0, 'cuda'))
    for i in (1, 2, 3):
        assert res[i].num_nodes <= 30 and res[i].num_edges <= 50
        assert res[i].edge_attr.shape[0] == res[i].num_edges
    for i in (0, 1, 2):
        assert int(res[i].super_index.max()) + 1 == res[i + 1].num_nodes
        assert torch.equal(res[i + 1].sub.to_super_index(), res[i].super_index)


@pytest.mark.gpu
def test_gpu_subgraph_sampling_matches_reference_vectors(gold, nags, monkeypatch):
    """Seeds drawn on the CPU (same torch seed as the reference run), neighbour search and
    selection on the device: the reference's output, bit for bit."""
    for case in gold['subgraphs']:
        with monkeypatch.context() as m:          # CPU draw through the oracle stand-ins
            for name, fn in (('radius_nodes', OS.radius_nodes), ('khop_nodes', OS.khop_nodes)):
                m.setattr(ops, name, fn)
            spec = nags[case['nag']]
            nag = to_product(spec['levels'], spec['start'])
            if case['batches'] is not None:
                for i, b in enumerate(case['batches']):
                    nag[i].batch = b
            cls = SampleKHopSubgraphs if case['kind'] == 'khop' else SampleRadiusSubgraphs
            torch.manual_seed(case['seed'])
            i_level = case['kw']['i_level']
            seeds = cls(disjoint=False, **case['kw']).seeds(nag, i_level)
        res, _ = subgraph_case(case, nags, 'cuda', seeds=seeds)
        check_subgraph(case, res)


@pytest.mark.gpu
def test_gpu_radius_and_khop_search_vs_oracle():
    g = torch.Generator().manual_seed(21)
    n = 50_000
    pos = torch.rand(n, 3, generator=g) * torch.tensor([20.0, 20.0, 4.0])
    batch = (pos[:, 0] > 10).long() + 2 * (pos[:, 1] > 10).long()
    seeds = torch.randperm(n, generator=g)[:5]
    for r, cyl, b, k_max in ((1.5, False, None, 10000), (2.0, True, None, 10000),
                             (2.5, False, batch, 10000), (3.0, True, batch, 10000),
                             (3.0, False, None, 150), (0.01, False, None, 10000)):
        want = OS.radius_nodes(pos, seeds, r, k_max=k_max, batch=b, cylindrical=cyl)
        got = ops.radius_nodes(pos.cuda(), seeds.cuda(), r, k_max=k_max,
                               batch=None if b is None else b.cuda(), cylindrical=cyl)
        if not torch.equal(got.cpu(), want):
            # only nodes sitting on the sphere to within fp32 rounding may differ (the device
            # evaluates sqrt(dx^2+dy^2+dz^2) unfused; torch's CPU norm may round differently)
            a, w = set(got.cpu().tolist()), set(want.tolist())
            m = torch.tensor([1.0, 1.0, 0.0 if cyl else 1.0])
            for i in a ^ w:
                d = ((pos[i] - pos[seeds]) * m).double().norm(dim=1)
                assert ((d - r).abs() < 1e-5 * r).any(), (r, cyl, k_max, i)
    ei = torch.randint(0, n, (2, 4 * n), generator=g)
    for hops in (0, 1, 2, 3):
        want = OS.khop_nodes(ei, seeds, hops, n)
        got = ops.khop_nodes(ei.cuda(), seeds.cuda(), hops, n)
        assert torch.equal(got.cpu(), want), hops


@pytest.mark.gpu
def test_gpu_sparse_sample_is_uniform_short_segments():
    """20 000 segments of 6 elements, 3 drawn from each: the 20 possible subsets must be
    equally likely (chi-square, 19 degrees of freedom; fixed seed)."""
    G, size = 20000, 6
    idx = torch.arange(G).repeat_interleave(size).cuda()
    samples, ptr = ops.sparse_sample(idx, n_max=4, n_min=1, return_pointers=True,
                                     num_segments=G, seed=123)
    assert int(ptr[-1]) == 3 * G                                 # floor(4 tanh(6/4)) = 3
    local = (samples.view(G, 3) % size).cpu()
    code = (2 ** local).sum(dim=1)
    counts = torch.bincount(code, minlength=64)
    counts = counts[counts > 0]
    assert counts.numel() == 20
    chi2 = float(((counts - G / 20.0) ** 2 / (G / 20.0)).sum())
    assert chi2 < 50.0, chi2                                     # p ~ 1e-4 at 19 dof


@pytest.mark.gpu
def test_gpu_sparse_sample_is_uniform_long_segments():
    """2 000 segments of 300 elements (the warp / radix-select path), 32 drawn from each: every
    position is kept with probability 32/300, and pairs of neighbours are not correlated."""
    G, size = 2000, 300
    k = int(ops.sampling_counts(torch.tensor([size], device='cuda'), 32, 1))   # 32 (or 31)
    idx = torch.arange(G).repeat_interleave(size).cuda()
    samples, ptr = ops.sparse_sample(idx, n_max=32, n_min=1, return_pointers=True,
                                     num_segments=G, seed=99)
    assert int(ptr[-1]) == k * G
    local = (samples.view(G, k) % size).cpu()
    assert (local[:, 1:] > local[:, :-1]).all()                  # distinct, candidate order
    counts = torch.bincount(local.flatten(), minlength=size).double()
    expect = G * k / size
    chi2 = float(((counts - expect) ** 2 / (expect * (1 - k / size))).sum())
    assert 200.0 < chi2 < 420.0, chi2                            # 299 dof, mean 299, sd 24.5
    kept = torch.zeros(G, size)
    kept.scatter_(1, local, 1.0)
    both = float((kept[:, 1:] * kept[:, :-1]).mean())
    want = k * (k - 1) / (size * (size - 1))
    assert abs(both - want) < 6 * (want / (G * (size - 1))) ** 0.5 + 1e-4


def check_synthetic_partition(nag):
    """SampleSubNodes / SampleSegments on a partition of the synthetic generator (levels 1-3, no
    label histograms, level-1 `node_size`)."""
    sizes = torch.bincount(nag[1].super_index, minlength=nag[2].num_nodes)
    out = SampleSubNodes(high=2, low=1, n_max=4, n_min=2, seed=5)(nag)
    want = OS.sampling_counts(sizes.cpu(), 4, 2)
    got = torch.bincount(out[1].super_index, minlength=out[2].num_nodes).cpu()
    assert torch.equal(got, want)                # every level-2 node keeps the reference's count
    assert out[2].num_nodes == nag[2].num_nodes and out[3].num_nodes == nag[3].num_nodes
    assert torch.equal(out[2].sub.to_super_index(), out[1].super_index)
    assert int(out[1].edge_index.max()) < out[1].num_nodes
    # the kept level-1 nodes carry their own attributes (pos is unique per node)
    assert torch.isin(out[1].pos[:, 0], nag[1].pos[:, 0]).all()

    torch.manual_seed(0)
    res = SampleSegments(ratio=[0.2, 0.5, 0.1], by_size=True, by_class=False)(nag)
    n3 = nag[3].num_nodes - int(nag[3].num_nodes * 0.1)
    assert res[3].num_nodes <= n3      # (a node that loses every child later goes too)
    for i in (1, 2):
        assert int(res[i].super_index.max()) + 1 == res[i + 1].num_nodes
        assert torch.equal(res[i + 1].sub.to_super_index(), res[i].super_index)
    assert res[2].num_nodes <= nag[2].num_nodes - int(nag[2].num_nodes * 0.5)


@pytest.mark.gpu
def test_gpu_sample_sub_nodes_and_segments_on_benchmark_partition():
    from superpoint_transformer_b200.synthetic import make_nag, CONFIGS
    check_synthetic_partition(make_nag(**CONFIGS['cfg2']).cuda())


def test_host_logic_sample_sub_nodes_and_segments_on_synthetic_partition(oracle_primitives):
    """The same checks on CPU tensors (device primitives stood in by the oracle): what the GPU
    test exercises above the kernels."""
    from superpoint_transformer_b200.synthetic import make_nag
    check_synthetic_partition(make_nag([6000, 1200, 240], mean_degree=8, seed=4))
