"""Node selection (SURVEY.md §8 f1: NAG.select / Data.select / Cluster.select).

CPU part: the oracle restatement (oracle/select.py) against tests/golden/select.pt — vectors
produced by the reference's own src/data/*.py (oracle/make_golden_select.py) — and the host
logic of the product's containers with the four device primitives replaced by oracle-based
stand-ins (tests may use the oracle; the product has no CPU path of its own).
GPU part: the product on CUDA tensors, through the C-ABI kernels of csrc/select.cu, against the
same vectors (bit-exact) and against the oracle on a benchmark-size partition."""
import os

import numpy as np
import pytest
import torch

from oracle import select as O
from superpoint_transformer_b200 import ops
from superpoint_transformer_b200.data import Data, NAG, Cluster

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden', 'select.pt')


@pytest.fixture(scope='module')
def gold():
    return torch.load(GOLDEN, weights_only=False)


# ----------------------------------------------------------------------------- helpers
def assert_level_equal(a, b, what, canonical_sub=False):
    """bit-exact equality of two level dicts (floats included: selection only moves data)."""
    if canonical_sub:
        a, b = O.canonical(a), O.canonical(b)
    assert sorted(a.keys()) == sorted(b.keys()), f'{what}: keys {sorted(a)} vs {sorted(b)}'
    for k in a:
        if k == 'sub':
            for f in ('pointers', 'points'):
                assert torch.equal(a[k][f], b[k][f]), f'{what}: sub.{f} differs'
        else:
            assert a[k].dtype == b[k].dtype, f'{what}: {k} dtype {a[k].dtype} vs {b[k].dtype}'
            assert torch.equal(a[k], b[k]), f'{what}: {k} differs'


def case_idx(case):
    idx = case['idx']
    return idx.numpy() if case.get('kind') == 'numpy' else idx


def to_product(levels, start, device='cpu'):
    datas = []
    for lv in levels:
        d = Data(**{k: v.to(device) for k, v in lv.items() if k != 'sub'})
        if 'sub' in lv:
            d.sub = Cluster(lv['sub']['pointers'].to(device), lv['sub']['points'].to(device))
        datas.append(d)
    return NAG(datas, start_i_level=start)


def level_of(data):
    out = {}
    for k in data.keys:
        if k.startswith('_'):
            continue
        v = data[k]
        out[k] = {'pointers': v.pointers.cpu(), 'points': v.points.cpu()} \
            if isinstance(v, Cluster) else v.cpu()
    return out


def levels_of(nag):
    return [level_of(nag[i]) for i in nag.level_range]


def idx_to(idx, device):
    return idx.to(device) if torch.is_tensor(idx) else idx


# ----------------------------------------------------------------------------- oracle vs golden
def test_oracle_nag_select_matches_reference(gold):
    for case in gold['nag_cases'] + gold['reference_drops']:
        nag = gold['nags'][case['nag']]
        out = O.nag_select(nag['levels'], nag['start'], case['i_level'], case_idx(case))
        for j, (a, b) in enumerate(zip(out, case['out'])):
            assert_level_equal(a, b, f"{case['nag']} L{case['i_level']} {case['kind']} level {j}",
                               canonical_sub=True)


def test_oracle_data_select_matches_reference(gold):
    for case in gold['data_cases']:
        nag = gold['nags'][case['nag']]
        level = nag['levels'][case['i_level'] - nag['start']]
        out, (idx_sub, sub_super), (idx_super, super_sub) = O.data_select(
            level, case['idx'], case['update_sub'], case['update_super'])
        what = f"{case['nag']} L{case['i_level']} sub={case['update_sub']} sup={case['update_super']}"
        assert_level_equal(out, case['out'], what)
        for name, mine in (('idx_sub', idx_sub), ('sub_super', sub_super),
                           ('idx_super', idx_super)):
            assert (mine is None) == (case[name] is None), f'{what}: {name}'
            if mine is not None:
                assert torch.equal(mine, case[name]), f'{what}: {name}'
        assert (super_sub is None) == (case['super_sub'] is None)
        if super_sub is not None:
            assert_level_equal({'sub': super_sub}, {'sub': case['super_sub']}, what, True)


def test_oracle_cluster_select_and_pointers_match_reference(gold):
    for case in gold['cluster_cases']:
        nag = gold['nags'][case['nag']]
        cl = nag['levels'][case['i_level'] - nag['start']]['sub']
        out, (idx_sub, sub_super) = O.cluster_select(cl, case['idx'], case['update_sub'])
        assert torch.equal(out['pointers'], case['out']['pointers'])
        assert torch.equal(out['points'], case['out']['points'])
        assert (idx_sub is None) == (case['idx_sub'] is None)
        if idx_sub is not None:
            assert torch.equal(idx_sub, case['idx_sub'])
            assert torch.equal(sub_super, case['sub_super'])
    for case in gold['pointer_cases']:
        p, v = O.index_select_pointers(case['pointers'], case['idx'])
        assert torch.equal(p, case['pointers_new']) and torch.equal(v, case['val_idx'])
    for case in gold['consecutive_cases']:
        inv, perm = O.consecutive_cluster(case['src'])
        assert torch.equal(inv, case['inv']) and torch.equal(case['src'][perm], case['unique'])


# ----------------------------------------------------------------------------- host logic (CPU)
@pytest.fixture
def oracle_primitives(monkeypatch):
    """The four device primitives of ops, stood in for by the oracle (host-logic tests only)."""
    def relabel_consecutive(ids, num_ids, payload=None):
        inv, perm = O.consecutive_cluster(ids)
        uniq = ids[perm]
        if payload is None:
            return inv, uniq
        by_new = torch.empty_like(uniq)
        by_new[inv] = payload
        return inv, uniq, by_new

    def select_edges(edge_index, idx, num_nodes):
        assert idx.unique().numel() == idx.numel() and int(idx.max()) < num_nodes
        if edge_index is None:
            return None, None
        reindex = torch.full((num_nodes,), -1, dtype=torch.int64)
        reindex[idx] = torch.arange(idx.shape[0])
        ei = reindex[edge_index]
        idx_edge = torch.where((ei != -1).all(dim=0))[0]
        return ei[:, idx_edge], idx_edge

    def csr_select(pointers, values, idx, want_group=False):
        p, v = O.index_select_pointers(pointers, idx)
        if not want_group:
            return p, values[v]
        sizes = p[1:] - p[:-1]
        return p, values[v], torch.arange(idx.shape[0]).repeat_interleave(sizes)

    def from_super_index(super_index, num_super):
        c = O.cluster_from_dense(super_index, torch.arange(super_index.shape[0]))
        return Cluster(c['pointers'], c['points'])

    def sparse_sample(idx, n_max=32, n_min=1, mask=None, return_pointers=False,
                      num_segments=None, seed=None):
        from oracle import sampling as OS
        samples, ptr = OS.sparse_sample(idx, n_max, n_min, mask)
        return (samples, ptr) if return_pointers else samples

    monkeypatch.setattr(ops, 'sparse_sample', sparse_sample)
    from oracle import sampling as OS
    monkeypatch.setattr(ops, 'radius_nodes', OS.radius_nodes)
    monkeypatch.setattr(ops, 'khop_nodes', OS.khop_nodes)
    monkeypatch.setattr(ops, 'relabel_consecutive', relabel_consecutive)
    monkeypatch.setattr(ops, 'select_edges', select_edges)
    monkeypatch.setattr(ops, 'csr_select', csr_select)
    monkeypatch.setattr(ops, 'take_rows', lambda t, idx: t[idx])
    monkeypatch.setattr(ops, 'take_rows_multi', lambda ts, idx: [t[idx] for t in ts])
    monkeypatch.setattr(Cluster, 'from_super_index', staticmethod(from_super_index))


def check_nag_cases(gold, device):
    for case in gold['nag_cases']:
        nag = gold['nags'][case['nag']]
        res = to_product(nag['levels'], nag['start'], device).select(
            case['i_level'], idx_to(case_idx(case), device))
        assert res.start_i_level == nag['start']
        for j, (a, b) in enumerate(zip(levels_of(res), case['out'])):
            assert_level_equal(a, b, f"{case['nag']} L{case['i_level']} {case['kind']} level {j}",
                               canonical_sub=True)
            # the product's own order inside a cluster is the ascending one
            assert_level_equal(a, O.canonical(a), 'ascending points inside clusters')


def check_kept_attributes(gold, device):
    """Where a neighbouring level needs no re-indexing the reference hands None across levels
    and LOSES that level's `super_index` / `sub` (nag.py:370, 383).  The product keeps them:
    every other attribute equals the reference's, the kept ones equal the input's."""
    assert len(gold['reference_drops']) > 0
    for case in gold['reference_drops']:
        nag = gold['nags'][case['nag']]
        res = to_product(nag['levels'], nag['start'], device).select(
            case['i_level'], idx_to(case_idx(case), device))
        for j, (a, b) in enumerate(zip(levels_of(res), case['out'])):
            src = nag['levels'][j]
            for k in ('super_index', 'sub'):
                if k in src and k not in b:
                    assert_level_equal({k: a.pop(k)}, {k: src[k]}, f'kept {k} of level {j}')
            assert_level_equal(a, b, f'level {j}', canonical_sub=True)


def test_host_logic_nag_select(gold, oracle_primitives):
    check_nag_cases(gold, 'cpu')
    check_kept_attributes(gold, 'cpu')


def test_host_logic_data_select_flags(gold, oracle_primitives):
    check_data_cases(gold, 'cpu')


def check_data_cases(gold, device):
    for case in gold['data_cases']:
        nag = gold['nags'][case['nag']]
        data = to_product(nag['levels'], nag['start'], device)[case['i_level']]
        out, (idx_sub, sub_super), (idx_super, super_sub) = data.select(
            case['idx'].to(device), update_sub=case['update_sub'],
            update_super=case['update_super'])
        what = f"{case['nag']} L{case['i_level']} sub={case['update_sub']} sup={case['update_super']}"
        assert isinstance(out, Data)
        assert_level_equal(level_of(out), case['out'], what)
        for name, mine in (('idx_sub', idx_sub), ('sub_super', sub_super),
                           ('idx_super', idx_super)):
            assert (mine is None) == (case[name] is None), f'{what}: {name}'
            if mine is not None:
                assert torch.equal(mine.cpu(), case[name]), f'{what}: {name}'
        assert (super_sub is None) == (case['super_sub'] is None)
        if super_sub is not None:
            mine = {'sub': {'pointers': super_sub.pointers.cpu(), 'points': super_sub.points.cpu()}}
            assert_level_equal(mine, {'sub': case['super_sub']}, what, True)


def test_select_identity_and_errors(gold, oracle_primitives):
    nag = gold['nags']['two']
    prod = to_product(nag['levels'], nag['start'])
    same = prod.select(0, torch.arange(60))
    for a, b in zip(levels_of(same), nag['levels']):
        assert_level_equal(a, b, 'identity')
    with pytest.raises(ValueError):        # like the reference, Python lists are rejected
        prod.select(0, [1, 2, 3])
    with pytest.raises(AssertionError):
        prod.select(5, torch.tensor([0]))


def test_index_helpers_follow_the_reference():
    """tensor_idx / is_arange / sizes_to_pointers / indices_to_pointers against the oracle's
    restatement and against what the reference's own tensor_idx (src/utils/tensor.py) returns
    for the same cases, recorded below."""
    from superpoint_transformer_b200.utils import (tensor_idx, is_arange, sizes_to_pointers,
                                                   indices_to_pointers)
    mask = torch.tensor([True, False, True, True])
    cases = [3, slice(2, 6), np.array([4, 1]), mask, torch.tensor([5, 0, 2], dtype=torch.int32),
             None]
    reference = [[3], [2, 3, 4, 5], [4, 1], [0, 2, 3], [5, 0, 2], None]   # all int64
    for c, want in zip(cases, reference):
        for impl in (tensor_idx, O.tensor_idx):
            got = impl(c)
            assert (got is None and want is None) or \
                (got.dtype == torch.int64 and got.tolist() == want), (impl, c)
    with pytest.raises(ValueError):
        tensor_idx([1, 2])
    assert is_arange(torch.arange(5), 5) and not is_arange(torch.arange(5), 6)
    assert not is_arange(torch.tensor([0, 2, 1]), 3) and is_arange(torch.arange(0), 0)
    sizes = torch.tensor([2, 0, 3])
    assert sizes_to_pointers(sizes).tolist() == [0, 2, 2, 5]
    ptr, order = indices_to_pointers(torch.tensor([2, 0, 2, 1, 0]))
    assert ptr.tolist() == [0, 2, 3, 5] and order.tolist() == [1, 4, 3, 0, 2]


def test_product_select_refuses_cpu_tensors(gold):
    """No CPU path in the product: the device primitives insist on CUDA tensors."""
    nag = gold['nags']['two']
    with pytest.raises(RuntimeError, match='CUDA tensors only'):
        to_product(nag['levels'], nag['start']).select(0, torch.tensor([3, 1]))


# ----------------------------------------------------------------------------- GPU: C-ABI kernels
@pytest.fixture(params=['fused', 'primitives'])
def select_path(request):
    """Data.select through one native call per level (default) or primitive by primitive."""
    prev = ops.SELECT_FUSED
    ops.set_select_fused(request.param == 'fused')
    yield request.param
    ops.set_select_fused(prev)


@pytest.mark.gpu
def test_gpu_nag_select_matches_reference_vectors(gold, select_path):
    check_nag_cases(gold, 'cuda')
    check_kept_attributes(gold, 'cuda')


@pytest.mark.gpu
def test_gpu_select_rejects_bad_indices(gold, select_path):
    nag = gold['nags']['two']
    prod = to_product(nag['levels'], nag['start'], 'cuda')
    for bad in ([1, 1], [0, 60], [-1, 3]):          # repeated / beyond the 60 nodes / negative
        with pytest.raises(IndexError):
            prod.select(0, torch.tensor(bad, device='cuda'))
    with pytest.raises(IndexError):
        prod.select(1, torch.tensor([9, 2], device='cuda'))     # level 1 has 9 nodes
    ok = prod.select(0, torch.tensor([5, 3], device='cuda'))    # the context is still healthy
    assert ok[0].num_nodes == 2


@pytest.mark.gpu
def test_gpu_data_and_cluster_select_match_reference_vectors(gold, select_path):
    check_data_cases(gold, 'cuda')
    for case in gold['cluster_cases']:
        nag = gold['nags'][case['nag']]
        cl = nag['levels'][case['i_level'] - nag['start']]['sub']
        cl = Cluster(cl['pointers'].cuda(), cl['points'].cuda())
        out, (idx_sub, sub_super) = cl.select(case['idx'].cuda(), update_sub=case['update_sub'])
        assert torch.equal(out.pointers.cpu(), case['out']['pointers'])
        assert torch.equal(out.points.cpu(), case['out']['points'])
        assert (idx_sub is None) == (case['idx_sub'] is None)
        if idx_sub is not None:
            assert torch.equal(idx_sub.cpu(), case['idx_sub'])
            assert torch.equal(sub_super.cpu(), case['sub_super'])
    for case in gold['pointer_cases']:
        p, v = Cluster.index_select_pointers(case['pointers'].cuda(), case['idx'].cuda())
        assert torch.equal(p.cpu(), case['pointers_new']) and torch.equal(v.cpu(), case['val_idx'])


@pytest.mark.gpu
def test_gpu_relabel_consecutive(gold):
    for case in gold['consecutive_cases']:
        new, uniq = ops.relabel_consecutive(case['src'].cuda(), case['num_ids'])
        assert torch.equal(new.cpu(), case['inv']) and torch.equal(uniq.cpu(), case['unique'])
    g = torch.Generator().manual_seed(5)
    for n, hi in ((1, 1), (4097, 4096), (1_000_000, 300_000), (10, 5_000_000)):
        src = torch.randint(0, hi, (n,), generator=g)
        inv, perm = O.consecutive_cluster(src)
        new, uniq = ops.relabel_consecutive(src.cuda(), hi)
        assert torch.equal(new.cpu(), inv) and torch.equal(uniq.cpu(), src[perm])
    with pytest.raises(IndexError):
        ops.relabel_consecutive(torch.tensor([0, 7]).cuda(), 5)


@pytest.mark.gpu
def test_gpu_primitives_edge_cases():
    dev = 'cuda'
    # no edge survives / every edge survives / empty selection of groups
    ei = torch.tensor([[0, 1, 2, 3], [1, 2, 3, 0]], device=dev)
    out, idx_edge = ops.select_edges(ei, torch.tensor([0, 2], device=dev), 4)
    assert out.shape == (2, 0) and idx_edge.numel() == 0
    out, idx_edge = ops.select_edges(ei, torch.tensor([3, 2, 1, 0], device=dev), 4)
    assert torch.equal(out.cpu(), torch.tensor([[3, 2, 1, 0], [2, 1, 0, 3]]))
    assert torch.equal(idx_edge.cpu(), torch.arange(4))
    with pytest.raises(IndexError):
        ops.select_edges(ei, torch.tensor([1, 1], device=dev), 4)       # repeated
    with pytest.raises(IndexError):
        ops.select_edges(None, torch.tensor([4], device=dev), 4)        # out of range
    ptr = torch.tensor([0, 0, 3, 3, 5], device=dev)
    val = torch.tensor([4, 0, 2, 1, 3], device=dev)
    p, v, grp = ops.csr_select(ptr, val, torch.tensor([3, 0, 1], device=dev), want_group=True)
    assert p.tolist() == [0, 2, 2, 5] and v.tolist() == [1, 3, 4, 0, 2]
    assert grp.tolist() == [0, 0, 2, 2, 2]
    p, v = ops.csr_select(ptr, val, torch.tensor([0, 2], device=dev))
    assert p.tolist() == [0, 0, 0] and v.numel() == 0
    with pytest.raises(IndexError):
        ops.csr_select(ptr, val, torch.tensor([4], device=dev))
    # rows of every unit width (16 / 8 / 4 / 1 bytes) and dtype
    g = torch.Generator().manual_seed(3)
    idx = torch.randperm(1000, generator=g)[:700]
    for shape, dtype in (((1000, 4), torch.float32), ((1000, 7), torch.int64),
                         ((1000, 3), torch.float32), ((1000,), torch.int64),
                         ((1000, 5), torch.uint8), ((1000, 3), torch.float16),
                         ((1000, 2, 3), torch.float64), ((1000,), torch.bool)):
        t = (torch.rand(shape, generator=g) * 200).to(dtype)
        assert torch.equal(ops.take_rows(t.cuda(), idx.cuda()).cpu(), t[idx]), (shape, dtype)
    # the same through the one-launch form, 19 tensors of mixed widths (two launches)
    ts = [(torch.rand((1000,) + tuple(range(2, 2 + i % 3)), generator=g) * 200).to(dt)
          for i, dt in enumerate([torch.float32, torch.int64, torch.uint8, torch.float16,
                                  torch.float64, torch.bool, torch.int32] * 3)][:19]
    ts.append(torch.empty(1000, 0))
    for mine, t in zip(ops.take_rows_multi([t.cuda() for t in ts], idx.cuda()), ts):
        assert mine.dtype == t.dtype and torch.equal(mine.cpu(), t[idx])


@pytest.mark.gpu
def test_gpu_nag_select_benchmark_size_vs_oracle(select_path):
    """BASELINE cfg 2 partition (100 k / 20 k / 4 k nodes, 1.6 M edges on level 1): the device
    path against the oracle at every level, plus size-independent properties."""
    from superpoint_transformer_b200.synthetic import make_nag, CONFIGS
    nag = make_nag(**CONFIGS['cfg2'])
    levels = [level_of(nag[i]) for i in nag.level_range]
    dev = nag.cuda()
    g = torch.Generator().manual_seed(9)
    for i_level in nag.level_range:
        n = nag[i_level].num_nodes
        idx = torch.randperm(n, generator=g)[:(3 * n) // 5]
        res = dev.select(i_level, idx.cuda())
        want = O.nag_select(levels, nag.start_i_level, i_level, idx)
        for j, (a, b) in enumerate(zip(levels_of(res), want)):
            assert_level_equal(a, b, f'cfg2 L{i_level} level {j}', canonical_sub=True)
        # properties: dense ids, consistent sub / super_index, edges inside the selection
        for i in res.level_range:
            d = res[i]
            if d.is_sub:
                up = res[i + 1]
                assert int(d.super_index.max()) + 1 == up.num_nodes
                assert torch.equal(up.sub.to_super_index(), d.super_index)
            if d.has_edges:
                assert int(d.edge_index.max()) < d.num_nodes and int(d.edge_index.min()) >= 0
        # idempotence: selecting everything again changes nothing
        again = res.select(i_level, torch.arange(res[i_level].num_nodes, device='cuda'))
        for a, b in zip(levels_of(again), levels_of(res)):
            assert_level_equal(a, b, 'idempotence')
