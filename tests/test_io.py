"""On-disk NAG format, read side (SURVEY.md §8 f4): the HDF5 subset reader and the loaders,
and a REAL partition as test data — tests/golden/demo_nag.pt is the reference's demo room
(notebooks/demo_nag_v3.h5: 41 568 points, 1 192 / 501 / 166 superpoints) as read by
superpoint_transformer_b200.io (tests/make_demo_fixture.py).  CPU only."""
import hashlib
import json
import lzma
import os

import pytest
import torch

from oracle import select as O
from oracle import sampling as OS
from superpoint_transformer_b200.data import NAG, Data, Cluster
from superpoint_transformer_b200.transforms import (SampleSubNodes, SampleSegments, SampleEdges,
                                                   NAGRestrictSize, SampleRadiusSubgraphs,
                                                   SampleKHopSubgraphs)

from test_select import assert_level_equal, levels_of, to_product, oracle_primitives  # noqa
from make_demo_fixture import FIXTURE_H5_XZ, FIXTURE_H5_JSON, hole_tensor

FIXTURE = os.path.join(os.path.dirname(__file__), 'golden', 'demo_nag.pt')


def as_long(level):
    out = {}
    for k, v in level.items():
        if isinstance(v, dict):
            out[k] = {f: t.long() for f, t in v.items()}
        else:
            out[k] = v if v.is_floating_point() or k == 'rgb' else v.long()
    return out


@pytest.fixture(scope='module')
def demo():
    raw = torch.load(FIXTURE, weights_only=False)
    return {'start': raw['start'], 'levels': [as_long(lv) for lv in raw['levels']]}


@pytest.fixture(scope='module')
def demo_h5(tmp_path_factory):
    """The reference's demo file, byte for byte: its committed copy with the holes refilled from
    demo_nag.pt (tests/make_demo_fixture.py), checked against the original's SHA-256."""
    with open(FIXTURE_H5_JSON) as fh:
        manifest = json.load(fh)
    with open(FIXTURE_H5_XZ, 'rb') as fh:
        buf = bytearray(lzma.decompress(fh.read()))
    raw = torch.load(FIXTURE, weights_only=False)
    for name, addr, nbytes in manifest['holes']:
        buf[addr:addr + nbytes] = hole_tensor(raw, name).numpy().tobytes()
    assert hashlib.sha256(buf).hexdigest() == manifest['sha256']
    path = tmp_path_factory.mktemp('demo') / 'demo_nag_v3.h5'
    path.write_bytes(buf)
    return str(path)


def test_demo_partition_is_a_consistent_hierarchy(demo):
    levels = demo['levels']
    assert demo['start'] == 0 and [lv['pos'].shape[0] for lv in levels] == [41568, 1192, 501, 166]
    for i in range(3):
        child, parent = levels[i], levels[i + 1]
        n_parent = parent['pos'].shape[0]
        assert int(child['super_index'].max()) + 1 == n_parent
        assert torch.equal(O.to_super_index(parent['sub']), child['super_index'])
        sizes = parent['sub']['pointers'][1:] - parent['sub']['pointers'][:-1]
        assert (sizes > 0).all() and int(sizes.sum()) == child['pos'].shape[0]
        # label histograms: a parent holds at least what its (sub-sampled) children hold
        up = torch.zeros_like(parent['y']).index_add_(0, child['super_index'], child['y'])
        assert (up <= parent['y']).all()
    for lv in levels[1:]:
        ei = lv['edge_index']
        assert ei.shape[0] == 2 and lv['edge_attr'].shape == (ei.shape[1], 7)
        assert int(ei.max()) < lv['pos'].shape[0] and (ei[0] < ei[1]).all()      # trimmed graph
    assert 'edge_index' not in levels[0] and levels[0]['rgb'].dtype == torch.uint8


def test_reader_and_loaders_reproduce_the_fixture(demo_h5):
    from superpoint_transformer_b200.io import H5File, load_nag
    raw = torch.load(FIXTURE, weights_only=False)
    with H5File(demo_h5) as f:
        assert f.keys() == ['level_0', 'level_1', 'level_2', 'level_3']
        assert int(f.attrs['start_i_level']) == 0
        assert f['level_1/_not_indexable_'].read() == ['sub', 'edge_attr', 'edge_index']
        assert f['level_0/pos'].shape == (41568, 3) and str(f['level_0/pos'].dtype) == 'float32'
        assert f['level_2/_cluster_/sub'].keys() == ['is_index_value', 'pointers', 'value_0']
    nag = NAG.load(demo_h5)
    assert isinstance(nag, NAG) and nag.num_points == [41568, 1192, 501, 166]
    for got, want in zip(levels_of(nag), raw['levels']):
        assert_level_equal(got, want, 'fixture')
    # integers widened, colours as floats, a level range, a key subset
    part = NAG.load(demo_h5, low=1, high=2, keys=['pos', 'super_index', 'sub', 'rgb'],
                    non_fp_to_long=True)
    assert part.start_i_level == 1 and part.num_levels == 2 and sorted(part[1].keys) == \
        ['pos', 'sub', 'super_index']
    assert part[1].super_index.dtype == torch.int64 and part[2].sub.points.dtype == torch.int64
    full = load_nag(demo_h5, non_fp_to_long=True, rgb_to_float=True)
    assert full[0].rgb.dtype == torch.float32 and float(full[0].rgb.max()) <= 1.0
    assert torch.equal((full[0].rgb * 255).round().byte(), nag[0].rgb)
    with pytest.raises(NotImplementedError):
        NAG.load(demo_h5, idx=torch.arange(10))
    level = Data.load(H5File(demo_h5)['level_3'], non_fp_to_long=True)
    assert level.num_nodes == 166 and isinstance(level.sub, Cluster)


def test_save_load_round_trip(demo, tmp_path):
    """NAG.save -> NAG.load on the real partition, a nano partition and a synthetic one: every
    tensor comes back (integers through their smallest dtype, `y` through CSR, `sub` through
    `_cluster_`), for the fp32 default and for fp16 features."""
    from superpoint_transformer_b200.io import H5File
    from superpoint_transformer_b200.synthetic import make_nag
    nano = NAG(to_product(demo['levels'], 0)._list[1:], start_i_level=1)
    cases = {'demo': to_product(demo['levels'], 0), 'nano': nano,
             'synthetic': make_nag([500, 100, 20], mean_degree=6, seed=1)}
    for name, nag in cases.items():
        path = str(tmp_path / f'{name}.h5')
        nag.save(path)
        back = NAG.load(path, low=nag.start_i_level, non_fp_to_long=True)
        assert back.start_i_level == nag.start_i_level and back.num_points == nag.num_points
        for a, b in zip(levels_of(back), levels_of(nag)):
            b = {k: (v if isinstance(v, dict) or v.is_floating_point() or k == 'rgb'
                     else v.long()) for k, v in b.items()}
            assert_level_equal(a, b, name)
        with H5File(path) as f:
            lvl = f[f'level_{nag.start_i_level + 1}']
            assert sorted(lvl['_not_indexable_'].read()) == ['edge_attr', 'edge_index', 'sub']
            assert int(f.attrs['start_i_level']) == nag.start_i_level
            stored = lvl['super_index'].dtype
            assert stored.itemsize < 8                       # smallest integer dtype on disk
    half = str(tmp_path / 'half.h5')
    cases['demo'].save(half, fp_dtype=torch.float16)
    back = NAG.load(half)
    assert back[1].edge_attr.dtype == torch.float16 and back[1].pos.dtype == torch.float32
    assert torch.equal(back[1].edge_attr, cases['demo'][1].edge_attr.half())
    one = str(tmp_path / 'level.h5')
    cases['demo'][2].save(one)
    level = Data.load(one, non_fp_to_long=True)
    assert level.num_nodes == 501 and torch.equal(level.sub.points, cases['demo'][2].sub.points)


def test_written_file_has_the_reference_files_structure(demo_h5, tmp_path):
    """Saving the loaded demo partition gives the reference file's own inventory (names,
    shapes, stored dtypes) and the same header messages byte for byte."""
    from superpoint_transformer_b200.io import H5File
    out = str(tmp_path / 'again.h5')
    NAG.load(demo_h5).save(out)

    def inventory(g, path=''):
        items = {}
        for k in g.keys():
            o = g[k]
            if hasattr(o, 'keys'):
                items.update(inventory(o, f'{path}/{k}'))
            else:
                items[f'{path}/{k}'] = (o.shape, str(o.dtype))
        return items

    ref, mine = H5File(demo_h5), H5File(out)
    assert inventory(ref) == inventory(mine) and len(inventory(mine)) == 63
    assert ref._r.buf[8:24] == mine._r.buf[8:24]                    # superblock parameters

    def header_messages(f, key):
        r = f._r
        group, name = key.rsplit('/', 1)
        addr = f[group]._links[name]
        out = []
        for mtype, size, body in r.messages(addr):
            if mtype in (0x01, 0x03, 0x05):                        # dataspace, datatype, fill
                out.append((mtype, bytes(r.buf[body:body + size])))
            elif mtype == 0x08:                                    # layout: class + size
                out.append((mtype, bytes(r.buf[body:body + 2]) + bytes(r.buf[body + 10:body + 18])))
        return out

    for key in ('level_1/pos', 'level_1/super_index', 'level_0/rgb', 'level_2/_not_indexable_',
                'level_3/_cluster_/sub/pointers', 'level_0/_csr_/y/shape'):
        assert header_messages(ref, key) == header_messages(mine, key), key
    for key in ('level_1/edge_attr', 'level_2/_csr_/y/values', 'level_3/_cluster_/sub/value_0'):
        assert (ref[key].read() == mine[key].read()).all()


def test_reader_rejects_what_it_does_not_parse(tmp_path):
    from superpoint_transformer_b200.io import H5File
    bad = tmp_path / 'not.h5'
    bad.write_bytes(b'plain text' * 10)
    with pytest.raises(ValueError):
        H5File(str(bad))
    newer = tmp_path / 'v2.h5'
    newer.write_bytes(b'\x89HDF\r\n\x1a\n' + bytes([2]) + bytes(100))
    with pytest.raises(NotImplementedError):
        H5File(str(newer))


def test_select_on_the_real_partition_matches_the_oracle(demo, oracle_primitives):
    g = torch.Generator().manual_seed(0)
    for i_level in range(4):
        n = demo['levels'][i_level]['pos'].shape[0]
        idx = torch.randperm(n, generator=g)[:n // 2]
        got = to_product(demo['levels'], 0).select(i_level, idx)
        want = O.nag_select(demo['levels'], 0, i_level, idx)
        for j, (a, b) in enumerate(zip(levels_of(got), want)):
            assert_level_equal({k: v for k, v in a.items() if k in b}, b,
                               f'level {i_level} -> {j}', canonical_sub=True)


def test_sampling_pipeline_on_the_real_partition(demo, oracle_primitives):
    """The on-device transforms of a training pipeline, chained, on real data."""
    nag = to_product(demo['levels'], 0)
    torch.manual_seed(0)
    out = SampleSubNodes(high=1, low=0, n_max=32, n_min=16)(nag)
    sizes = torch.bincount(nag[0].super_index, minlength=1192)
    assert torch.equal(torch.bincount(out[0].super_index, minlength=1192),
                       OS.sampling_counts(sizes, 32, 16))
    out = SampleRadiusSubgraphs(r=2.0, i_level=1, k=2, disjoint=False)(out)
    out = SampleSegments(ratio=0.2, by_size=True, by_class=True)(out)
    out = SampleEdges(level='1+', n_min=4, n_max=8)(out)
    out = NAGRestrictSize(level='1+', num_nodes=400, num_edges=2000)(out)
    assert 0 < out[1].num_nodes <= 400 and out[1].num_edges <= 2000
    for i in range(3):
        assert int(out[i].super_index.max()) + 1 == out[i + 1].num_nodes
        assert torch.equal(out[i + 1].sub.to_super_index(), out[i].super_index)
        if out[i + 1].edge_index is not None and out[i + 1].num_edges:
            assert int(out[i + 1].edge_index.max()) < out[i + 1].num_nodes
    # label histograms still add up after all the re-indexing
    for i in range(3):
        up = torch.zeros_like(out[i + 1].y).index_add_(0, out[i].super_index, out[i].y)
        assert (up <= out[i + 1].y).all()      # (children were sampled away, never added)
    hop = SampleKHopSubgraphs(hops=1, i_level=2, k=1, disjoint=False)(nag)
    assert 0 < hop[2].num_nodes < nag[2].num_nodes
