"""(Fixture script, not a test.)  Two fixtures from the reference's demo partition
(notebooks/demo_nag_v3.h5 of the reference project, a 4-level S3DIS room: 41 568 points,
1 192 / 501 / 166 superpoints):
    python tests/make_demo_fixture.py <path to demo_nag_v3.h5>

* tests/golden/demo_nag.pt: the partition as read by superpoint_transformer_b200.io.  Integers
  are kept in the file's own (smallest) dtypes to keep the fixture at the size of the file;
  tests cast with `.long()`.
* tests/golden/demo_nag_v3.h5.xz + .json: the file itself, byte for byte, except the raw data of
  every dataset that demo_nag.pt holds verbatim, which is zeroed (the "holes" listed in the
  .json with the SHA-256 of the whole file).  Tests refill the holes from demo_nag.pt and check
  the hash, so they read the reference's own file without the 2.7 MB of it in the repository."""
import hashlib
import json
import lzma
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from superpoint_transformer_b200.data import Cluster          # noqa: E402
from superpoint_transformer_b200.io import H5File, load_nag   # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
OUT = os.path.join(GOLDEN, 'demo_nag.pt')
FIXTURE_H5_XZ = os.path.join(GOLDEN, 'demo_nag_v3.h5.xz')
FIXTURE_H5_JSON = os.path.join(GOLDEN, 'demo_nag_v3.h5.json')


def to_plain(nag):
    levels = []
    for i in nag.level_range:
        lv = {}
        for k in nag[i].keys:
            v = nag[i][k]
            lv[k] = {'pointers': v.pointers, 'points': v.points} if isinstance(v, Cluster) else v
        levels.append(lv)
    return {'start': nag.start_i_level, 'levels': levels}


def hole_tensor(plain, dataset):
    """The tensor of `plain` (to_plain's format) whose bytes are the raw data of `dataset`, or
    None (`y` is stored as CSR, not verbatim)."""
    level, key = dataset.split('/', 1)
    lv = plain['levels'][int(level[len('level_'):])]
    if key == '_cluster_/sub/value_0':
        return lv['sub']['points']
    return None if key == 'y' else lv.get(key)


def write_holed_copy(src, plain):
    buf = bytearray(open(src, 'rb').read())
    holes = []
    with H5File(src) as f:
        for i, lv in enumerate(plain['levels']):
            for k in lv:
                name = f'level_{i}/_cluster_/sub/value_0' if k == 'sub' else f'level_{i}/{k}'
                t = hole_tensor(plain, name)
                if t is None:
                    continue
                kind, addr, nbytes = f[name]._layout
                assert kind == 'contiguous' and bytes(buf[addr:addr + nbytes]) == \
                    t.numpy().tobytes(), name
                holes.append([name, addr, nbytes])
    digest = hashlib.sha256(buf).hexdigest()
    for _, addr, nbytes in holes:
        buf[addr:addr + nbytes] = bytes(nbytes)
    with open(FIXTURE_H5_XZ, 'wb') as fh:
        fh.write(lzma.compress(bytes(buf), preset=9 | lzma.PRESET_EXTREME))
    with open(FIXTURE_H5_JSON, 'w') as fh:
        json.dump({'sha256': digest, 'holes': holes}, fh, indent=1)


if __name__ == '__main__':
    src = sys.argv[1]
    plain = to_plain(load_nag(src))
    torch.save(plain, OUT)
    write_holed_copy(src, plain)
    for path in (OUT, FIXTURE_H5_XZ, FIXTURE_H5_JSON):
        print(path, os.path.getsize(path))
