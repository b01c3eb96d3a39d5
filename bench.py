#!/usr/bin/env python
"""bench.py — superpoints/s (fwd+bwd) of the hierarchical superpoint-graph
attention + pooling stack on the BASELINE.json cfg-2 workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Own arm (default): one process per GPU (torchrun for N>1), every rank owns one
cfg-2 scene (scene-shard data parallelism, weak scaling), one flat NCCL gradient
all-reduce per step.  Prints ONE JSON line (contract in the task statement) with
`value` (inputs resident in HBM), `e2e` (host buffers -> H2D -> on-device
transforms -> CSR build -> fwd+bwd+step -> D2H loss), `roofline` (dominant
kernel, timed live with CUDA events), `cpu_baseline` (oracle port on host cores,
bounded sample).

Reference arm (--impl reference): the reference's CPU path for the same metric —
the oracle restatement of its source (oracle/path.py; the reference itself is
Python and cannot be installed here: torch_scatter / torch_geometric /
lightning / hydra are absent, SURVEY.md §8c) on all host threads, each step a
bounded sample of the workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "superpoints/sec (fwd+bwd) on 100k-SP 3-level NAG"
UNIT = "superpoints/s"
MEAN_DEGREE = 16
DIM, HEADS, QK_DIM, RPE_DIM, HF_DIM, NUM_CLASSES = 128, 4, 4, 32, 12, 13
_MODEL = ("nano-3 SPT C=128 H=4 qk_dim=4 F=32 (h_edge_mlp 18->32->32, node_mlp 12->32->32), "
          "3 blocks/down level + 1 block/up level, k/q/v RPE, max-pool, GraphNorm, 13-class CE "
          "head, AdamW step; fp32 (ieee matmul)")
_LAW = "sym. degree ~clamp(Poisson16,1,30)+self-loop, random node ids"

# BASELINE.json configs (SURVEY.md §8d).  cfg2 is the configuration the metric is quoted on
# (the default, one scene per GPU: weak scaling).  cfg4 / cfg5 are the 8-GPU workloads: a fixed
# set of scenes / tiles per step sharded over the ranks (strong scaling).
BENCH_CONFIGS = {
    'cfg2': dict(levels=[100_000, 20_000, 4_000], no_ffn=True, scaling='weak', seed=1,
                 metric=METRIC,
                 workload=f"cfg2: S3DIS-shaped 3-level NAG 100k/20k/4k superpoints, {_LAW}; "
                          f"{_MODEL}"),
    'cfg3': dict(levels=[500_000, 100_000, 20_000], no_ffn=True, scaling='weak', seed=2,
                 attn_storage='bf16',
                 metric="superpoints/sec (fwd+bwd) on 500k-SP 3-level NAG (DALES tile), bf16 storage",
                 workload=f"cfg3: DALES-tile 3-level NAG 500k/100k/20k superpoints, {_LAW}; "
                          f"{_MODEL}; bf16 STORAGE of the attention operands (fused projections "
                          f"qkv and edge features), fp32 accumulation / outputs / gradients / "
                          f"everything else"),
    'cfg4': dict(levels=[50_000, 10_000, 2_000], no_ffn=False, scaling='strong', seed=100,
                 scenes=64, scenes_per_batch=8,
                 metric="superpoints/sec (fwd+bwd), 64 scenes x 50k-SP 3-level NAGs per step",
                 workload=f"cfg4: KITTI-360-scan stream, 64 independent scenes x 50k/10k/2k "
                          f"superpoints per optimizer step (seeds 100..163), NAGBatch of 8 scenes "
                          f"per micro-batch, scenes LPT-sharded over the ranks by edge count, "
                          f"gradient accumulation + one NCCL all-reduce per step; {_LAW}; "
                          f"{_MODEL} with FFN branch (no_ffn=False, ffn_ratio=1: "
                          f"configs/experiment/semantic/kitti360.yaml:22-27)"),
    'cfg5': dict(levels=[1_000_000, 200_000, 40_000], no_ffn=True, scaling='strong', seed=3,
                 tiles=8,
                 metric="superpoints/sec (fwd+bwd) on a 1M-SP 3-level graph in 8 tiles",
                 workload=f"cfg5: SuperCluster-size graph 1M/200k/40k superpoints cut into 8 "
                          f"tiles by level-3 ancestor (spatial stripes balanced by edge count), "
                          f"spatially coherent synthetic graph (neighbours close along x), cross-tile edges dropped (reference SampleXYTiling, "
                          f"src/transforms/sampling.py:471), tiles LPT-sharded over the ranks, "
                          f"one NCCL all-reduce per step; {_LAW}; {_MODEL}"),
}
# not a BASELINE configuration: a 2k-superpoint scene for the CPU tests of this script
BENCH_CONFIGS['tiny'] = dict(levels=[2_000, 400, 80], no_ffn=True, scaling='weak', seed=1,
                             metric=METRIC, workload=f"tiny: 2k/400/80 superpoints (test only); {_MODEL}")
LEVELS = BENCH_CONFIGS['cfg2']['levels']
WORKLOAD = BENCH_CONFIGS['cfg2']['workload']
DUMP_BYTES = 60 << 20   # --dump-outputs: 64 MB in all, with room for the .npy headers


def model_kwargs(S=None, no_ffn=True):
    inj = 3 + 1 + 32
    return dict(
        nano=True, segment_hf=['hf'], down_dim=[DIM] * 3,
        down_in_mlp=[[inj, DIM, DIM], [inj + DIM, DIM, DIM], [inj + DIM, DIM, DIM]],
        down_num_heads=HEADS, down_num_blocks=3, down_ffn_ratio=1, up_dim=[DIM] * 2,
        up_in_mlp=[[inj + 2 * DIM, DIM, DIM], [inj + 2 * DIM, DIM, DIM]], up_num_heads=HEADS,
        up_num_blocks=1, node_mlp=[HF_DIM, 32, 32], h_edge_mlp=[18, RPE_DIM, RPE_DIM],
        qk_dim=QK_DIM, in_rpe_dim=RPE_DIM, k_rpe=True, q_rpe=True, v_rpe=True, no_ffn=no_ffn,
        use_diameter_parent=True, pool='max')


def bench_config(cfg_name, world):
    """the `config` object of the JSON line: identical for the own and the reference arm"""
    c = BENCH_CONFIGS[cfg_name]
    par = (f"scene-shard dp{world} (one scene per GPU, flat NCCL grad all-reduce)"
           if c['scaling'] == 'weak' else
           f"scene/tile-shard dp{world} (fixed work per step split over the ranks by edge "
           f"count, flat NCCL grad all-reduce)")
    out = {"workload": c['workload'], "name": cfg_name, "levels": c['levels'],
           "parallelism": par,
           "l2": "inputs_exceed_l2 (per-step working set > 126 MB; no flush needed)"}
    if (DIM, HEADS) != (128, 4):   # --model shipped64 / shipped128: not a BASELINE configuration
        out["model_variant"] = f"C={DIM}, {HEADS} heads (head layout of the shipped configs)"
    return out


# --------------------------------------------------------------------------- #
#  clocks sampler (nvidia-smi while the timed region runs)
# --------------------------------------------------------------------------- #
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}',
                 '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.rows:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            parts = [p.strip() for p in line.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax = float(parts[1])
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
                                  'sw_power_cap'), parts[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- #
#  workload
# --------------------------------------------------------------------------- #
def _pin(nag, labels):
    """fp16 raw edge attributes (configs/datamodule/semantic/default.yaml:40-42), pinned"""
    nbytes = 0
    pin = torch.cuda.is_available()
    for d in nag:
        if d.edge_attr is not None and d.edge_attr.dtype != torch.float16:
            d.edge_attr = d.edge_attr.half()
        d.sub = None  # rebuilt on device from super_index (bit-exact, tests)
        for k in d.keys:
            v = d[k]
            if torch.is_tensor(v):
                d[k] = v.pin_memory() if pin else v
                nbytes += v.numel() * v.element_size()
    labels = labels.pin_memory() if pin else labels
    nbytes += labels.numel() * 8
    return nag, labels, nbytes


def scene_labels(n1, seed):
    return torch.randint(0, NUM_CLASSES, (n1,), generator=torch.Generator().manual_seed(seed + 7))


def host_scene(levels, seed):
    """compact host-side NAG as the reference ships it to the device (trimmed graph,
    fp16 raw edge attributes), pinned."""
    from superpoint_transformer_b200.synthetic import make_nag
    nag = make_nag(levels, mean_degree=MEAN_DEGREE, seed=seed)
    return _pin(nag, scene_labels(levels[0], seed))


def cut_tiles(nag, num_tiles):
    """Cut a NAG into `num_tiles` independent NAGs by top-level ancestor (cfg 5): the top-level
    nodes are sorted along x and split into stripes of equal level-1 EDGE count; every lower
    node follows its ancestor, edges whose ends fall into different tiles are dropped (the
    reference tiles at preprocessing and treats tiles as independent samples,
    src/transforms/sampling.py:471).  Host-side, once (outside every timed region).  Returns
    (tiles, kept_edge_fraction)."""
    import numpy as np
    from superpoint_transformer_b200.data import Data, NAG, Cluster
    levels = list(nag.level_range)
    top = levels[-1]
    # ancestor of every node at the top level
    anc = {top: torch.arange(nag[top].num_nodes)}
    for l in reversed(levels[:-1]):
        anc[l] = anc[l + 1][nag[l].super_index]
    # level-1 edges per top-level ancestor (of the source node) -> balanced x-stripes
    l1 = levels[0]
    e_per_top = torch.bincount(anc[l1][nag[l1].edge_index[0]], minlength=nag[top].num_nodes)
    order = torch.argsort(nag[top].pos[:, 0])
    csum = torch.cumsum(e_per_top[order].double(), 0)
    tile_of_sorted = torch.clamp((csum / csum[-1] * num_tiles).long(), max=num_tiles - 1)
    tile_top = torch.empty_like(tile_of_sorted)
    tile_top[order] = tile_of_sorted
    tiles, kept, total = [], 0, 0
    for tl in range(num_tiles):
        datas, new_id = [], {}
        for l in levels:
            keep = tile_top[anc[l]] == tl
            idx = torch.nonzero(keep).view(-1)
            nid = torch.full((nag[l].num_nodes,), -1, dtype=torch.long)
            nid[idx] = torch.arange(idx.numel())
            new_id[l] = nid
        for l in levels:
            d, nid = nag[l], new_id[l]
            idx = torch.nonzero(nid >= 0).view(-1)
            out = {}
            for k in d.keys:
                v = d[k]
                if k in ('edge_index', 'edge_attr', 'super_index', 'sub') or not torch.is_tensor(v):
                    continue
                out[k] = v[idx]
            ei = d.edge_index
            ek = (nid[ei[0]] >= 0) & (nid[ei[1]] >= 0)
            out['edge_index'] = nid[ei[:, ek]]
            out['edge_attr'] = d.edge_attr[ek]
            if l == l1:
                kept += int(ek.sum()); total += int((nid[ei[0]] >= 0).sum())
            if d.super_index is not None:
                out['super_index'] = new_id[l + 1][d.super_index[idx]]
            datas.append(Data(**out))
        for i in range(1, len(datas)):
            datas[i].sub = Cluster.from_super_index(datas[i - 1].super_index, datas[i].num_nodes)
        tiles.append(NAG(datas, start_i_level=nag.start_i_level))
    return tiles, kept / max(total, 1)


def rank_micro_batches(cfg_name, rank, world):
    """Host-side inputs of this rank for one step: list of (pinned NAG, labels, bytes, n1, E1)
    micro-batches + a description of the sharding (per-rank edge totals)."""
    from superpoint_transformer_b200.synthetic import make_nag
    from superpoint_transformer_b200.distributed import shard_indices
    from superpoint_transformer_b200.data import NAGBatch
    c = BENCH_CONFIGS[cfg_name]
    if c['scaling'] == 'weak':
        nag, labels, nb = host_scene(c['levels'], seed=c['seed'] + rank)
        return [(nag, labels, nb, c['levels'][0])], None
    if cfg_name == 'cfg4':
        seeds = [c['seed'] + i for i in range(c['scenes'])]
        # every rank generates all scenes (deterministic in the seed, ~0.2 s each, setup only),
        # so all ranks derive the same LPT assignment by level-1 edge count without talking
        allsc = [make_nag(c['levels'], mean_degree=MEAN_DEGREE, seed=sd) for sd in seeds]
        weights = [float(sc[1].edge_index.shape[1]) for sc in allsc]
        mine = shard_indices(len(seeds), rank, world, weights=weights)
        per_rank = [sum(weights[i] for i in shard_indices(len(seeds), r, world, weights=weights))
                    for r in range(world)]
        scenes = [allsc[i] for i in mine]
        del allsc
        e_mine = sum(int(sc[1].edge_index.shape[1]) for sc in scenes)
        out = []
        spb = c['scenes_per_batch']
        for j in range(0, len(scenes), spb):
            group = scenes[j:j + spb]
            labels = torch.cat([scene_labels(c['levels'][0], seeds[mine[j + i]])
                                for i in range(len(group))])
            batch = NAGBatch.from_nag_list(group) if len(group) > 1 else group[0]
            nag, labels, nb = _pin(batch, labels)
            out.append((nag, labels, nb, c['levels'][0] * len(group)))
        return out, dict(items=len(seeds), mine=len(mine), trimmed_edges_level1_mine=e_mine,
                         edges_per_rank=[int(x) for x in per_rank],
                         imbalance_max_over_mean=round(max(per_rank) * world / sum(per_rank), 4))
    if cfg_name == 'cfg5':
        full = make_nag(c['levels'], mean_degree=MEAN_DEGREE, seed=c['seed'], spatial=True)
        tiles, kept = cut_tiles(full, c['tiles'])
        w = [float(t[1].edge_index.shape[1]) for t in tiles]
        mine = shard_indices(len(tiles), rank, world, weights=w)
        per_rank = [sum(w[i] for i in shard_indices(len(tiles), r, world, weights=w))
                    for r in range(world)]
        out = []
        for i in mine:
            n1 = tiles[i][1].num_nodes
            nag, labels, nb = _pin(tiles[i], scene_labels(n1, c['seed'] + 31 * i))
            out.append((nag, labels, nb, n1))
        return out, dict(items=len(tiles), mine=len(mine), kept_edge_fraction=round(kept, 4),
                         trimmed_edges_level1_per_tile=[int(x) for x in w],
                         edges_per_rank=[int(x) for x in per_rank],
                         imbalance_max_over_mean=round(max(per_rank) * world / sum(per_rank), 4))
    raise ValueError(cfg_name)


def write_outputs(out_dir, loss, logits, grad, budget=DUMP_BYTES):
    """--dump-outputs: what one step of the own arm computed, as float32 .npy files in `out_dir`:
    loss.npy (cross-entropy of every micro-batch of this rank), logits.npy (the head's output on
    the level-1 rows of those micro-batches, in order) and grad.npy (the flat gradient buffer the
    optimizer stepped with).  Where all of it would exceed `budget` bytes, logits.npy holds a
    fixed, seeded sample of the rows, ascending, and logits_rows.npy (float64) their row numbers."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    loss, logits, grad = (t.detach().float().cpu().numpy() for t in (loss, logits, grad))
    if loss.nbytes + logits.nbytes + grad.nbytes > budget:
        room = (budget - loss.nbytes - grad.nbytes) // (logits[0].nbytes + 8)
        assert room > 0, f'loss and gradient alone exceed the {budget}-byte budget'
        rows = torch.randperm(logits.shape[0], generator=torch.Generator().manual_seed(0))[:room]
        rows = rows.sort().values.numpy()
        logits = logits[rows]
        np.save(os.path.join(out_dir, 'logits_rows.npy'), rows.astype(np.float64))
    for name, a in (('loss', loss), ('logits', logits), ('grad', grad)):
        np.save(os.path.join(out_dir, f'{name}.npy'), a)


def device_transforms(S, nag):
    nag = S.transforms.NodeSize()(nag)
    # csr_order: edges emitted grouped by source (the model is invariant to edge order), so the
    # attention blocks read edge_attr in place
    return S.transforms.OnTheFlyHorizontalEdgeFeatures(add_self_loops=True, csr_order=True)(nag)


def attn_bytes(tag, m, elt=4, idx=4):
    """ALGORITHMIC (compulsory) bytes of one launch: every input / output tensor once
    (DESIGN.md §Kernels).  HD2 = 2*H*D, C = H*Dv."""
    R, E, H, D, Dv, F = m['R'], m['E'], m['H'], m['D'], m['Dv'], m['F']
    T = m.get('T', R)
    C, HD2, HF = H * Dv, 2 * H * D, H * F
    abar = HF if m.get('abar') else 0
    if tag == 'attn_fwd':       # qkv in; a in; rowptr+col; agg+abar+sump+m+z out
        return (R * (HD2 + C) + E * F + R * (C + abar + 3 * H)) * elt + (R + 1 + E) * idx
    if tag == 'attn_bwd_rows':  # qkv, a, stats, agg/abar, dY/dabar in; dq, da, P, G out
        da = E * F if m.get('da') else 0
        return (R * (HD2 + C) + E * F + 2 * R * H + 2 * R * (C + abar) + R * HD2 // 2 + da +
                E * H + E * HD2) * elt + (R + 1 + E) * idx
    if tag == 'attn_bwd_targets':  # P, dk_e half of G, dY in; dk, dv out
        return (E * H + E * HD2 // 2 + R * C + T * (HD2 // 2 + C)) * elt + (T + 1 + 2 * E) * idx
    if tag == 'attn_bwd_weights':  # G, a in
        return (E * HD2 + E * F) * elt
    return 0


def kernel_bytes(tag, m):
    """algorithmic bytes per launch (DESIGN.md §3): every input / output tensor once"""
    if tag.startswith('gemm'):   # A [M,K] + W [N,K] + C [M,N] once each (dW: A, B in, C out)
        return (m['M'] * m['K'] + m['N'] * m['K'] + m['M'] * m['N']) * 4
    if tag == 'graphnorm_fwd':   # x read for the statistics, x read + y written by the apply
        return 3 * m['N'] * m['C'] * 4
    if tag == 'graphnorm_bwd':   # x, dy (+ saved activation) read twice, dx written
        return (5 + (2 if m.get('act') else 0)) * m['N'] * m['C'] * 4
    if tag == 'segment_pool_fwd':
        return (m['Nc'] + m['Np'] * (2 if m['r'] >= 2 else 1)) * m['C'] * 4 + (m['Np'] + m['Nc']) * 4
    if tag == 'segment_pool_bwd':
        return (m['Nc'] + m['Np'] * (2 if m['r'] >= 2 else 1)) * m['C'] * 4 + m['Nc'] * 8
    if tag == 'gather_rows':
        return 2 * m['n'] * m['C'] * 4 + m['n'] * 4
    if tag == 'group_index':
        return m['n'] * (8 + 4 + (12 if m.get('other') else 0)) + (m['G'] + 1) * 4
    if tag == 'edge_features':
        return m['Eh'] * (16 + 28) + (2 * m['Eh'] + (m['N'] if m.get('loops') else 0)) * (16 + 72)
    if tag == 'unitsphere':
        return m['N'] * (12 + 12 + 4 + 8) + m['Np'] * 16
    if tag == 'vrpe_epilogue':   # agg, rv in; y out (sump / bias negligible)
        return 3 * m['N'] * m['C'] * 4
    if 'R' not in m or 'E' not in m:
        return 0
    return attn_bytes(tag, m)


def run_own(args):
    import superpoint_transformer_b200 as S
    from superpoint_transformer_b200 import ops
    from superpoint_transformer_b200.distributed import (FlatGradients,
                                                         init_process_group_from_env)
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (own arm) needs a CUDA device; there is no CPU fallback")
    cfg_name = args.config
    cfg = BENCH_CONFIGS[cfg_name]
    rank, world, local = init_process_group_from_env()
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    torch.backends.cuda.matmul.allow_tf32 = False   # fp32 parity setting ('highest')
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(0)

    ops.set_attention_storage(args.attn_storage or cfg.get('attn_storage', 'fp32'))
    net = S.SPT(mlp_norm=S.nn.GraphNorm, norm=S.nn.GraphNorm,
                **model_kwargs(S, no_ffn=cfg['no_ffn']))
    net.apply(S.init_weights)
    head = S.nn.Classifier(DIM, NUM_CLASSES)
    model = torch.nn.ModuleDict(dict(net=net, head=head)).to(dev)
    params = list(model.parameters())
    flat = FlatGradients(params)
    opt = torch.optim.AdamW(params, lr=1e-3, weight_decay=1e-4, fused=True,
                            capturable=not args.no_graph)
    init_params = [p.detach().clone() for p in params]

    def reset_training_state():
        """Every step of the resident phase trains from the seeded initial parameters and a
        fresh AdamW state.  The gradient reductions add with float atomics, so a chain of
        optimizer steps would drift apart from run to run; this way the same arguments give
        the same inputs to every step and the same outputs up to rounding."""
        with torch.no_grad():
            torch._foreach_copy_(params, init_params)
            state = [t for p in params for t in opt.state[p].values() if torch.is_tensor(t)]
            if state:
                torch._foreach_zero_(state)

    # this rank's share of one step: a list of micro-batches (host side, pinned)
    micro, shard_info = rank_micro_batches(cfg_name, rank, world)
    n_mb = len(micro)
    sp_rank = sum(m[3] for m in micro)                  # level-1 superpoints per step, this rank
    h2d_bytes = sum(m[2] for m in micro)
    sp_total = torch.tensor([float(sp_rank)], device=dev)
    if world > 1:
        dist.all_reduce(sp_total)
    sp_total = float(sp_total.item())
    # every micro-batch is averaged over the GLOBAL number of superpoints of the step, so the
    # accumulated gradient is the gradient of the mean loss of the whole step
    loss_scale = [m[3] / sp_total * world for m in micro]   # all_reduce divides by world

    last = {}   # micro-batch -> (loss, logits) of the latest step, for --dump-outputs

    def fwd_bwd(nag, labels, i_mb):
        flat.release()
        out = net(nag)
        logits = head(out)
        loss = torch.nn.functional.cross_entropy(logits, labels)
        if args.dump_outputs:
            last[i_mb] = (loss, logits)
        # the backward reuses the logits' memory; holding them through it costs ~0.7 % of a
        # cfg-2 step, so only a dumping run does
        del logits
        (loss * loss_scale[i_mb] if (n_mb > 1 or world > 1) else loss).backward()
        flat.collect(accumulate=i_mb > 0)
        return loss

    class Graphed:
        """A callable captured as a CUDA graph after two eager warm-up runs on a side stream."""

        def __init__(self, body, pool=None):
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    body()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            self.g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.g, pool=pool):
                self.out = body()

        def __call__(self):
            self.g.replay()
            return self.out

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(fn, steps):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        sync_all()
        t1 = time.time()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), t0, t1

    # ---- resident-input phase ------------------------------------------------
    resident = []
    for nag_h, lab_h, _, _ in micro:
        nag = device_transforms(S, nag_h.to(dev, non_blocking=True))
        lab = lab_h.to(dev, non_blocking=True)
        base = {l: (nag[l].x, nag[l].edge_attr, nag[l]['hf']) for l in nag.level_range}
        resident.append((nag, lab, base))
    edges_l1 = int(sum(r[0][1].edge_index.shape[1] for r in resident))

    def restore(i):
        # SPT.forward rewrites x / edge_attr / hf on the NAG: restore the inputs (no copy)
        nag, _, base = resident[i]
        for l, (x, ea, hf) in base.items():
            d = nag[l]
            d.x, d.edge_attr, d['hf'] = x, ea, hf
            d.diameter = None

    def eager_step():
        loss = None
        reset_training_state()
        for i in range(n_mb):
            restore(i)
            loss = fwd_bwd(resident[i][0], resident[i][1], i)
        flat.all_reduce()
        opt.step()
        return loss

    # parity of the timed path: loss of the untouched model on micro-batch 0 (compared with
    # the CPU oracle's loss on the same scene, same parameters, below)
    with torch.no_grad():
        restore(0)
        loss0_gpu = float(torch.nn.functional.cross_entropy(
            head(net(resident[0][0])), resident[0][1]).item())

    graph_mode, run_resident = False, eager_step
    if not args.no_graph:
        try:
            pool = torch.cuda.graph_pool_handle()
            graphs = []
            for i in range(n_mb):
                def body(i=i):
                    restore(i)
                    return fwd_bwd(resident[i][0], resident[i][1], i)
                graphs.append(Graphed(body, pool=pool))
            g_opt = Graphed(lambda: opt.step(), pool=pool)
            g_reset = Graphed(reset_training_state, pool=pool)   # after g_opt made the state

            def run_resident():   # noqa: F811
                g_reset()
                for gph in graphs:
                    loss = gph()
                flat.all_reduce()
                g_opt()
                return loss
            graph_mode = True
        except Exception as ex:  # noqa: BLE001
            sys.stderr.write(f"[bench] CUDA graph capture failed, running eager: {ex!r}\n")
            torch.cuda.synchronize()
            run_resident = eager_step
    for _ in range(args.warmup):
        run_resident()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    ms, t0, t1 = timed(run_resident, args.steps)
    clocks = sampler.stop(t0, t1) if sampler else None
    if args.dump_outputs and rank == 0:
        # a CUDA graph replays into the tensors it captured, so `last` holds the last timed step
        write_outputs(args.dump_outputs, torch.stack([last[i][0] for i in range(n_mb)]),
                      torch.cat([last[i][1] for i in range(n_mb)]), flat.flat)
    # count my launches per step and time my kernels with CUDA events (eager steps: the
    # same kernels on the same inputs; events cannot be read back from a graph replay)
    for _ in range(2):
        eager_step()
    ops.enable_event_timing(True)
    l0 = ops.launch_count()
    n_evt_steps = 3
    ms_eager, _, _ = timed(eager_step, n_evt_steps)
    launches_per_step = (ops.launch_count() - l0) // n_evt_steps
    records = ops.timing_records()
    ops.enable_event_timing(False)
    ms_eager_step = ms_eager / n_evt_steps
    launches = launches_per_step * args.steps
    ms_per_step = ms / args.steps
    value = sp_total / (ms_per_step * 1e-3)

    # ---- per-kernel roofline from the live events ------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:  # noqa: BLE001
        pass
    peak_gbs, peak_src = (peaks['hbm_gbs'], 'measured (MEASURED_PEAKS.json hbm_gbs)') \
        if 'hbm_gbs' in peaks else (6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)')
    agg = {}
    for tag, meta, s, e in records:
        size = meta.get('E', meta.get('M', meta.get('N', meta.get('Nc', meta.get('n')))))
        shape = f"E={meta['E']},rows={meta['R']}" if 'E' in meta else \
            ','.join(f"{k}={v}" for k, v in meta.items())
        key = (tag, shape)
        a = agg.setdefault(key, dict(tag=tag, E=size, R=shape, ms=0.0, n=0, meta=meta,
                                     bytes=kernel_bytes(tag, meta)))
        a['ms'] += s.elapsed_time(e)
        a['n'] += 1
    kernels = []
    for a in agg.values():
        avg = a['ms'] / a['n']
        gbs = a['bytes'] / (avg * 1e-3) / 1e9
        kernels.append(dict(kernel=a['tag'], E=a['E'], shape=a['R'], launches=a['n'],
                            avg_ms=round(avg, 4), share_of_step=round(a['ms'] / ms_eager, 4),
                            algorithmic_MB=round(a['bytes'] / 1e6, 2),
                            achieved_GBs=round(gbs, 1), frac=round(gbs / peak_gbs, 4)))
    kernels.sort(key=lambda k: -k['share_of_step'])
    own_share = round(sum(k['share_of_step'] for k in kernels), 4)
    # SURVEY §8(d) block formula for the attention core (fwd + bwd rows + bwd targets of the
    # largest level): (5NC + 3EF) elt + 2((N+1)+2E) idx + 2NH 4, over the summed launch times
    survey = None
    big = [a for a in agg.values() if a['tag'] in ('attn_fwd', 'attn_bwd_rows', 'attn_bwd_targets')]
    if big:
        emax = max(a['E'] for a in big)
        grp = [a for a in big if a['E'] == emax]
        if len(grp) == 3:
            m0 = grp[0]['meta']
            N_, E_, C_, F_, H_ = m0['R'], m0['E'], m0['H'] * m0['Dv'], m0['F'], m0['H']
            bytes_d = (5 * N_ * C_ + 3 * E_ * F_) * 4 + 2 * ((N_ + 1) + 2 * E_) * 4 + 2 * N_ * H_ * 4
            t_ms = sum(a['ms'] / a['n'] for a in grp)
            survey = dict(formula="SURVEY §8(d): 5NC*4 + 3EF*4 + 2((N+1)+2E)*4 + 2NH*4 over "
                                  "attn_fwd + attn_bwd_rows (incl. the dW product) + attn_bwd_targets",
                          rows=N_, edges=E_, algorithmic_bytes=int(bytes_d),
                          ms=round(t_ms, 4), achieved_GBs=round(bytes_d / t_ms / 1e6, 1),
                          frac=round(bytes_d / t_ms / 1e6 / peak_gbs, 4))
    if args.kernels_out and rank == 0:
        with open(args.kernels_out, 'w') as fh:
            json.dump(dict(eager_ms_per_step=ms_eager_step, steps=n_evt_steps,
                           own_kernel_share_of_eager_step=own_share, attention_block=survey,
                           kernels=kernels), fh, indent=1)
    roofline = None
    if kernels:
        top = kernels[0]
        traffic = None
        try:
            prof = json.load(open(os.path.join(ROOT, 'profiles', 'dram_traffic.json')))
            traffic = prof.get(f"{top['kernel']}:{top['E']}")
        except Exception:  # noqa: BLE001
            pass
        roofline = dict(bound='hbm', kernel=f"{top['kernel']} ({top['shape']})",
                        achieved=top['achieved_GBs'], peak=peak_gbs, unit='GB/s',
                        frac=top['frac'], traffic=traffic, peak_source=peak_src,
                        algorithmic_bytes=int(top['algorithmic_MB'] * 1e6),
                        avg_launch_ms=top['avg_ms'], share_of_step=top['share_of_step'],
                        attention_block_survey_8d=survey)

    # ---- end-to-end phase: host buffers every step -------------------------------
    def fresh(i):
        nag = micro[i][0].to(dev, non_blocking=True)
        return device_transforms(S, nag), micro[i][1].to(dev, non_blocking=True)

    def e2e_step():
        loss = None
        for i in range(n_mb):
            nag, labels = fresh(i)
            loss = fwd_bwd(nag, labels, i)
        flat.all_reduce()
        opt.step()
        return float(loss.item())  # D2H read of the step's result

    e2e_graph = False
    e2e_h2d = "eager: one pinned->device copy per tensor on the compute stream"
    if graph_mode:
        def make_static_set(i, pool):
            # static device input buffers + the graph (transforms + CSR build + fwd + bwd)
            snag = micro[i][0].to(dev)
            slab = micro[i][1].to(dev)
            pairs = []
            for l in micro[i][0].level_range:
                hd, sd_ = micro[i][0][l], snag[l]
                for k in hd.keys:
                    if torch.is_tensor(hd[k]):
                        pairs.append((sd_[k], hd[k]))
            pairs.append((slab, micro[i][1]))

            def body():
                nag = device_transforms(S, snag.clone())
                return fwd_bwd(nag, slab, i)
            return pairs, Graphed(body, pool=pool)

        try:
            # inputs are double-buffered: while micro-batch j replays on the compute stream the
            # pinned-memory H2D copy of the NEXT one runs on a copy stream into its own buffer
            # set.  Every step still uploads all its inputs and reads its loss back.
            pool2 = torch.cuda.graph_pool_handle()
            slots = [make_static_set(i, pool2) for i in range(n_mb)]
            if n_mb == 1:
                slots.append(make_static_set(0, pool2))   # second buffer set of the same scene
            copy_stream = torch.cuda.Stream()
            h2d_done = [torch.cuda.Event() for _ in slots]
            state = {'j': 0}

            def enqueue_h2d(sl):
                # the graph that last read slot sl is already enqueued on the compute stream
                copy_stream.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(copy_stream):
                    for dst, src in slots[sl][0]:
                        dst.copy_(src, non_blocking=True)
                    h2d_done[sl].record(copy_stream)

            enqueue_h2d(0)

            def e2e_step():  # noqa: F811
                loss = None
                for _ in range(n_mb):
                    sl = state['j'] % len(slots)
                    enqueue_h2d((sl + 1) % len(slots))
                    torch.cuda.current_stream().wait_event(h2d_done[sl])
                    loss = slots[sl][1]()
                    state['j'] += 1
                flat.all_reduce()
                g_opt()
                return float(loss.item())
            e2e_step()
            e2e_graph = True
            e2e_h2d = ("double-buffered: the pinned->device copy of the next micro-batch overlaps "
                       "the compute of the current one (copy stream), every step uploads all inputs")
        except Exception as ex:  # noqa: BLE001
            sys.stderr.write(f"[bench] pipelined e2e failed ({ex!r}); eager e2e\n")
            torch.cuda.synchronize()

    for _ in range(max(1, min(args.warmup, 3))):
        e2e_step()
    e2e_steps = args.steps
    ms_e2e, _, _ = timed(e2e_step, e2e_steps)
    e2e_value = sp_total / (ms_e2e / e2e_steps * 1e-3)

    # ---- CPU baseline (oracle port, rank 0, N=1 only) ----------------------------
    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_sample(cfg_name, target_seconds=20.0)
        if cpu.get('loss') is not None and cpu.get('same_scene'):
            parity = {"loss_gpu": loss0_gpu, "loss_cpu_oracle": cpu['loss'],
                      "abs_diff": abs(loss0_gpu - cpu['loss']),
                      "what": "cross-entropy of the untouched model on the step's first "
                              "micro-batch: CUDA path vs oracle/path.py on the host (same seed, "
                              "same parameters, same fp16-rounded raw edge attributes)"}

    if rank == 0:
        config = bench_config(cfg_name, world)
        line = {
            "metric": cfg['metric'], "value": round(value, 1), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4),
            "higher_is_better": True, "scaling": cfg['scaling'], "vs_baseline": None,
            "dtype": "f32" if ops.ATTN_STORAGE == 'fp32' else
                     "bf16 storage (attention operands) / f32 accumulate",
            "data": "synthetic",
            "config": config,
            "exec": {"superpoints_per_step": int(sp_total), "superpoints_this_rank": int(sp_rank),
                     "micro_batches_this_rank": n_mb, "edges_level1_this_rank": edges_l1,
                     "sharding": shard_info,
                     "cuda_graph": {"value": graph_mode, "e2e": e2e_graph,
                                    "eager_ms_per_step": round(ms_eager_step, 4)},
                     "own_kernel_share_of_eager_step": own_share,
                     "matmul": "fp32-accurate 3xTF32 on tcgen05 tensor cores, TMEM accumulators, "
                               "TMA (csrc/gemm_umma.cu)",
                     "csr": "graph CSR cached across steps in `value` (amortised, SURVEY §8d); "
                            "rebuilt every step in `e2e`; on-the-fly edges emitted in CSR order "
                            "(OnTheFlyHorizontalEdgeFeatures(csr_order=True))",
                     "training_state": "every step of `value` starts from the seeded initial "
                                       "parameters and a fresh AdamW state (one captured copy + "
                                       "zero): the same arguments give the same outputs up to "
                                       "the rounding of one backward"},
            "clocks": clocks,
            "e2e": {"value": round(e2e_value, 1), "unit": UNIT,
                    "ms_per_step": round(ms_e2e / e2e_steps, 4),
                    "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": 4,
                    "h2d": e2e_h2d},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "kernels": kernels[:10],
            "cpu_baseline": cpu,
            "parity": parity,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# --------------------------------------------------------------------------- #
#  CPU reference (oracle port)
# --------------------------------------------------------------------------- #
def _cpu_scene(levels, seed):
    """same generator + the oracle's CPU transforms -> NAG ready for spt_forward (raw edge
    attributes rounded through fp16 exactly like the device path's host buffers)"""
    from oracle import path as P
    from superpoint_transformer_b200.synthetic import make_nag
    nag = make_nag(levels, mean_degree=MEAN_DEGREE, seed=seed)
    size = nag[1].node_size
    for l in nag.level_range:
        d = nag[l]
        ei, ea = P.horizontal_edge_features(d.edge_index, d.edge_attr.half().float(), d.pos,
                                            d.normal, d['log_length'], d['log_surface'],
                                            d['log_volume'], d['log_size'])
        d.edge_index, d.edge_attr = P.add_self_loops(ei, ea, d.num_nodes)
        if l > 1:
            size = torch.from_numpy(P.node_size_np(nag[l - 1].super_index.numpy(), d.num_nodes,
                                                   size.numpy()))
            d.node_size = size
    return nag


def _cpu_state_dict(no_ffn=True):
    """random-init parameters with the reference key names (built from the product's
    module tree on CPU — construction only, no product compute)"""
    import superpoint_transformer_b200 as S
    torch.manual_seed(0)
    net = S.SPT(mlp_norm=S.nn.GraphNorm, norm=S.nn.GraphNorm, **model_kwargs(S, no_ffn=no_ffn))
    net.apply(S.init_weights)
    head = S.nn.Classifier(DIM, NUM_CLASSES)
    sd = {k: v.detach().clone().requires_grad_(v.is_floating_point())
          for k, v in net.state_dict().items()}
    hw = head.classifier.weight.detach().clone().requires_grad_(True)
    hb = head.classifier.bias.detach().clone().requires_grad_(True)
    return sd, hw, hb


def cpu_step(sd, hw, hb, nag, labels, opt=None):
    from oracle import path as P
    for v in list(sd.values()) + [hw, hb]:
        if v.grad is not None:
            v.grad = None
    out = P.spt_forward(sd, nag, num_heads=HEADS, qk_dim=QK_DIM, nano=True, num_down=2, num_up=2,
                        use_diameter_parent=True, pool_reduce='max')
    loss = torch.nn.functional.cross_entropy(torch.nn.functional.linear(out, hw, hb), labels)
    loss.backward()
    if opt is not None:
        opt.step()
    return float(loss.detach())


def _cpu_optimizer(sd, hw, hb):
    ps = [v for v in sd.values() if v.requires_grad] + [hw, hb]
    return torch.optim.AdamW(ps, lr=1e-3, weight_decay=1e-4)


def _scaled_levels(n1):
    return [n1, max(n1 // 5, 2), max(n1 // 25, 1)]


def _available_cores():
    """host cores this process may use: affinity mask capped by the cgroup CPU quota"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
        if quota != 'max':
            n = min(n, max(1, int(float(quota) / float(period) + 0.999)))
    except Exception:  # noqa: BLE001
        pass
    return max(1, n)


def _pick_threads(sd, hw, hb):
    """The reference's torch CPU path does not scale to every core of a many-core
    host on graphs this small; give it its best case: probe 8,16,32,... threads on
    a 1k-superpoint NAG and keep the fastest.  Returns (threads, seconds per
    superpoint at that setting)."""
    avail = _available_cores()
    nag = _cpu_scene(_scaled_levels(1000), seed=1)
    labels = torch.randint(0, NUM_CLASSES, (1000,))
    cands = sorted({c for c in (8, 16, 32, 64, avail) if c <= avail} or {avail})
    best = None
    for c in cands:
        torch.set_num_threads(c)
        cpu_step(sd, hw, hb, nag, labels)
        t = time.time()
        cpu_step(sd, hw, hb, nag, labels)
        dt = time.time() - t
        if best is None or dt < best[1]:
            best = (c, dt)
        elif dt > 1.5 * best[1]:
            break
    torch.set_num_threads(best[0])
    return best[0], best[1] / 1000, avail


def _reference_scene_levels(cfg_name):
    """what ONE reference step processes: cfg2/cfg3 the full scene of the own arm's rank 0;
    cfg4 one of the 64 scenes; cfg5 a scene of one tile's size (bounded samples, stated)."""
    c = BENCH_CONFIGS[cfg_name]
    if cfg_name == 'cfg5':
        return [l // c['tiles'] for l in c['levels']], c['seed'], "one tile-sized scene (1/8 of the graph)"
    if cfg_name == 'cfg4':
        return c['levels'], c['seed'], "one of the 64 scenes"
    return c['levels'], c['seed'], "the full scene of rank 0"


def cpu_reference_sample(cfg_name='cfg2', target_seconds=20.0):
    c = BENCH_CONFIGS[cfg_name]
    sd, hw, hb = _cpu_state_dict(no_ffn=c['no_ffn'])
    threads, per_sp, avail = _pick_threads(sd, hw, hb)
    levels, seed, _ = _reference_scene_levels(cfg_name)
    # the full scene when one step of it stays within ~2x the target, else a scaled-down one
    same = per_sp * levels[0] <= 2.5 * target_seconds and c['scaling'] == 'weak'
    if same:
        n1 = levels[0]
        nag = _cpu_scene(levels, seed=seed)
    else:
        n1 = int(min(max(target_seconds / max(per_sp, 1e-9), 1000), levels[0]))
        n1 = max(1000, (n1 // 1000) * 1000)
        nag = _cpu_scene(_scaled_levels(n1), seed=seed)
    labels = scene_labels(n1, seed)
    t = time.time()
    loss = cpu_step(sd, hw, hb, nag, labels)
    dt = time.time() - t
    return {"value": round(n1 / dt, 1), "unit": UNIT, "cores": threads, "kind": "port",
            "host_cores_available": avail, "loss": loss, "same_scene": bool(same),
            "sample": f"one fwd+bwd of the same model on a {n1}/{nag[2].num_nodes}/"
                      f"{nag[3].num_nodes}-superpoint NAG of the same law "
                      f"({'the scene of rank 0' if same else 'bounded sample'}, {dt:.1f} s); "
                      f"oracle/path.py (reference glue restated, torch CPU leaves), fp32, "
                      f"{threads} threads (fastest of the probed thread counts on this "
                      f"{avail}-core host)"}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    cfg_name = args.config
    c = BENCH_CONFIGS[cfg_name]
    sd, hw, hb = _cpu_state_dict(no_ffn=c['no_ffn'])
    threads, per_sp, avail = _pick_threads(sd, hw, hb)
    levels, seed, what = _reference_scene_levels(cfg_name)
    n1 = levels[0]
    nag = _cpu_scene(levels, seed=seed)          # the stated configuration, not a scaled sample
    labels = scene_labels(n1, seed)
    opt = _cpu_optimizer(sd, hw, hb)
    for _ in range(args.warmup):
        cpu_step(sd, hw, hb, nag, labels, opt)
    t = time.time()
    for _ in range(args.steps):
        cpu_step(sd, hw, hb, nag, labels, opt)
    dt = time.time() - t
    ms = dt / args.steps * 1e3
    value = n1 / (ms * 1e-3)
    sample = (f"each step = fwd + bwd + AdamW on {what}: a {n1}/{levels[1]}/{levels[2]}-superpoint "
              f"NAG (seed {seed}), oracle/path.py on {threads} threads (fastest probed; host has "
              f"{avail} cores)")
    print(json.dumps({
        "impl": "reference", "metric": c['metric'], "value": round(value, 1), "unit": UNIT,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": c['scaling'],
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(cfg_name, world),
        "cpu_baseline": {"value": round(value, 1), "unit": UNIT, "cores": threads,
                         "kind": "port", "sample": sample},
        "e2e": {"value": round(value, 1), "unit": UNIT, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='own', choices=['own', 'reference'])
    ap.add_argument('--config', default=os.environ.get('BENCH_CONFIG', 'cfg2'),
                    choices=sorted(BENCH_CONFIGS))
    ap.add_argument('--attn-storage', default=None, choices=['fp32', 'bf16'],
                    help="override the configuration's storage of the attention operands")
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='eager launches, no CUDA graphs')
    ap.add_argument('--kernels-out', default=None, help='write the full per-kernel timing table (JSON)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the loss, logits and gradient of the last timed step as .npy '
                         'files in DIR (own arm)')
    ap.add_argument('--model', default='baseline', choices=['baseline', 'shipped64', 'shipped128'],
                    help="'baseline': the BASELINE.json model (C=128, 4 heads); 'shipped64' / "
                         "'shipped128': the head layout of the shipped configs (16 heads, C = 64 "
                         "as S3DIS / DALES, C = 128 as KITTI-360) on the same graphs — not a "
                         "BASELINE configuration, reported with `config.model_variant`")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes what the own arm computed; the reference arm has none')
    if args.model != 'baseline':
        global DIM, HEADS
        DIM, HEADS = (64, 16) if args.model == 'shipped64' else (128, 16)
    args.warmup = max(args.warmup, 3) if args.impl == 'own' else args.warmup
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_own(args)


if __name__ == '__main__':
    main()
