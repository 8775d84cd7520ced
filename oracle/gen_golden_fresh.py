"""Mint golden vectors on fresh seeds from the UNMODIFIED reference staged under oracle/_ref (oracle/build_ref.py): the SuperGlue
module's forward pass on configurations no other fixture covers (``use_offset``, a regularisation != 1, six side-info channels),
ground-truth matches from a homography (models/gt_matches_generation.py) and the matching loss (utils/losses.py).

TEST INFRASTRUCTURE.  Output: tests/golden/fresh_seeds.pt (tests/test_oracle_golden.py).  Inputs and weights are not stored: the
functions below regenerate them from the seeds.  The context descriptors are stored as a strided sample plus per-channel fp64 sums.

    python oracle/build_ref.py && python oracle/gen_golden_fresh.py
"""
from __future__ import annotations

import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from openglue_b200.synthetic import default_config, synthetic_pairs, synthetic_state_dict  # noqa: E402

# (seed, default_config keywords, (N, M)); batch 2, planted pairs
SUPERGLUE_CASES = [
    (11, dict(descriptor_dim=64, num_stages=2, num_iters=15), (97, 61)),
    (12, dict(descriptor_dim=128, num_stages=2, num_iters=7, side_info_size=6, use_offset=True, reg=0.7), (50, 75)),
]
# (seed, (batch, N, M))
LABEL_CASES = [(21, (2, 60, 45)), (22, (3, 33, 80))]
CTX_STRIDE = 2


def superglue_inputs(seed, kw, nm):
    cfg = default_config(**kw)
    sd = synthetic_state_dict(cfg, seed=seed)
    data = synthetic_pairs(2, nm[0], nm[1], cfg['descriptor_dim'], cfg['positional_encoding']['side_info_size'],
                           family='planted', seed=seed)
    return cfg, sd, data


def label_inputs(seed, b, n, m):
    """Keypoints related by a homography (planted correspondences + clutter), its transformation dict and log-scores."""
    g = torch.Generator().manual_seed(seed)
    k0 = torch.rand(b, n, 2, generator=g) * torch.tensor([640.0, 480.0])
    H = torch.tensor([[0.9, 0.05, 20.0], [-0.04, 0.95, 12.0], [1e-5, 2e-5, 1.0]]).repeat(b, 1, 1)
    k0h = torch.cat([k0, torch.ones(b, n, 1)], -1) @ H.transpose(1, 2)
    k0w = k0h[..., :2] / k0h[..., 2:]
    npl = min(n, m // 2)
    k1 = torch.cat([k0w[:, :npl] + 0.3 * torch.randn(b, npl, 2, generator=g),
                    torch.rand(b, m - npl, 2, generator=g) * torch.tensor([640.0, 480.0])], 1)
    tf = {'type': ['perspective'] * b, 'H': H}
    scores = torch.log_softmax(torch.randn(b, n + 1, m + 1, generator=g), dim=-1)
    return k0, k1, tf, scores


def main():
    from oracle.build_ref import import_reference
    ref = import_reference()
    if ref is None:
        raise SystemExit('oracle/_ref is not staged: run oracle/build_ref.py first')
    SuperGlueRef, ref_criterion, ref_generate = ref
    fx = {'reference': 'models/superglue, models/gt_matches_generation.py, utils/losses.py of the unmodified reference, '
                       'fp32 CPU, torch ' + torch.__version__, 'ctx_stride': CTX_STRIDE, 'superglue': [], 'labels': []}
    for seed, kw, nm in SUPERGLUE_CASES:
        cfg, sd, data = superglue_inputs(seed, kw, nm)
        model = SuperGlueRef(dict(cfg)).eval()
        model.load_state_dict(sd, strict=True)
        with torch.no_grad():
            out = model(data)
        entry = {'scores': out['scores'].clone()}
        for i in (0, 1):
            ctx = out[f'context_descriptors{i}']
            entry[f'ctx{i}_sample'] = ctx[:, ::CTX_STRIDE, ::CTX_STRIDE].clone()
            entry[f'ctx{i}_f64_sum'] = ctx.double().sum(-1)
        fx['superglue'].append(entry)
    for seed, (b, n, m) in LABEL_CASES:
        k0, k1, tf, scores = label_inputs(seed, b, n, m)
        feat = lambda k: {'keypoints': k, 'local_descriptors': torch.zeros(b, k.shape[1], 4), 'side_info': torch.zeros(b, k.shape[1], 1)}
        _, y_true = ref_generate({'transformation': tf}, feat(k0), feat(k1), positive_threshold=3.0, negative_threshold=5.0)
        y_pred = {'scores': scores, 'context_descriptors0': torch.zeros(b, 8, n), 'context_descriptors1': torch.zeros(b, 8, m)}
        loss = ref_criterion(y_true, y_pred, margin=None)
        fx['labels'].append({'gt_matches0': y_true['gt_matches0'].clone(), 'gt_matches1': y_true['gt_matches1'].clone(),
                             'loss': loss['loss'].detach().clone(), 'metric_loss': float(loss['metric_loss'])})
    path = os.path.join(ROOT, 'tests', 'golden', 'fresh_seeds.pt')
    torch.save(fx, path)
    print(f'{path}: {os.path.getsize(path)} bytes')


if __name__ == '__main__':
    main()
