"""Pin the oracle: it must reproduce the reference's own outputs (tests/golden/, minted by
oracle/gen_golden.py from the unmodified reference) before anything is compared against it."""
import os

import pytest
import torch

from oracle import superglue_oracle as O
from conftest import GOLDEN_BIG, GOLDEN_DIR, GOLDEN_FULL, GOLDEN_SAMPLED


@pytest.fixture(scope='module')
def golden_fresh():
    return torch.load(os.path.join(GOLDEN_DIR, 'fresh_seeds.pt'), weights_only=False)


@pytest.mark.parametrize('name', GOLDEN_FULL)
def test_oracle_matches_reference_full(golden, name):
    fx = golden(name)
    out = O.run(fx['state_dict'], fx['config'], fx['data'], fx['match_threshold'])
    # same ATen ops, same order => fp32 agreement to rounding noise
    assert (out['scores'] - fx['scores_f32']).abs().max() <= 2e-6
    assert (out['context_descriptors0'] - fx['context_descriptors0_f32']).abs().max() <= 1e-5
    assert (out['context_descriptors1'] - fx['context_descriptors1_f32']).abs().max() <= 1e-5
    assert torch.equal(out['matches0'], fx['matches0'])
    assert (out['matching_scores0'] - fx['matching_scores0']).abs().max() <= 2e-6
    # fp64 oracle vs fp64 reference
    out64 = O.run(fx['state_dict'], fx['config'], fx['data'], fx['match_threshold'], dtype=torch.float64)
    assert (out64['scores'] - fx['scores_f64']).abs().max() <= 1e-10


@pytest.mark.parametrize('name', GOLDEN_SAMPLED)
def test_oracle_matches_reference_c1(golden, name):
    """BASELINE.json configs[0]: 1 pair, N=M=512, d=256, 9 stages, 20 Sinkhorn iterations."""
    fx = golden(name)
    out = O.run(fx['state_dict'], fx['config'], fx['data'], fx['match_threshold'])
    s = out['scores']
    assert (s[:, ::7, ::5] - fx['scores_f32_sample']).abs().max() <= 5e-6
    assert (s[:, -1, :] - fx['scores_f32_lastrow']).abs().max() <= 5e-6
    assert (s[:, :, -1] - fx['scores_f32_lastcol']).abs().max() <= 5e-6
    assert (out['context_descriptors0'][:, ::4, ::8] - fx['ctx0_f32_sample']).abs().max() <= 2e-5
    assert torch.equal(out['matches0'], fx['matches0'])
    assert (out['matching_scores0'] - fx['matching_scores0']).abs().max() <= 5e-6
    rel = (s.double().sum(2) - fx['scores_f64_rowsum']).abs().max() / fx['scores_f64_rowsum'].abs().max()
    assert rel < 1e-6


@pytest.mark.parametrize('name', GOLDEN_BIG)
def test_oracle_matches_reference_big(golden, name):
    """BASELINE.json configs[1], [2], [4] at full depth: the oracle on the fixture's scored pairs (the first two of the
    batch bench.py times) against the reference's fp32 run of the same pairs."""
    fx = golden(name)
    k = fx['scored_pairs']
    data = {key: (v[:k] if torch.is_tensor(v) else v) for key, v in fx['data'].items()}
    out = O.run(fx['state_dict'], fx['config'], data, fx['match_threshold'])
    s, (sr, sc) = out['scores'], fx['sample_stride']
    # same ATen ops on the same B = k batch: rounding noise only (|scores| reaches ~80 on the planted inputs)
    assert (s[:, ::sr, ::sc] - fx['scores_f32_sample']).abs().max() <= 2e-5
    assert (s[:, -1, :] - fx['scores_f32_lastrow']).abs().max() <= 2e-5
    assert (s[:, :, -1] - fx['scores_f32_lastcol']).abs().max() <= 2e-5
    assert (out['context_descriptors0'][:, ::4, ::8] - fx['ctx0_f32_sample']).abs().max() <= 5e-5
    # matches0 / matching_scores0 of the fixture come from the reference's MatchingTrainingModule.forward over the WHOLE batch
    assert torch.equal(out['matches0'], fx['matches0'][:k])
    assert (out['matching_scores0'] - fx['matching_scores0'][:k]).abs().max() <= 2e-5
    rel = (s.double().sum(2) - fx['scores_f64_rowsum']).abs().max() / fx['scores_f64_rowsum'].abs().max()
    assert rel < 2e-5                       # fp32 run against the fp64 reference (ref32-vs-ref64 is ~1e-4 absolute here)
    if 'planted' in name:
        planted = fx['data']['planted_matches0']
        has = planted >= 0
        assert (fx['matches0'][has] == planted[has]).float().mean() > 0.995


def test_planted_matches_are_recovered(golden):
    fx = golden('C1_planted')
    planted = fx['data']['planted_matches0']
    m0 = fx['matches0']
    has = planted >= 0
    assert has.sum() >= 300
    assert torch.equal(m0[has], planted[has])              # every planted pair is recovered


def test_sinkhorn_marginals():
    """Property of the algorithm (optimal_transport.py:20-28): after the v update the column
    marginals of exp(Z+u+v) equal b exactly, the row marginals approximately."""
    torch.manual_seed(0)
    s = torch.randn(2, 30, 41, dtype=torch.float64) * 3
    lp = O.matching_log_probs(s, torch.tensor(1.0, dtype=torch.float64), 200, 1.0)
    m, n = 30, 41
    p = (lp + (-torch.log(torch.tensor(float(m + n))))).exp()
    col = p.sum(1)
    assert torch.allclose(col[:, :-1], torch.full((2, n), 1.0 / (m + n), dtype=torch.float64), atol=1e-12)
    assert torch.allclose(col[:, -1], torch.full((2,), m / (m + n), dtype=torch.float64), atol=1e-12)
    assert torch.allclose(p.sum(2)[:, :-1], torch.full((2, m), 1.0 / (m + n), dtype=torch.float64), atol=1e-6)


def test_extract_matches_ties_first_index():
    s = torch.full((1, 4, 4), -5.0)
    s[0, 0, 1] = s[0, 0, 2] = -0.1          # row tie -> first index (1)
    s[0, 1, 1] = -0.2
    out = O.extract_matches(s, 0.2)
    assert out['matches0'][0, 0].item() == 1
    assert out['matches0'][0, 1].item() == -1      # column 1's best row is 0, not mutual


def test_oracle_equals_staged_reference(golden_fresh):
    """The oracle restatement against the unmodified reference module on fresh seeds (tests/golden/fresh_seeds.pt, minted by
    oracle/gen_golden_fresh.py) - including `use_offset`, a regularisation != 1 and 6 side-info channels, which no other fixture
    covers.  Where the fixture was minted the two agree bit for bit; the bounds allow for another CPU's fp32 rounding at
    |scores| <= 86 (the bounds of test_oracle_matches_reference_big)."""
    from oracle.gen_golden_fresh import SUPERGLUE_CASES, superglue_inputs
    st = golden_fresh['ctx_stride']
    for (seed, kw, nm), want in zip(SUPERGLUE_CASES, golden_fresh['superglue'], strict=True):
        cfg, sd, data = superglue_inputs(seed, kw, nm)
        got = O.run(sd, cfg, data, 0.2)
        assert got['scores'].shape == want['scores'].shape
        assert (got['scores'] - want['scores']).abs().max() <= 2e-5
        for i in (0, 1):
            ctx = got[f'context_descriptors{i}']
            assert (ctx[:, ::st, ::st] - want[f'ctx{i}_sample']).abs().max() <= 1e-5
            assert (ctx.double().sum(-1) - want[f'ctx{i}_f64_sum']).abs().max() <= 1e-5 * ctx.shape[-1]


def test_label_and_loss_oracles_equal_staged_reference(golden_fresh):
    """The two neighbouring steps on fresh seeds against the unmodified reference (tests/golden/fresh_seeds.pt): ground-truth
    matches from a homography (models/gt_matches_generation.py:17-93 vs oracle/gt_matches_oracle.py) bit for bit, and the
    matching loss (utils/losses.py:7-53 vs oracle/loss_oracle.py) to fp32 rounding."""
    from oracle import gt_matches_oracle as G
    from oracle import loss_oracle as L
    from oracle.gen_golden_fresh import LABEL_CASES, label_inputs
    for (seed, (b, n, m)), want in zip(LABEL_CASES, golden_fresh['labels'], strict=True):
        k0, k1, tf, scores = label_inputs(seed, b, n, m)
        g0, g1, _ = G.gt_matches(k0, k1, tf)
        assert torch.equal(g0, want['gt_matches0']) and torch.equal(g1, want['gt_matches1'])
        assert int((g0 >= 0).sum()) > 0
        got = L.criterion({'gt_matches0': g0, 'gt_matches1': g1}, {'scores': scores})
        assert abs(float(got['loss']) - float(want['loss'])) <= 1e-6 * max(1.0, abs(float(want['loss'])))
        assert float(got['metric_loss']) == want['metric_loss'] == 0.0
