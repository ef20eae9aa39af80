"""The training step's hidden dropout and read-removal augmentation against float64 autograd with the same masks.

Dropout: dropout_kernel (dl4vc_b200/csrc/dan_train.cu) keeps element b * ld + k of site j when a counter-based hash of (seed, j, index)
clears p * 2^32; oracle/dan_torch_ref.dropout_keep restates that hash in numpy, and the CPU tests below check that the restatement is a
fair Bernoulli(1 - p) draw, independent across sites, seeds and rows. The GPU tests record the seed each training step uses (or choose
it) and give the float64 reference the same keep masks, so a wrong 1 / (1 - p) scale, a mask undone with the wrong site or row stride in
the backward, or dropout 0 undone in the wrong place behind the post-pool ReLU shows up as a gradient or head error.

Read removal: Basic2DNet._choose_removed picks the reads; the CPU tests check its counts, sets and draw rates. The GPU tests choose the
removed reads themselves (reads 0, R - 1 and one in the middle, every read of a full-coverage candidate, an already-empty slot whose
only change is var_len, the read holding the batch's only token 9, candidates with nothing removed) or take what _choose_removed picks
through model(...), and compare with dan_torch_ref.forward(removed=...). That restates the empty-read encoding as the port documents it
at encode_channel (dl4vc_b200/csrc/dan_kernels_common.cuh): token 0 in the read half, so nn.Embedding's scale_grad_by_freq counts
padding there; the reference half unchanged; the q, strand, ref-agreement, var-agreement and var_len channels zero. These tests show that
the kernels follow that contract. They do not show that the contract matches the reference's own read removal (model.py:633-716), whose
source is not part of this repository; the least certain point is that a removed read's var_len channel is 0.

Bars, kink treatment and batches are those of tests/test_gpu_config_space.py::test_training_step_matches_float64_autograd.
"""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from dl4vc_b200 import model as model_mod
from dl4vc_b200.config import small_config
from dl4vc_b200.factory import build_model
from dl4vc_b200.model import Basic2DNet
from dl4vc_b200.weights import synth_state_dict
from oracle import dan_torch_ref
from test_gpu_config_space import _batch, _check_train_step, _train_reference, _train_step

SIGMAS = 5.0


# ---------------------------------------------------------------------------------------------------------------- the restated hash (CPU)
@pytest.mark.parametrize("p", [0.1, 0.5])
def test_restated_dropout_hash_keeps_each_element_with_probability_1_minus_p(p):
    keep = dan_torch_ref.dropout_keep(p, 12345, 0, 1024, 1024, 1024)           # 2^20 elements
    n = keep.size
    assert abs(keep.mean() - (1 - p)) < SIGMAS * np.sqrt(p * (1 - p) / n), keep.mean()


@pytest.mark.parametrize("p", [0.1, 0.5])
def test_restated_dropout_masks_are_independent_across_sites_seeds_and_rows(p):
    """Two independent Bernoulli(1 - p) masks agree at a rate of p^2 + (1 - p)^2."""
    rows, width = 1024, 1024
    base = dan_torch_ref.dropout_keep(p, 777, 0, rows, width, width)
    pairs = {
        "salt 0 / salt 1": (base, dan_torch_ref.dropout_keep(p, 777, 1, rows, width, width)),
        "seed s / s + 1": (base, dan_torch_ref.dropout_keep(p, 778, 0, rows, width, width)),
        "row b / b + 1": (base[0::2], base[1::2]),                               # disjoint pairs of neighbouring rows
    }
    agree = p * p + (1 - p) * (1 - p)
    for name, (a, b) in pairs.items():
        rate = float((a == b).mean())
        assert abs(rate - agree) < SIGMAS * np.sqrt(agree * (1 - agree) / a.size), (name, rate, agree)


def test_restated_dropout_at_p_0_keeps_everything():
    assert dan_torch_ref.dropout_keep(0.0, 2 ** 62 - 1, 3, 7, 48, 40).all()
    assert [k.shape for k in dan_torch_ref.dropout_masks(small_config(), 3, 0.0, 1)[1]] == [(3, small_config().fc_in_features), (3, 64), (3, 32)]


# ---------------------------------------------------------------------------------------------------------------- _choose_removed (CPU)
_R, _VAR_TOKEN, _OTHER_TOKEN = 12, 2, 1


def _crafted(n_agree, n_other, n_off):
    """Candidate b: n_agree[b] reads carrying the variant proposal (token 2 at column 100), n_other[b] reads covering column 100 with
    token 1, n_off[b] reads that do not cover column 100, the rest empty; each kind in random slots. Returns the uint8 inputs in
    _u8_inputs order and the (B, R) sets of agreeing / covering-but-not-agreeing reads."""
    rng = np.random.default_rng(5)
    B, P = len(n_agree), 201
    reads = np.zeros((B, P, _R), np.uint8)
    var_masks = np.zeros((B, P), np.uint8)
    var_masks[:, 100] = _VAR_TOKEN
    agree = np.zeros((B, _R), bool)
    other = np.zeros((B, _R), bool)
    for b in range(B):
        slots = rng.permutation(_R)
        a, o, f = np.split(slots[: n_agree[b] + n_other[b] + n_off[b]], [n_agree[b], n_agree[b] + n_other[b]])
        reads[b, 40:160, a] = 3
        reads[b, 100, a] = _VAR_TOKEN
        reads[b, 40:160, o] = 3
        reads[b, 100, o] = _OTHER_TOKEN
        reads[b, 120:190, f] = 4
        agree[b, a], other[b, o] = True, True
    z = np.zeros_like(reads)
    u8 = tuple(torch.from_numpy(t) for t in (reads, z, z, np.full((B, P), 1, np.uint8), var_masks.copy(), var_masks))
    return u8, agree, other


def _choose(u8, rm_non_var_reads, rm_var_reads, seed=0, use_masks=True):
    torch.manual_seed(seed)
    out = Basic2DNet._choose_removed(SimpleNamespace(use_reads_ref_var_mask=use_masks), u8, rm_non_var_reads, rm_var_reads)
    return None if out is None else out.numpy().astype(bool)


def _counts():
    """64 candidates: every combination of 0-3 agreeing and 0-4 other covering reads, plus a few that cover nothing."""
    combos = [(a, o) for a in range(4) for o in range(5)]
    rng = np.random.default_rng(11)
    picks = [combos[i % len(combos)] for i in range(64)]
    n_agree, n_other = (np.array(x) for x in zip(*picks))
    n_off = np.minimum(rng.integers(0, 3, 64), _R - n_agree - n_other)
    return n_agree, n_other, n_off


@pytest.mark.parametrize("k_var,k_non", [(1, 0), (2, 0), (3, 0), (0, 1), (0, 2), (0, 4), (2, 4), (3, 3)])
def test_read_removal_removes_exactly_min_k_eligible_distinct_reads_per_candidate(k_var, k_non):
    n_agree, n_other, n_off = _counts()
    u8, agree, other = _crafted(n_agree, n_other, n_off)
    for seed in range(5):
        removed = _choose(u8, k_non, k_var, seed)
        assert removed.shape == agree.shape
        assert not (removed & ~(agree | other)).any(), "a read outside both eligible sets was removed"
        got_var, got_non = (removed & agree).sum(1), (removed & other).sum(1)
        want_var, want_non = np.minimum(k_var, n_agree), np.minimum(k_non, n_other)
        short = np.flatnonzero((got_var != want_var) | (got_non != want_non))
        assert short.size == 0, (f"seed {seed}: {short.size} of {len(n_agree)} candidates lost the wrong number of reads, e.g. candidate "
                                 f"{short[0]}: {got_var[short[0]]} agreeing (want {want_var[short[0]]}), {got_non[short[0]]} other "
                                 f"(want {want_non[short[0]]})")
        nothing = (n_agree == 0) & (n_other == 0)
        assert nothing.any() and not removed[nothing].any(), "a candidate without eligible reads lost one"


@pytest.mark.parametrize("k_var,k_non", [(1, 0), (2, 0), (0, 1), (0, 3)])
def test_read_removal_draws_each_eligible_read_at_rate_k_over_eligible(k_var, k_non):
    """3 agreeing and 5 other covering reads per candidate in random slots: over 40 seeds x 64 candidates, every agreeing read is removed
    at a rate of k_var / 3 and every other one at k_non / 5, each within a binomial bound."""
    B = 64
    u8, agree, other = _crafted(np.full(B, 3), np.full(B, 5), np.full(B, 2))
    hits, seeds = np.zeros((B, _R)), 40
    for seed in range(seeds):
        hits += _choose(u8, k_non, k_var, 100 + seed)
    for kind, mask, rate in (("agreeing", agree, k_var / 3), ("other", other, k_non / 5)):
        # the i-th read of that kind of every candidate: seeds x B draws of a Bernoulli(rate)
        per_rank = np.array([hits[b][mask[b]] for b in range(B)])            # (B, count of that kind)
        got = per_rank.sum(0) / (seeds * B)
        bound = SIGMAS * np.sqrt(rate * (1 - rate) / (seeds * B)) + 1e-12
        assert np.all(np.abs(got - rate) <= bound), (kind, got, rate, bound)


def test_read_removal_is_off_for_k_0_and_without_the_masks():
    u8, _, _ = _crafted(np.full(4, 2), np.full(4, 2), np.zeros(4, int))
    assert _choose(u8, 0, 0) is None
    assert _choose(u8, 2, 1, use_masks=False) is None


# ---------------------------------------------------------------------------------------------------------------- GPU: float64 autograd
@pytest.fixture
def recorded(monkeypatch):
    return _recorder(monkeypatch)


def _recorder(monkeypatch):
    """Records (removed, dropout p, seed) of every training step and substitutes `override`'s removed mask / seed where set."""
    seen, override, orig = [], {}, model_mod._DanTrainFunction.apply

    def apply(module, u8, removed, dropout_p, seed, *params):
        if "removed" in override:
            removed = torch.as_tensor(override["removed"], dtype=torch.uint8).to(u8[0].device).contiguous()
        seed = override.get("seed", seed)
        seen.append((None if removed is None else removed.cpu().numpy().astype(bool), dropout_p, seed))
        return orig(module, u8, removed, dropout_p, seed, *params)

    monkeypatch.setattr(model_mod._DanTrainFunction, "apply", apply)
    return SimpleNamespace(seen=seen, override=override)


def _step_against_reference(name, cfg, arrays, recorded, label=None, **kw):
    """One training step of the kernels against float64 autograd with the masks the step used; weights and d(loss)/d(heads) are seeded
    from `name`, `label` (default `name`) names the case in the TRAIN line."""
    seed = sum(map(ord, name))
    sd = synth_state_dict(cfg, seed=seed)
    B = len(arrays[0])
    cw = np.random.default_rng(seed + 2).standard_normal((B, 27)).astype(np.float32)
    model = build_model(cfg, sd, precision="fp32").train()
    heads = _train_step(model, arrays, cw, **kw)
    (removed, p, dseed), = recorded.seen
    assert p == pytest.approx(cfg.hidden_dropout)
    dropout = dan_torch_ref.dropout_masks(cfg, B, p, dseed) if p > 0 else None
    ref, kink = _train_reference(cfg, sd, arrays, cw, removed=removed, dropout=dropout)
    _check_train_step(label or name, model, heads, ref, kink)
    return removed


DROPOUT_CASES = [
    ("prod_p0.1", small_config()),                                                   # PROD topology, sites 0-2
    ("p0.5", small_config(hidden_dropout=0.5)),                                      # a missing 1 / (1 - p) is a 2x error
    ("fc64_32_32_32", small_config(layer_sizes=(64, 32, 32, 32))),                   # sites 0-4
    ("d96", small_config(pool_combine_dimension=96)),                                # dropout 0 undone before the post-pool ReLU mask
    ("hw_averaged_skip_max", small_config(concat_hw_reads=False, skip_final_maxpool=True)),
]
DROPOUT_SEEDS = [0, 2 ** 62 - 1]         # the ends of the range forward_train_heads draws from


@pytest.mark.gpu
@pytest.mark.parametrize("seed", DROPOUT_SEEDS, ids=["seed0", "seed2^62-1"])
@pytest.mark.parametrize("name,cfg", DROPOUT_CASES, ids=[c[0] for c in DROPOUT_CASES])
def test_training_step_with_dropout_matches_float64_autograd(name, cfg, seed, recorded):
    recorded.override["seed"] = seed
    arrays = tuple(a[[0, 1, 3, 5]] for a in _batch(cfg.num_reads, sum(map(ord, name)) + 1))      # 2 Poisson, 1 full, 1 empty
    # the weights depend on the configuration only, so the two seeds differ in their dropout masks alone
    _step_against_reference("dropout:" + name, cfg, arrays, recorded, label=f"dropout:{name}:seed{seed}")


REMOVAL_CASES = [
    ("prod", small_config(hidden_dropout=0.0)),
    ("reads21", small_config(hidden_dropout=0.0, num_reads=21)),         # a one-read block behind a full one
    ("in144", small_config(hidden_dropout=0.0, embed_dim=64)),           # CinPad 144, the widest encoder rows
]


def _removal_batch(R, seed):
    """_batch's 3 Poisson, 2 full and 1 empty candidate; candidate 1's last slot is emptied (a Poisson depth can reach R) and its read 1
    carries the batch's only token 9. Returns the arrays and the reads to remove."""
    arrays = tuple(a.copy() for a in _batch(R, seed))
    reads, q, s, ref = arrays[:4]
    reads[1, :, R - 1] = q[1, :, R - 1] = s[1, :, R - 1] = 0
    covered = np.flatnonzero(reads[1, :, 1])
    assert covered.size
    reads[1, covered[len(covered) // 2], 1] = 9
    assert (reads == 9).sum() == 1 and not (ref == 9).any()
    removed = np.zeros((6, R), bool)
    removed[0, 0] = True                     # first read of a Poisson candidate
    removed[1, [1, R - 1]] = True            # the token-9 read, an empty slot (only var_len differs from the unremoved encoding)
    removed[3, :] = True                     # every read of a full-coverage candidate
    removed[4, [0, R // 2, R - 1]] = True    # first, middle and last read of the other one; candidates 2 and 5 keep all their reads
    return arrays, removed


@pytest.mark.gpu
@pytest.mark.parametrize("name,cfg", REMOVAL_CASES, ids=[c[0] for c in REMOVAL_CASES])
def test_training_step_with_removed_reads_matches_float64_autograd(name, cfg, recorded):
    arrays, removed = _removal_batch(cfg.num_reads, sum(map(ord, name)) + 1)
    recorded.override["removed"] = removed
    _step_against_reference("removal:" + name, cfg, arrays, recorded)


@pytest.mark.gpu
def test_training_step_with_dropout_and_chosen_reads_removed_matches_float64_autograd(recorded):
    """PROD topology at hidden_dropout 0.1 with the trainer's augmentation through model(...): the seed and the reads
    _choose_removed picks are recorded, not chosen."""
    cfg = small_config()
    arrays = tuple(a[[0, 1, 3, 5]] for a in _batch(cfg.num_reads, 4242))
    torch.manual_seed(3)
    removed = _step_against_reference("dropout+removal:prod", cfg, arrays, recorded, rm_non_var_reads=1, rm_var_reads=1)
    assert removed is not None and removed.any() and not removed[-1].any()      # the empty candidate has no eligible read
