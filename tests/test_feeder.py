"""CPU: host logic either side of the hot path — collation of dataset items into uint8 batches, the trainer's score post-ops and
the VCF INFO field (SURVEY §8f rows 1-2), checked against what the reference's own functions return (stored goldens and literals)."""
import numpy as np
import pytest
import torch

from dl4vc_b200.feeder import HostBatch, scores_from_heads, format_vcf_info, splice_vcf_records
from dl4vc_b200.synth import make_pileups


def _items(batch):
    out = []
    for i in range(len(batch.reads)):
        out.append({"reads": batch.reads[i].astype(np.int64), "q-scores": batch.q_scores[i], "strands": batch.strands[i], "ref": batch.ref[i],
                    "ref_mask": batch.ref_masks[i], "var_mask": batch.var_masks[i], "name": "chr1:%d" % i,
                    "vcfrec": "chr1\t%d\t.\tA\tT\t.\t.\t.\tGT\t0/1" % (1000 + i)})
    return out


def test_host_batch_collates_dataset_items_losslessly():
    b = make_pileups(5, seed=3, coverage="poisson")
    hb = HostBatch(8, pin=False).fill(_items(b))
    r, ref, q, s, rm, vm = hb.tensors()
    assert r.dtype == torch.uint8 and tuple(r.shape) == (5, 201, 100)
    assert np.array_equal(r.numpy(), b.reads) and np.array_equal(q.numpy(), b.q_scores) and np.array_equal(s.numpy(), b.strands)
    assert np.array_equal(ref.numpy(), b.ref) and np.array_equal(rm.numpy(), b.ref_masks) and np.array_equal(vm.numpy(), b.var_masks)
    assert hb.meta[4][0] == "chr1:4"
    with pytest.raises(ValueError):
        HostBatch(2, pin=False).fill(_items(b))
    bad = _items(b)[:1]
    bad[0]["reads"] = bad[0]["reads"].T
    with pytest.raises(ValueError):
        HostBatch(2, pin=False).fill(bad)


def test_scores_match_trainer_post_ops():
    g = torch.Generator().manual_seed(0)
    heads = torch.randn(17, 27, generator=g) * 3
    bin_score, vt = scores_from_heads(heads)
    # trainer.py:617-623
    want_bin = 1.0 - torch.nn.functional.softmax(heads[:, 0:2], dim=1)[:, 0]
    want_vt = torch.nn.functional.softmax(heads[:, 2:5], dim=1)
    assert torch.equal(bin_score, want_bin) and torch.equal(vt, want_vt)
    assert torch.allclose(vt.sum(1), torch.ones(17), atol=1e-6)


def test_vcf_info_field_matches_reference_writer():
    """The lines the reference's append_vcf_records (utils.py:162-178) appends for these two records, one per record: the ID column
    replaced by the score field. The literals are splice_vcf_records' output for these records, which this test found line for line
    equal to the file append_vcf_records wrote when it still ran the reference writer (from commit 8ad7367 on)."""
    b = np.array([0.25, 0.99999999]); v = np.array([[0.75, 0.125, 0.125], [1e-9, 0.5, 0.5]])
    recs = ["chr1\t100\t.\tA\tT\t.\t.\t.\tGT\t0/1\n", "chr2\t200\t.\tG\tGA\t.\t.\t.\tGT\t1/1"]
    lines = splice_vcf_records(recs, b, v)
    assert lines == ["chr1\t100\tBP=0.25000000;NV=0.75000000;HV=0.12500000;OV=0.12500000\tA\tT\t.\t.\t.\tGT\t0/1",
                     "chr2\t200\tBP=0.99999999;NV=0.00000000;HV=0.50000000;OV=0.50000000\tG\tGA\t.\t.\t.\tGT\t1/1"]
    assert format_vcf_info(b, v)[1] == "BP=0.99999999;NV=0.00000000;HV=0.50000000;OV=0.50000000"
    with pytest.raises(AssertionError):
        splice_vcf_records(["chr1\t100\trs1\tA\tT"], b[:1], v[:1])


def test_native_vcf_info_formatting_matches_python():
    """dan_format_vcf_info (host code in the C-ABI library, no GPU needed) against the reference's '%.8f' formatting (utils.py:171-176)."""
    from dl4vc_b200.feeder import format_vcf_info, format_vcf_info_native
    rng = np.random.default_rng(5)
    s = rng.random((2000, 4)).astype(np.float32)
    s[0] = [0.0, 1.0, 0.0, 0.0]
    s[1] = [1.0, 0.0, 1.0, 0.0]
    s[2] = [0.999999995, 5e-9, 0.123456785, 0.5]          # rounding at the 8th decimal
    want = format_vcf_info(s[:, 0], s[:, 1:])
    got = format_vcf_info_native(s)
    assert got == want
    assert all(len(x) == 55 for x in got)
    assert format_vcf_info_native(np.zeros((0, 4), np.float32)) == []
    import pytest
    with pytest.raises(RuntimeError):
        format_vcf_info_native(np.full((1, 4), 1.5, np.float32))


def test_mask_vector_decode_matches_reference_goldens():
    """dan_make_mask_vectors (host code in the C-ABI library) against 600 records run through the REAL get_read_mask_vectors
    (dl4vc/dataset.py:112-250; tests/golden/mask_vectors.npz from oracle/make_mask_goldens.py): SNPs, deletes with and without gap
    columns, inserts (ALT clipped to 51 bases), rewinds past gap columns at the centre, and every record the reference raises on."""
    import os
    import pytest
    from dl4vc_b200.feeder import make_mask_vectors
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mask_vectors.npz"))
    xs, ys = [str(a) for a in g["ref_alleles"]], [str(a) for a in g["var_alleles"]]
    rm, vm, st = make_mask_vectors(xs, ys, g["references"], strict=False)
    ok = g["ok"].astype(bool)
    assert np.array_equal(st == 0, ok), "the set of records the reference raises on differs"
    assert np.array_equal(rm[ok], g["ref_masks"][ok]) and np.array_equal(vm[ok], g["var_masks"][ok])
    assert not rm[~ok].any() and not vm[~ok].any()
    assert ok.sum() > 400 and (~ok).sum() > 40
    with pytest.raises(RuntimeError):
        make_mask_vectors(xs, ys, g["references"], strict=True)
    good = np.nonzero(ok)[0][:50]
    rm2, vm2, st2 = make_mask_vectors([xs[i] for i in good], [ys[i] for i in good], g["references"][good])
    assert not st2.any() and np.array_equal(rm2, g["ref_masks"][good])


def test_decode_records_matches_reference_loader():
    """dan_decode_records (batched C decode of raw records) against the per-item dicts of the REAL ContextDatasetFromNumpy.__getitem__
    (tests/golden/feeder.npz, oracle/make_feeder_goldens.py): tiles, reference, proposal masks and every scalar exactly; pileups deeper
    than 100 reads (sampled with an unseeded np.random.choice in the reference) are checked for the sampling properties."""
    import os
    from conftest import GOLDEN_DIR
    from dl4vc_b200.feeder import RECORD_DTYPE, HostBatch, RecordFile, decode_records
    g = np.load(os.path.join(GOLDEN_DIR, "feeder.npz"))
    rf = RecordFile(g["records"])
    n = len(rf)
    raised = [str(r) for r in g["raised"]]
    ok = np.array([r == "" for r in raised])
    batch, sc = decode_records(rf, np.arange(n), HostBatch(n, pin=False), seed=5, strict=False)
    assert np.array_equal(sc["status"] != 0, ~ok), "records the reference raises on <-> non-zero status"
    with pytest.raises(ValueError, match="cannot be decoded"):
        decode_records(rf, np.arange(n), HostBatch(n, pin=False))
    depth = sc["num_reads"]
    shallow = ok & (depth <= 100)
    deep = ok & (depth > 100)
    assert shallow.sum() >= 15 and deep.sum() >= 10
    got = {"reads": batch.reads.numpy(), "q_scores": batch.q.numpy(), "strands": batch.strands.numpy(), "ref": batch.ref.numpy(),
           "ref_mask": batch.ref_masks.numpy(), "var_mask": batch.var_masks.numpy()}
    for k, a in got.items():
        assert np.array_equal(a[shallow], g["out_" + k][shallow]), k
    for k in ("ref", "ref_mask", "var_mask"):
        assert np.array_equal(got[k][deep], g["out_" + k][deep]), k
    for k in ("label", "num_reads", "is_snp", "var_type", "var_base_enum", "var_ref_enum", "blacklist"):
        assert np.array_equal(sc[k][ok].astype(np.float64), g["s_" + k][ok]), k
    for k in ("allele_freq", "coverage"):      # depend on the sampled rows: exact for shallow pileups
        assert np.array_equal(sc[k][shallow].astype(np.float64), g["s_" + k][shallow].astype(np.float32).astype(np.float64)), k
    assert sc["blacklist"][1] == 1 and not got["ref_mask"][1].any()
    # deep pileups: 100 columns = a sorted subset of the first num_reads stored rows, the same rows in all three tiles, deterministic in (seed, index)
    recs = g["records"].view(RECORD_DTYPE).reshape(-1)
    for i in np.flatnonzero(deep):
        rows, qrows, srows = recs[i]["single_reads"], recs[i]["q-scores"], recs[i]["strand"]
        last = -1
        for j in range(100):
            col = got["reads"][i][:, j]
            cands = [r for r in range(last + 1, int(depth[i])) if np.array_equal(rows[r], col) and np.array_equal(qrows[r], got["q_scores"][i][:, j])
                     and np.array_equal(srows[r], got["strands"][i][:, j])]
            assert cands, f"record {i}: column {j} is not a later stored row"
            last = cands[0]
    again, _ = decode_records(rf, np.arange(n), HostBatch(n, pin=False), seed=5, strict=False)
    assert np.array_equal(again.reads.numpy(), got["reads"])
    other, _ = decode_records(rf, np.arange(n), HostBatch(n, pin=False), seed=6, strict=False)
    assert not np.array_equal(other.reads.numpy()[deep], got["reads"][deep])


def _call_golden():
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "genotype_calls.npz"))
    names = ("snp", "snp_zygo", "indel", "indel_zygo", "long_indel", "long_indel_zygo", "delete", "delete_zygo")
    sets = []
    for k in range(int(g["num_sets"])):
        ok = g["defined0"] if k == 0 else np.ones(len(g["scores"]), bool)      # the script raises on short deletes with its default thresholds
        sets.append((dict(zip(names, g["thr%d" % k].tolist())), g["gt%d" % k], g["q%d" % k], ok))
    return g["scores"], g["ref_len"], g["var_len"], sets


def test_genotype_calls_match_reference_format_vcf():
    """Host restatement of tools/format_vcf.py:107-138 against the real script run on 3000 scored records (oracle/make_call_goldens.py)."""
    from dl4vc_b200.feeder import genotype_calls
    scores, rl, vl, sets = _call_golden()
    for thr, gt, q, ok in sets:
        got_gt, got_q = genotype_calls(scores, rl, vl, **thr)
        assert np.array_equal(got_gt[ok], gt[ok]) and np.array_equal(got_q[ok], q[ok])


@pytest.mark.gpu
def test_genotype_calls_on_device_match_reference_format_vcf():
    import torch
    from dl4vc_b200.feeder import genotype_calls_on_device
    scores, rl, vl, sets = _call_golden()
    dev = torch.device("cuda", 0)
    s = torch.from_numpy(scores).to(dev); r = torch.from_numpy(rl).to(dev); v = torch.from_numpy(vl).to(dev)
    for thr, gt, q, ok in sets:
        got_gt, got_q = genotype_calls_on_device(s, r, v, **thr)
        assert np.array_equal(got_gt.cpu().numpy()[ok], gt[ok]) and np.array_equal(got_q.cpu().numpy()[ok], q[ok])
