"""CPU checks of the widened rows (SURVEY.md section 8 a2, a6, f1, f3, f4): the oracle against the vectors produced by
the reference's own metric code (tests/golden/make_golden_metrics.py), the retrieval result files against the
reference parser's logic, the Q/K/V store, and the host logic of the batched drivers."""
import os
import zlib

import pytest
import torch

from conftest import checksum, clip_images, dino_images, gram_features, ip_images
from oracle import aas_oracle as O


# ------------------------------------------------------------------------------------------------------
# oracle vs the reference run
# ------------------------------------------------------------------------------------------------------
def test_oracle_ip_adapter_matches_reference_run(metrics_golden):
    for case in metrics_golden["ip_adapter"]["cases"]:
        imgs = ip_images(case["seed"], case["ip_tokens"], case["n_adapters"], case["alpha"])
        for im, cs in zip(imgs, case["checksums"]):
            assert [checksum(im[0])] + [checksum(t) for t in im[1] + im[2]] == cs
        (qa, ka, va), (qb, kb, vb) = imgs
        t0 = O.aas_ip_adapter_score(qa, ka, va, qb, kb, vb, tier="T0")
        assert t0 == pytest.approx(case["score_fp32_math"], rel=5e-5)
        assert case["score_native_f16"] == pytest.approx(t0, rel=2e-3)
        # the reference's MSE branch for this path is not executable (diffsim/diffsim.py:191-192)
        assert case["mse_error"] == "AttributeError"


def test_oracle_clip_cross_matches_reference_run(metrics_golden):
    c = metrics_golden["clip_cross"]
    (qa, ka, va), (qb, kb, vb), w, b = clip_images()
    assert [[checksum(t) for t in im] for im in ((qa, ka, va), (qb, kb, vb), (w, b))] == c["checksums"]
    shape = (1, qa.shape[2], qa.shape[1] * qa.shape[3])
    got = O.clip_cross_score(qa, ka, va, qb, kb, vb, c["scale"], shape, w, b)
    assert got == pytest.approx(c["score_fp32_math"], rel=5e-5)
    a_on_b = O.clip_attention_calc(qa, kb, vb, c["scale"], shape, w, b)
    assert (a_on_b - c["attention_calc_a_on_b_fp32"].double()).abs().max().item() < 2e-5


def test_oracle_dino_cross_matches_reference_run(metrics_golden):
    c = metrics_golden["dino_cross"]
    A, B = dino_images()
    assert [[checksum(t) for t in im] for im in (A, B)] == c["checksums"]
    got = O.aas_pair_score(*A, *B, mode="cosine", scale=c["attention_head_size"] ** -0.5, tier="T0")
    assert got == pytest.approx(c["score_fp32_math"], rel=5e-5)


def test_oracle_gram_matches_reference_run(metrics_golden):
    c = metrics_golden["gram"]
    fa, fb = gram_features()
    assert [checksum(fa), checksum(fb)] == c["checksums"]
    assert (O.gram_matrix(fa) - c["gram_a_fp32"].double()).abs().max().item() < 1e-2   # fp32 sums of 384 products ~ 600
    assert O.gram_similarity(fa, fb) == pytest.approx(c["score_fp32_math"], rel=2e-6)


# ------------------------------------------------------------------------------------------------------
# retrieval result files (retrieval_vis.py:57-68,121-132,197)
# ------------------------------------------------------------------------------------------------------
def _score_matrix(n, seed=0):
    g = torch.Generator().manual_seed(seed)
    s = torch.rand(n, n, generator=g)
    return (s + s.t()) / 2


def test_retrieval_files_are_what_the_reference_parser_reads(tmp_path):
    from diffsim_b200 import retrieval as R

    names = [f"{c:03d}_{i}" for c in range(3) for i in range(1, 5)]   # Sref-like: <style>_<image id>
    s = _score_matrix(len(names))
    paths = R.write_retrieval_results(s, names, str(tmp_path), topk=5)
    assert len(paths) == len(names) and os.path.exists(os.path.join(tmp_path, "001", "3.txt"))
    order, vals = R.ranked_indices(s, 5)
    for qi in (0, 5, 11):
        got = R.read_retrieval_result(paths[qi], limit=4)
        want = [os.path.join(names[j].split("_")[0], names[j].split("_")[1] + ".png") for j in order[qi, :4].tolist()]
        assert got == want
        assert qi not in order[qi].tolist()                      # the query itself is never retrieved
        assert (vals[qi][:-1] >= vals[qi][1:]).all()             # best first
    # the IP variant of the parser skips image id 1 (retrieval_vis.py:197)
    got = R.read_retrieval_result(paths[0], limit=4, skip_first_id=True)
    assert all(not p.endswith(os.sep + "1.png") for p in got)
    # flat (COCO) layout
    flat = [f"{i:012d}" for i in range(6)]
    p2 = R.write_retrieval_results(_score_matrix(6, 1), flat, str(tmp_path / "coco"), topk=3, layout="flat")
    assert R.read_retrieval_result(p2[0], layout="flat")[0].endswith(".jpg")
    # distances (mse): smaller is closer
    o_small, _ = R.ranked_indices(s, 1, larger_is_closer=False)
    s2 = s.clone()
    s2.fill_diagonal_(float("inf"))
    assert o_small[:, 0].tolist() == s2.argmin(dim=1).tolist()
    with pytest.raises(ValueError):
        R.write_retrieval_results(s, ["a_b_c"] * len(names), str(tmp_path / "bad"))


def test_retrieval_accuracy_on_block_structure():
    from diffsim_b200 import retrieval as R

    labels = [c for c in range(5) for _ in range(4)]
    y = torch.tensor(labels)
    s = (y[:, None] == y[None, :]).float() + 0.01 * _score_matrix(20)
    acc = R.retrieval_accuracy(s, labels, topk=3)
    assert acc["hit@k"] == 1.0 and acc["precision@k"] == 1.0 and acc["k"] == 3


def test_qkv_store_round_trip(tmp_path):
    from diffsim_b200 import retrieval as R, synth
    from diffsim_b200.scoring import QKVCache

    m = synth.SynthModel(2, 2, 64, 40, seed=1)
    images, _ = synth.make_pairs(m, 2, torch.float16, seed=3)
    cache = QKVCache.from_images(images)
    key = R.store_key("sd15", "up_blocks", [0], 600, "2333", 512)
    path = str(tmp_path / "cache.safetensors")
    R.save_qkv(path, cache, ["a", "b", "c", "d"], key)
    back, names = R.load_qkv(path, expect_key=key)
    assert names == ["a", "b", "c", "d"] and back.shape == cache.shape
    for t0, t1 in zip((cache.q, cache.k, cache.v), (back.q, back.k, back.v)):
        assert t1.stride() == t0.stride() and torch.equal(t0, t1)      # the hook's head-split view layout survives
    with pytest.raises(ValueError, match="different model"):
        R.load_qkv(path, expect_key=R.store_key("sd15", "up_blocks", [0], 500, "2333", 512))
    with pytest.raises(ValueError):
        R.save_qkv(path, cache, ["a"], key)


# ------------------------------------------------------------------------------------------------------
# drivers: host logic (the scoring call is replaced by the oracle; the CUDA path is covered by -m gpu)
# ------------------------------------------------------------------------------------------------------
class _CountingScorer:
    def __init__(self):
        from diffsim_b200 import synth

        self.m = synth.SynthModel(1, 2, 64, 40, seed=4)
        self.base = self.m.new_base(torch.Generator().manual_seed(1))
        self.calls = []

    def diffsim_value(self, image, img_size, prompt, target_block, target_layer, target_step, seed="2333", device="cpu"):
        self.calls.append(image)
        concept, _, alpha = image.partition("@")
        g = torch.Generator().manual_seed(zlib.crc32(image.encode()) & 0xFFFF)
        return self.m.image(self.base, float(alpha), torch.float16, "sd", g)


def test_drivers_extract_each_image_once_and_decide_like_the_reference(monkeypatch):
    from diffsim_b200 import drivers, ops

    def fake_triplets(q, k, v, trip, similarity="cosine", scale=None, round_scores=False, want_flags=True):
        ab, ac = [], []
        for r, l, rt in trip.tolist():
            ab.append(O.aas_pair_score(q[r], k[r], v[r], q[l], k[l], v[l], mode=similarity))
            ac.append(O.aas_pair_score(q[r], k[r], v[r], q[rt], k[rt], v[rt], mode=similarity))
        c, c2, flags = O.twoafc(ab, ac, similarity)
        return (torch.tensor(ab), torch.tensor(ac), torch.tensor([c, c2], dtype=torch.int32),
                torch.tensor(flags, dtype=torch.uint8))

    monkeypatch.setattr(ops, "aas_triplets", fake_triplets)
    sc = _CountingScorer()
    trips = [("x@1.0", "x@0.9", "x@0.2"), ("x@1.0", "x@0.3", "x@0.8"), ("x@0.9", "x@1.0", "x@0.2")]
    r = drivers.run_2afc(sc, trips, device="cpu")
    assert sorted(sc.calls) == sorted({im for t in trips for im in t})       # 5 distinct images, each extracted once
    assert r.total == 3 and r.correct == 2 and r.flags.tolist() == [1, 0, 1]
    assert r.accuracy == pytest.approx(200.0 / 3)
    assert drivers.format_report("CUTE", r)[0] == "Current total samples: 3"
    # NIGHTS: predicted (1 = left closer) compared with the annotators' vote (night_main.py:157-163)
    rows = [(a, b, c, v) for (a, b, c), v in zip(trips, (1, 1, 0))]
    rn = drivers.run_nights(sc, rows, device="cpu")
    assert rn.correct == 1 and rn.total == 3
    # mse flips the comparison (cute_main.py:196-200)
    rm = drivers.run_2afc(sc, trips, similarity="mse", device="cpu")
    assert rm.flags.tolist() == [1, 0, 1]


def test_ensemble_majority_vote_rules():
    """cute_main.py:187-195 and night_main.py:148-152: ties vote for the positive; two of three decide."""
    from diffsim_b200 import drivers

    t = torch.tensor
    diff = (t([0.9, 0.2, 0.5, 0.1]), t([0.1, 0.8, 0.5, 0.3]))     # votes 1, 0, 1 (tie), 0
    clip = (t([0.7, 0.9, 0.1, 0.2]), t([0.6, 0.1, 0.9, 0.9]))     # votes 1, 1, 0, 0
    dino = (t([0.1, 0.1, 0.4, 0.9]), t([0.5, 0.5, 0.3, 0.1]))     # votes 0, 0, 1, 1
    # sums: 2, 1, 2, 1 -> correct: yes, no, yes, no
    assert drivers.ensemble_votes([diff, clip, dino]) == 2
    # NIGHTS: vote 1 needs sum >= 2, vote 0 needs sum <= 1
    assert drivers.ensemble_votes([diff, clip, dino], votes=t([1, 0, 0, 1])) == 2
    with pytest.raises(ValueError):
        drivers.ensemble_votes([diff, clip])
