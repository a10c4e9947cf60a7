"""oracle DBoW2 transform (oracle/bow.h) == the reference's own DBoW2 compiled in oracle/_ref/libref.so, on a synthetic vocabulary in ORBvoc.txt's format.
The reference's results are read from tests/golden/ref_oracle_bow.npz (tests/refgold.py)."""
import numpy as np
import pytest

from cubemapslam_b200 import synth
from oracle import ref
from tests.refgold import RECORD, gold  # noqa: F401


@pytest.mark.parametrize("k,L,levelsup", [(10, 4, 2), (6, 5, 4), (10, 3, 4)])
def test_transform_matches_reference_dbow2(oracle, tmp_path, gold, k, L, levelsup):
    voc = synth.vocabulary(k=k, L=L, seed=k + L)
    path = tmp_path / "voc.txt"
    synth.write_vocabulary_text(voc, str(path))
    rv = ref.RefVocabulary(str(path)) if RECORD else None
    key = "k%d_L%d_up%d" % (k, L, levelsup)
    assert gold.value("size_" + key, lambda: rv.size()) == k ** L
    ov = oracle.Vocabulary(k, L, voc["parent"], voc["is_leaf"], voc["desc"], voc["weight"])
    rng = np.random.default_rng(1)
    # features near words (realistic) plus pure noise
    leaves = np.nonzero(voc["is_leaf"])[0]
    f1 = voc["desc"][rng.choice(leaves, 1500)] ^ np.packbits(rng.random((1500, 256)) < 0.05, axis=1, bitorder="little")
    feats = np.concatenate([f1, rng.integers(0, 256, (500, 32), dtype=np.uint8)])
    bw, bv, node, word = ov.transform(feats, levelsup)
    # BowVector: same words, bit-identical L1-normalised doubles; FeatureVector membership of every feature
    assert gold.same("transform_" + key, (bw, bv, node), lambda: rv.transform(feats, levelsup))
    assert abs(bv.sum() - 1.0) < 1e-12 and len(bw) > 300
    assert (node[word >= 0] >= 0).mean() > 0.95                           # a few stopped words (weight 0) are excluded like in the reference
