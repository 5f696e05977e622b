"""Fixture of the reference's known-answer test for the WORDS matcher (opensfm/test/test_matching.py:23-70), made from
the reference's own vocabulary file, which is not part of this repository:

    python tests/golden/make_words_golden.py <OpenSfM checkout>/opensfm/data/bow/bow_hahog_root_uchar_10000.npz

Features as in `example_features` (seeded), their `bow_words_to_match` = 50 closest visual words computed the way
opensfm/bow.py `map_to_words(..., "BRUTEFORCE")` does (cv2 BruteForce knnMatch against the vocabulary; the test itself
asks for FLANN, the approximate version of the same query).  Saved: the seed and the word matrices."""
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SEED, NFEATURES, NUM_WORDS = 0, 1000, 50


def example_features(seed=SEED, nfeatures=NFEATURES):
    rng = np.random.RandomState(seed)
    f1 = rng.normal(size=(nfeatures, 128)).astype(np.float32)
    f1 /= np.linalg.norm(f1)
    f2 = f1 + rng.normal(size=f1.shape).astype(np.float32) / 500.0
    f2 /= np.linalg.norm(f2)
    return f1, f2


if __name__ == "__main__":
    words = np.load(sys.argv[1])["words"].astype(np.float32)
    f1, f2 = example_features()
    matcher = cv2.DescriptorMatcher_create("BruteForce")

    def closest(f):
        return np.array([[n.trainIdx for n in m] for m in matcher.knnMatch(f, words, k=NUM_WORDS)], dtype=np.int16)

    w1, w2 = closest(f1), closest(f2)
    np.savez_compressed(os.path.join(HERE, "words_golden.npz"), seed=SEED, nfeatures=NFEATURES, w1=w1, w2=w2)
    print("vocabulary", words.shape, "distinct first words of image 2:", len(np.unique(w2[:, 0])))
