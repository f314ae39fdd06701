"""Run in a process of its own with one environment switch set (the switches are read once per process):
a fixed subset of test_gpu_initial_sort.py's cases against the same reference.  Exits non-zero on a mismatch.
Used by test_gpu_initial_sort.py."""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "dsm-framework_b200"))
sys.path.insert(0, HERE)


def main():
    import numpy as np
    import test_gpu_initial_sort as t
    # whole sweep tiles and a partial last tile (3 M pairs), the tile and heads-chunk edges, every alphabet width,
    # a carried and an uncarried key, and a text keyed in word ranges
    for sigma in (5, 8, 255):
        for n in (2, 129, 257, 4095, 4097, 3_000_017):
            t.run(t.random_docs(n, t.alphabet(sigma, sigma), seed=n * 7 + sigma))
        for fkb in (0, 64):
            t.run(t._shaped_docs("around_first_key", sigma, t.shape(np.append(t.alphabet(sigma, 100 + sigma), np.uint8(0)), fkb)[2]), fkb)
        t.run(t.random_docs(100_003, t.alphabet(sigma, sigma), seed=sigma), word_cuts=[127, 128, 129, 1000])
    print("INITIAL_SORT_VARIANT_OK")


if __name__ == "__main__":
    main()
