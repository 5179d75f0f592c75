"""Search the fused actor's Philox Gaussian draws (``oracle_np.philox_normal_pair``) for keys whose 24-bit words hit the
tails of Box-Muller, and print them as the ``TAIL_TARGETS`` table of tests/test_random_streams_cpu.py.

    python tests/golden/gen_random_tail_targets.py

Targets: the radius word k1 at 2^24 - 1 (u1 = 1 exactly, r = 0), at the next eight u1 values below 1 (k1 = 2^24 - 2j:
the float32 add of 0.5 rounds k1 = 2^24 - 2j + 1 to the same u1) and at 0 and 1 (the largest radii); the angle word k2 at
0, 2^22, 2^23, 3 2^22 (theta = 0 and the quadrant edges) and 2^24 - 1 (just below 2 pi).  Each hit has probability 2^-24
per draw, so the search scans about 2^26 environments x 8 (stream, pair) combinations: about 30 s.
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from oracle import oracle_np as o  # noqa: E402

SEED = 0xD1B54A32D192ED03          # both key words non-zero, above 2^63
STEP = 0x80000005                  # above 2^31
ENV0 = 2 ** 32 - 2 ** 25           # the scan crosses the 2^32 word boundary of the env id
K1_TARGETS = [2 ** 24 - 1] + [2 ** 24 - 2 * j for j in range(1, 9)] + [0, 1]
K2_TARGETS = [0, 2 ** 22, 2 ** 23, 3 * 2 ** 22, 2 ** 24 - 1]


def search(chunk=2 ** 21):
    found = {}
    env0 = ENV0
    while len(found) < len(K1_TARGETS) + len(K2_TARGETS):
        env = np.arange(env0, env0 + chunk, dtype=np.uint64)
        for stream in (7, 8):
            for blk in range(4):
                k1, k2, _, _ = o.philox_normal_pair(SEED, env, STEP, blk, stream)
                for word, ks, targets in (("k1", k1, K1_TARGETS), ("k2", k2, K2_TARGETS)):
                    for k in targets:
                        if (word, k) not in found:
                            hit = np.nonzero(ks == k)[0]
                            if hit.size:
                                found[(word, k)] = (int(env[hit[0]]), stream, blk)
        env0 += chunk
    return found


if __name__ == "__main__":
    found = search()
    print("TAIL_TARGETS = [   # (word, k, env id, stream, blk); seed 0x%X, step 0x%X" % (SEED, STEP))
    for word, targets in (("k1", K1_TARGETS), ("k2", K2_TARGETS)):
        for k in targets:
            env, stream, blk = found[(word, k)]
            print("    (%r, 0x%06X, 0x%X, %d, %d)," % (word, k, env, stream, blk))
    print("]")
