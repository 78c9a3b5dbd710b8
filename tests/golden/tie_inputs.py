"""Inputs that drive the tie audit's recovery steps (resolver, forced cut) on every entry path.

Shared by tests/test_tie_inputs.py, which checks on the CPU model that each input still exercises what it was chosen
for, and tests/test_gpu_tie_paths.py, which runs them on the device.  All images are oracle.generate(1, 1920, 1080, seed)
(G1, 1080p) unless a tag says otherwise.

`int_wrong`: the exact-integer palette alone differs from the reference's (oracle quant_varpart_fast with
exact_counts=True != the restatement), so a path that skips the resolver returns a wrong palette.
`forced`: the resolver model needs at least one forced cut (the reference cuts a node on the other side of an integer).
"""

# golden frames (tests/golden/frames.npz) whose audit fires: (tag, seed)
C4_FLAGGED = (12410, 12830, 12832, 13124)        # 1920x1080, K=64; 12832 needs a forced cut
C4_FORCED = 12832
C4_INT_WRONG = (12410, 12830, 13124)              # one LSB off without the resolver
C4_CLEAN = (12411, 12831, 12833, 13125)           # neighbours the audit leaves alone
BENCH_FLAGGED = (12359, 12519, 12545)            # 3840x2160, K=256
BENCH_CLEAN = 12345

# quant_varpart_fast, rows=1 (one row of 2 073 600 pixels): (seed, num_bits, dec_factor, K, int_wrong, forced)
VARPART_1D = (
    (12345, 8, 3, 256, True, False),
    (12347, 7, 2, 256, True, False),
    (12356, 7, 2, 256, True, False),
    (12369, 7, 2, 256, True, False),
    (12371, 8, 3, 256, True, False),
    (12374, 7, 2, 256, True, False),
    (12394, 8, 3, 256, True, False),
    (12397, 7, 2, 256, True, False),
    (12402, 7, 1, 64, True, False),
    (12364, 7, 2, 256, False, True),
    (12348, 8, 3, 256, False, False),
    (12359, 7, 2, 256, False, False),
)

# quant_varpart_fast, rows=1080, cols=1920: the reference samples inPixels[ic + ir*numRows], so the sampled pixels (and
# the flagged inputs) differ from the one-row form
VARPART_2D = (
    (12348, 8, 3, 256, True, False),
    (12350, 8, 3, 256, True, False),
    (12352, 7, 2, 256, True, False),
    (12356, 7, 2, 256, True, False),
    (12398, 7, 2, 256, True, False),
    (12365, 8, 3, 256, True, True),
    (12391, 8, 2, 64, False, True),
    (12350, 6, 1, 64, False, False),
    (12368, 8, 3, 256, False, False),
)
