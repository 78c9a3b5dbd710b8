"""CPU test of the label table the batch remap reads (dq_host_build_label_table): for every entry of the sorted palette,
the caller's index of the last palette entry with that 24-bit colour -- what the reference's
mapQuantPixelsToColortableIndexes gives a pixel mapped to that entry.  No device work."""
import numpy as np


def test_host_label_table_matches_oracle(pkg, oracle):
    dq = pkg.DivQuant.__new__(pkg.DivQuant)
    dq.lib = pkg.load_library()
    rng = np.random.default_rng(31)
    for trial in range(200):
        k = int(rng.integers(1, 601))
        pal = rng.integers(0, 1 << 24, k, dtype=np.uint32)
        if trial % 2:  # duplicate words
            pal[rng.integers(0, k, k // 2 + 1)] = pal[rng.integers(0, k)]
        if trial % 5 == 0:  # greys and a coarse lattice: many equal sums and duplicates
            g = rng.integers(0, 4, (k, 3)) * 64
            pal = ((g[:, 0] << 16) | (g[:, 1] << 8) | g[:, 2]).astype(np.uint32)
            pal[::3] = (rng.integers(0, 256, pal[::3].size) * 0x010101).astype(np.uint32)
        if trial % 3 == 0:  # alpha bits: the same colour under several alphas counts as one colour
            pal |= (rng.integers(0, 256, k).astype(np.uint32) << 24)
        srt, _ = oracle.build_search_tables(pal)
        lab = dq.host_build_label_table(pal)
        assert np.array_equal(lab, oracle.colortable_indexes(srt, pal)), trial
        assert np.array_equal(pal[lab] & 0xFFFFFF, srt & 0xFFFFFF), trial
