"""Seeded remap inputs on which the tie-break decides the output, and a plain numpy reference of the remap.

The reference's map_colors_mps returns, for every pixel, argmin over (dist, rank) in the palette sorted by r+g+b, with
rank(s) = 0, rank(s+d) = 2d-1, rank(s-d) = 2d from the start index s = lut_init[r+g+b] (csrc/dq_map.cu).  The rank only
matters when several entries lie at the minimal distance, and the device formulations differ exactly there.  These
generators put most pixels on such ties:

* lattice palettes (levels every `step`, a ball of the lattice around a random centre, shuffled, optional duplicate
  words and alpha bytes) with pixels half a step off lattice points: equidistant from 2, 4 or 8 entries;
* star palettes: entries on the shell |v|^2 = 9 t^2 around random centres, padded with lattice entries; pixels at the
  centres, equidistant from every entry of their star;
* grey palettes: entries (g+d, g-d, g) and their permutations, so that every entry has an equal-sum neighbour; pixels
  grey or nearly so.

Shared by tests/test_remap_tie_inputs.py (CPU: the oracle's walk, its brute force and nearest_dist_rank agree, and
every input keeps its share of tie pixels) and tests/test_gpu_remap_paths.py (each device formulation against the
oracle).  Plain numpy, no GPU.
"""
import numpy as np

# palette sizes around every switch of the device remap: 512 (integer arg-min), 8192 (shared-memory palette) and
# 11 466 (the most a 20-byte-per-entry shared-memory palette plus its LUT can hold in 227 KB)
KS = (1, 2, 3, 255, 256, 257, 511, 512, 513, 8191, 8192, 8193, 11467, 16384)

# integer vectors with |v|^2 = 9: (+-3, 0, 0) and (+-2, +-2, +-1) in every order
_SHELL = np.array([v for v in np.ndindex(7, 7, 7) if sum((c - 3) ** 2 for c in v) == 9]) - 3


def pack(rgb):
    rgb = np.asarray(rgb, np.int64)
    return ((rgb[..., 0] << 16) | (rgb[..., 1] << 8) | rgb[..., 2]).astype(np.uint32)


def unpack(words):
    w = np.asarray(words, np.uint32).astype(np.int64)
    return np.stack([(w >> 16) & 0xFF, (w >> 8) & 0xFF, w & 0xFF], axis=-1)


def _finish(rng, words, dup, alpha):
    words = np.asarray(words, np.uint32)[rng.permutation(len(words))]
    if dup > 0 and words.size > 1:
        pick = np.flatnonzero(rng.random(words.size) < dup)
        words[pick] = words[rng.integers(0, words.size, pick.size)]
    if alpha:
        words = words | (rng.integers(0, 256, words.size).astype(np.uint32) << 24)
    return np.ascontiguousarray(words, np.uint32)


def _lattice_ball(rng, k, step):
    """k lattice points nearest a random centre (random order among equals); repeats once the lattice is used up."""
    lv = np.arange(0, 256, step)
    pts = np.stack(np.meshgrid(lv, lv, lv, indexing="ij"), -1).reshape(-1, 3)
    centre = rng.integers(0, 256, 3)
    order = np.argsort(((pts - centre) ** 2).sum(1) + rng.random(len(pts)))
    take = pts[order[:min(k, len(pts))]]
    if k > len(pts):
        take = np.concatenate([take, pts[rng.integers(0, len(pts), k - len(pts))]])
    return take


def lattice_palette(rng, k, step=32, dup=0.0, alpha=False):
    return _finish(rng, pack(_lattice_ball(rng, k, step)), dup, alpha)


def midpoint_pixels(rng, pal, n, step=32, alpha=True):
    """Pixels half a step off the palette's own colours, in each channel independently (or on it)."""
    base = unpack(pal)[rng.integers(0, len(pal), n)]
    half = step // 2
    off = rng.choice(np.array([-half, 0, half]), size=(n, 3), p=[0.4, 0.2, 0.4])
    px = pack(np.clip(base + off, 0, 255))
    if alpha:
        px |= rng.integers(0, 256, n).astype(np.uint32) << 24
    return np.ascontiguousarray(px, np.uint32)


def star_palette(rng, k, pad_step=32, dup=0.0, alpha=False):
    """Returns (palette, centres): up to 30 entries on the shell |v|^2 = 9 t^2 around each centre, the whole palette up
    to 60 entries, half of it (at most 64 stars) above; the rest lattice entries."""
    in_stars = k if k <= 60 else min(k // 2, 64 * len(_SHELL))
    stars = -(-in_stars // len(_SHELL))
    entries, centres = [], []
    for i in range(stars):
        t = int(rng.choice([2, 3, 4, 6, 8]))
        c = rng.integers(3 * t, 256 - 3 * t, 3)
        take = in_stars * (i + 1) // stars - in_stars * i // stars
        entries.append(c + t * _SHELL[rng.permutation(len(_SHELL))[:take]])
        centres.append(c)
    if k > in_stars:
        entries.append(_lattice_ball(rng, k - in_stars, pad_step))
    return _finish(rng, pack(np.concatenate(entries)), dup, alpha), pack(np.array(centres))


def star_pixels(rng, centres, n, alpha=True):
    px = centres[rng.integers(0, len(centres), n)].copy()
    if alpha:
        px |= rng.integers(0, 256, n).astype(np.uint32) << 24
    return np.ascontiguousarray(px, np.uint32)


def grey_palette(rng, k, dup=0.0, alpha=False):
    """Entries (g+d, g-d, g) in all six orders for a few d per grey level g: equal sums everywhere, no grey itself."""
    entries = []
    while sum(len(e) for e in entries) < k:
        g = int(rng.integers(8, 248))
        for d in rng.choice(np.arange(1, 8), size=2, replace=False):
            v = np.array([[g + d, g - d, g], [g + d, g, g - d], [g, g + d, g - d],
                          [g - d, g + d, g], [g - d, g, g + d], [g, g - d, g + d]])
            entries.append(v)
    return _finish(rng, pack(np.concatenate(entries)[:k]), dup, alpha)


def grey_pixels(rng, pal, n, alpha=True):
    """Greys at the palette's levels, some one step off in a channel."""
    g = unpack(pal).sum(1)[rng.integers(0, len(pal), n)] // 3
    px = np.stack([g, g, g], -1) + rng.choice(np.array([-1, 0, 0, 0, 1]), size=(n, 3))
    px = pack(np.clip(px, 0, 255))
    if alpha:
        px |= rng.integers(0, 256, n).astype(np.uint32) << 24
    return np.ascontiguousarray(px, np.uint32)


def generate(kind, k, n, seed, dup=0.0, alpha=False, step=None):
    """(pixels, palette) of one of the kinds above: "lattice", "star" or "grey"."""
    rng = np.random.default_rng(seed)
    if kind == "lattice":
        step = step or (32 if k <= 512 else 16 if k <= 4096 else 8)
        pal = lattice_palette(rng, k, step, dup, alpha)
        return midpoint_pixels(rng, pal, n, step), pal
    if kind == "star":
        pal, centres = star_palette(rng, k, dup=dup, alpha=alpha)
        return star_pixels(rng, centres, n), pal
    if kind == "grey":
        pal = grey_palette(rng, k, dup, alpha)
        return grey_pixels(rng, pal, n), pal
    raise ValueError(kind)


def lattice_image(seed, step, colours, repeats):
    """`colours` distinct points of the lattice with levels every `step`, each repeated `repeats` times, shuffled: the
    quantizer's cluster means of such an image fall on ties with the lattice points (quant_recurse's remap)."""
    rng = np.random.default_rng(seed)
    lv = np.arange(0, 256, step)
    idx = rng.choice(lv.size ** 3, colours, replace=False)
    pts = pack(np.stack(np.unravel_index(idx, (lv.size,) * 3), -1) * step)
    return np.ascontiguousarray(np.tile(pts, repeats)[rng.permutation(colours * repeats)], np.uint32)


# quant_recurse inputs: (K, seed, step, colours, repeats, share of pixels on a tie of the oracle's palette, at least).
# The first four have 2U <= n, so the palette reaches the remap through the unique-colour table; the last has 2U > n.
QUANT_CASES = (
    (200, 1, 16, 4096, 2, 0.15),     # K <= 256: tables in the kernel's parameter block
    (400, 2, 16, 4096, 2, 0.15),     # 257..512: integer arg-min, uploaded tables
    (1000, 3, 8, 32768, 2, 0.01),    # > 512: float arg-min in shared memory
    (12000, 4, 4, 40000, 3, 0.005),  # > 11 466: palette in global memory
    (300, 5, 16, 4096, 1, 0.15),     # 2U > n: brute force
)


def _chunks(px, pal, oracle, budget=1 << 22):
    """Yields (slice, dist, rank, sorted words, start index) per chunk of pixels: int64 (rows, K) blocks."""
    srt, lut = oracle.build_search_tables(pal)
    e = unpack(srt)
    p = unpack(np.asarray(px, np.uint32) & 0xFFFFFF)
    k = len(srt)
    idx = np.arange(k)
    rows = max(1, budget // k)
    for a in range(0, len(p), rows):
        q = p[a:a + rows]
        d = ((q[:, None, :] - e[None, :, :]) ** 2).sum(-1)
        s = lut[q.sum(1)].astype(np.int64)[:, None]
        rank = np.where(idx > s, 2 * (idx - s) - 1, 2 * (s - idx))
        yield slice(a, a + len(q)), d, rank, srt, s[:, 0]


def nearest_dist_rank(px, pal, oracle):
    """The remap by its definition: argmin over (dist, rank) of the sorted palette, for every pixel."""
    out = np.empty(len(px), np.uint32)
    for sl, d, rank, srt, _ in _chunks(px, pal, oracle):
        out[sl] = srt[np.argmin((d << 32) | rank, axis=1)]
    return out


def tie_classes(px, pal, oracle):
    """Counts of pixels whose minimal distance is reached by at least two distinct palette words ("multi"), split by
    where the start index s lies against the first (ka) and last (kb) sorted entry at that distance: "inside"
    (ka < s <= kb, the start lies in the run: both walking directions matter), "below" (s <= ka), "above" (s > kb)."""
    c = {"multi": 0, "inside": 0, "below": 0, "above": 0}
    for _, d, _, srt, s in _chunks(px, pal, oracle):
        at = d == d.min(1, keepdims=True)
        w = srt.astype(np.int64)[None, :]
        multi = np.where(at, w, -1).max(1) != np.where(at, w, 1 << 40).min(1)
        ka = np.argmax(at, axis=1)
        kb = at.shape[1] - 1 - np.argmax(at[:, ::-1], axis=1)
        c["multi"] += int(multi.sum())
        c["inside"] += int((multi & (ka < s) & (s <= kb)).sum())
        c["below"] += int((multi & (s <= ka)).sum())
        c["above"] += int((multi & (s > kb)).sum())
    return c
