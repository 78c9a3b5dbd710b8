"""The contiguous-input histogram of inputs with a 32 768-pixel chunk per SM or more (hist_insert_chunked_kernel,
csrc/dq_hist_chunk.cuh) counts each CTA's pixel chunk in a shared-memory table before the L2 atomics; smaller inputs take
the per-pixel kernel.  dq_pixel_histogram goes through the same choice, so it must equal np.unique on the 24-bit pixels for
inputs that exercise every branch: coherent frames (most pixels counted in shared memory), uniform random pixels (every
chunk overflows and goes direct), one colour, chunks with the table's fill limit of distinct colours and more, sizes
around the switch between the two kernels and around a chunk, and alpha bytes that differ between pixels of the same
colour."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W4K, H4K = 3840, 2160
CHUNK = 32768         # pixels per chunk
SWITCH = 148 * CHUNK  # smallest input of the chunked kernel on a 148-SM B200
PASS = 4096           # pixels of one CTA pass
SLOTS = 8192          # shared table slots
FILL_MAX = 5120       # distinct colours after which the rest of a chunk is counted directly


def _check(dq, px):
    keys, counts = dq.pixel_histogram(px)
    ek, ec = np.unique(px & 0xFFFFFF, return_counts=True)
    assert keys.size == ek.size, (keys.size, ek.size)
    assert np.array_equal(keys, ek)
    assert np.array_equal(counts, ec)


@pytest.mark.parametrize("kind,w,h", [(1, W4K, H4K), (2, W4K, H4K), (1, 1920, 1080), (2, 1920, 1080)],
                         ids=["g1_4k", "g2_4k", "g1_1080p", "g2_1080p"])
def test_generated_frames(dq, oracle, kind, w, h):
    _check(dq, oracle.generate(kind, w, h, 12345))


def test_one_colour_4k(dq):
    _check(dq, np.full(W4K * H4K, 0xFF123456, np.uint32))


@pytest.mark.parametrize("distinct", [FILL_MAX - 1, FILL_MAX, FILL_MAX + 1, SLOTS - 1, SLOTS, SLOTS + 1, CHUNK])
def test_chunk_at_table_capacity(dq, distinct):
    """Every chunk of a 4K frame holds exactly `distinct` colours (each chunk its own set, shuffled)."""
    rng = np.random.default_rng(distinct)
    n = W4K * H4K
    idx = np.arange(n, dtype=np.int64)
    chunk = idx // CHUNK
    colour = (chunk * 40503 + (idx % CHUNK) % distinct) & 0xFFFFFF
    px = colour.astype(np.uint32) | 0xFF000000
    for c in range(0, n, CHUNK):  # shuffle inside each chunk, so slots fill in an arbitrary order
        seg = px[c:c + CHUNK]
        seg[:] = seg[rng.permutation(seg.size)]
    _check(dq, px)


@pytest.mark.parametrize("n", list(range(1, 8)) + [SWITCH - 1, SWITCH, SWITCH + 1, SWITCH + 3, SWITCH + PASS - 1,
                                                    SWITCH + PASS + 1, SWITCH + CHUNK - 1, SWITCH + CHUNK + 1])
def test_sizes(dq, oracle, n):
    """Tails of fewer than 4 pixels, the switch to the chunked kernel +- 1, and a last chunk of one pixel, one pass +- 1
    and one chunk +- 1."""
    w = 3840
    px = oracle.generate(1, w, -(-n // w), 777)[:n].copy()
    _check(dq, px)


def test_alpha_bytes_differ(dq, oracle):
    rng = np.random.default_rng(5)
    px = oracle.generate(1, W4K, H4K, 12377)
    px = (px & 0xFFFFFF) | (rng.integers(0, 256, px.size, dtype=np.uint32) << 24)
    _check(dq, px)


def test_varpart_fast_cut_bits_on_chunks(dq, oracle):
    """num_bits < 8 masks and shifts inside the chunked kernel: quant_varpart_fast against the oracle on a frame that spans
    many chunks."""
    from oracle import muted
    px = oracle.generate(1, W4K, H4K, 12345)
    for bits in (4, 5):
        with muted():
            ref_vp, ref_empty = oracle.quant_varpart_fast(px, 16, num_bits=bits, rows=1, cols=px.size)
        with muted((2,)):
            vp, empty = dq.quant_varpart_fast(px, 16, num_bits=bits, rows=1, cols=px.size)
        assert np.array_equal(vp, ref_vp) and empty == ref_empty, bits
