"""The stream-K work-unit schedule of the CTA-pair GEMM (csrc/gemm.cu: UnitWalk + the sk_lo choice in launch_gemm<2, BN>), mirrored
in Python and checked as a property over many shapes: every (tile, K block) is covered exactly once, by contiguous pieces,
bias goes to exactly one unit per tile, and no cluster does more than its fair share + one tile boundary.  The numerical
check of the kernel itself is tests/test_gemm_gpu.py::test_gemm_stream_k_residual."""
import random

SK_MIN_KBLOCKS, SK_MIN_PIECE = 32, 8   # GEMM_SK_MIN_KBLOCKS, GEMM_SK_MIN_PIECE


def launch_params(tiles: int, kblocks: int, max_clusters: int = 74, reduce_add: bool = True):
    """-> (clusters, sk_lo) as launch_gemm<2, BN> chooses them."""
    clusters = min(tiles, max_clusters)
    sk_lo = tiles
    if reduce_add and kblocks >= SK_MIN_KBLOCKS and tiles % max_clusters != 0:
        tail = tiles % max_clusters
        if (tail * kblocks + max_clusters - 1) // max_clusters >= SK_MIN_PIECE:
            sk_lo, clusters = tiles - tail, max_clusters
    return clusters, sk_lo


def unit_walk(cluster: int, W: int, total_tiles: int, sk_lo: int, kblocks: int):
    """The units (tile, k0, k1) cluster `cluster` of W processes, in order (UnitWalk::next)."""
    units = []
    t = cluster
    while t < sk_lo:
        units.append((t, 0, kblocks))
        t += W
    total = (total_tiles - sk_lo) * kblocks
    piece = (total + W - 1) // W
    pos = cluster * piece
    end = min(pos + piece, total)
    while pos < end:
        j = pos // kblocks
        k0 = pos - j * kblocks
        k1 = min(kblocks, k0 + (end - pos))
        units.append((sk_lo + j, k0, k1))
        pos += k1 - k0
    return units


def check(tiles, kblocks, max_clusters=74, reduce_add=True):
    W, sk_lo = launch_params(tiles, kblocks, max_clusters, reduce_add)
    cover = {}
    per_cluster = []
    for c in range(W):
        units = unit_walk(c, W, tiles, sk_lo, kblocks)
        per_cluster.append(sum(k1 - k0 for _, k0, k1 in units))
        for tile, k0, k1 in units:
            assert 0 <= tile < tiles and 0 <= k0 < k1 <= kblocks
            for k in range(k0, k1):
                assert (tile, k) not in cover, f"K block {(tile, k)} done twice (tiles={tiles}, kblocks={kblocks})"
                cover[(tile, k)] = c
    assert len(cover) == tiles * kblocks, f"{tiles * kblocks - len(cover)} K blocks never done (tiles={tiles}, kblocks={kblocks})"
    # bias: exactly one unit per tile starts at K block 0
    starts = sum(1 for c in range(W) for tile, k0, _ in unit_walk(c, W, tiles, sk_lo, kblocks) if k0 == 0)
    assert starts == tiles
    if sk_lo < tiles:   # balance: whole tiles before sk_lo are dealt round-robin, the tail is cut into equal pieces
        assert max(per_cluster) - min(per_cluster) <= (tiles - sk_lo) * kblocks // W + kblocks
    return W, sk_lo, max(per_cluster)


def test_the_shapes_of_the_model():
    # encoder fc2 (10960 x 1024 x 4096): 43 x 4 tiles, 64 K blocks -> 2 waves + 24 tiles, 149 instead of 192 K blocks per pair
    W, sk_lo, worst = check(172, 64)
    assert (W, sk_lo) == (74, 148) and worst == 2 * 64 + 21
    # info-sharing fc2 (10953 x 768 x 3072): 43 x 3 tiles, 48 K blocks -> 1 wave + 55 tiles
    W, sk_lo, worst = check(129, 48)
    assert (W, sk_lo) == (74, 74) and worst == 48 + 36
    # 2 views (2740 rows): fewer tiles than CTA pairs -> everything is cut
    W, sk_lo, worst = check(44, 64)
    assert (W, sk_lo) == (74, 0) and worst == 39
    # attention projection (K = 1024): too few K blocks, whole tiles only
    assert launch_params(172, 16) == (74, 172)
    # not a reduce-add epilogue: whole tiles only
    assert launch_params(172, 64, reduce_add=False) == (74, 172)
    # full waves: nothing to cut
    assert launch_params(148, 64) == (74, 148)


def test_every_k_block_exactly_once_over_random_shapes():
    rng = random.Random(0)
    for _ in range(400):
        tiles = rng.randint(1, 700)
        kblocks = rng.choice([1, 2, 12, 16, 31, 32, 33, 48, 64, 65, 100, 128])
        clusters = rng.choice([1, 2, 7, 64, 66, 74])
        check(tiles, kblocks, clusters)
    for tiles in range(1, 160):   # every tail length around the real machine size
        check(tiles, 64)
        check(tiles, 33)
