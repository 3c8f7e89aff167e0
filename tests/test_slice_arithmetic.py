"""Host-side model of the sliced hand-out's arithmetic (fdreadoutlibs_b200/csrc/swtpg_kernels.cuh, wibeth_kernel: `slice_of`,
`slices_before` and the per-link counter protocol). The kernel relies on four properties, for equal AND halving slices and for
every unit count incl. fewer units than slices: (1) the slices partition [0, n); (2) the LAST slice is never empty when n >= 1
(it is the one that re-arms the link's counter); (3) `slices_before` equals the number of non-empty slices in front of a slice
wherever the kernel uses it (a slice that waits, a slice that publishes); (4) processing the items of a launch in claim order with
any number of persistent warps never dead-locks and leaves every counter at zero. No GPU: this pins the formulas, the CUDA side
is covered by tests/test_gpu_parity.py::test_links_handed_out_in_slices (forced slice counts) and by
tests/test_gpu_launch_geometry.py (the production launch geometries, every link against the oracle)."""
import numpy as np
import pytest


def slice_of(n, part, parts_log2, geom):
    P = 1 << parts_log2
    if geom:
        u0 = n - ((n + (1 << part) - 1) >> part)
        u1 = n if part + 1 == P else n - ((n + (2 << part) - 1) >> (part + 1))
    else:
        u0 = (part * n) >> parts_log2
        u1 = ((part + 1) * n) >> parts_log2
    return u0, u1


def slices_before(n, part, u0, geom):
    if not geom:
        return min(part, u0)
    return min(part, (n - 1).bit_length() if n > 1 else 0)  # 32 - clz(n - 1)


@pytest.mark.parametrize("geom", [0, 1])
@pytest.mark.parametrize("parts_log2", [0, 1, 2, 3])
def test_slices_partition_and_counts(geom, parts_log2):
    P = 1 << parts_log2
    for n in range(0, 300):
        sl = [slice_of(n, p, parts_log2, geom) for p in range(P)]
        assert sl[0][0] == 0 and sl[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(sl, sl[1:])) and all(u0 <= u1 for u0, u1 in sl)
        if n >= 1:
            assert sl[-1][0] < sl[-1][1], "the last slice re-arms the counter: it must run"
        for p, (u0, u1) in enumerate(sl):
            if u0 < u1:  # only slices that run wait or publish
                assert slices_before(n, p, u0, geom) == sum(1 for a, b in sl[:p] if a < b)
        if geom and n >= P:  # halving: each slice at most as long as the one before, the last two equal for powers of two
            sizes = [b - a for a, b in sl]
            assert all(x >= y for x, y in zip(sizes[:-2], sizes[1:-1]))


@pytest.mark.parametrize("geom", [0, 1])
def test_claim_order_never_deadlocks(geom):
    """Items are claimed in increasing order by whichever warp is free; a slice may start only when the link's counter shows all
    non-empty slices in front of it done. With every warp resident, a round-robin of 'advance one warp' must finish."""
    rng = np.random.default_rng(5)
    for trial in range(60):
        parts_log2 = int(rng.integers(1, 4))
        P = 1 << parts_log2
        n_links = int(rng.integers(1, 40))
        warps = int(rng.integers(1, n_links + 1))
        units = rng.integers(0, 20, n_links)
        done = np.zeros(n_links, dtype=int)
        processed = np.zeros(n_links, dtype=int)
        n_items, cursor = n_links * P, warps
        current = list(range(warps))  # warp w starts on item w
        remaining = [None] * warps    # work left in the current item (None = not started)
        active, steps = warps, 0
        while active:
            steps += 1
            assert steps < 200000, "hand-out dead-locked"
            for w in range(warps):
                it = current[w]
                if it is None:
                    continue
                link, part = it % n_links, it // n_links
                u0, u1 = slice_of(int(units[link]), part, parts_log2, geom)
                if remaining[w] is None:
                    if u0 == u1:  # empty slices are skipped by the producer
                        remaining[w] = -1
                    elif part != 0 and u0 != 0 and done[link] != slices_before(int(units[link]), part, u0, geom):
                        continue  # wait_for_slices
                    else:
                        assert processed[link] == u0, "slices of a link run in order and exactly once"
                        remaining[w] = int(rng.integers(1, 4))
                if remaining[w] > 0:
                    remaining[w] -= 1
                    if remaining[w] > 0:
                        continue
                    processed[link] = u1
                    done[link] = 0 if part + 1 == P else slices_before(int(units[link]), part, u0, geom) + 1
                # next item
                remaining[w] = None
                if cursor < n_items:
                    current[w], cursor = cursor, cursor + 1
                else:
                    current[w] = None
                    active -= 1
        assert (processed == units).all() and (done == 0).all()
