"""The statistics kernels of swtpg_stats.cu at the work-item geometries production runs, every link against exact integer sums.

launch_channel_stats (ADC statistics and noise lags) and launch_products (channel products) cut each link's units into `parts`
work items of `chunk` units, from the SM count, the link count and units_stride. The other statistics tests run small handles,
where an item holds at most a few units; the bench and the probes run items of 32 to 64 units. What only such items do (sums
past an item's first units, the lags of many WIB2 segments summed in one item, the third and later slabs of a product CTA) is
tested here. The split rules are restated below; test_restated_split_rules_match_the_source pins them to the source, and
test_cases_reach_every_regime checks that the cases take every regime, at 148 SMs and on the GPU at hand.

Each case runs one handle with all three flags over two batches generated on the device, a ragged one and a full one. The
references are computed on the host from a copy of those frames:
- every link: the ADC statistics exactly; the channel products by integer Freivalds projections, P v == X^T (X v) in int64 for
  four seeded vectors v, with samples, channel sums and the diagonal of P equal to the statistics; lag[0] equal to the sum of
  squares over the link's whole segments, and the segments counted;
- a seeded sample of links (the first and last, the rails, one link of each ragged count): every product word and every lag."""
import os
import re
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import frames as F
from util import adc_of, channels, combine, lags_of, ragged_units, sms, stats_of, ticks_per_unit, unit_bytes, words_of

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "fdreadoutlibs_b200", "csrc")


# ---- the split rules, restated ----------------------------------------------------------------------------------------------
# swtpg_stats.cu: launch_channel_stats and launch_products with their constants. Every item covers units
# [part * chunk, min(n_units, part * chunk + chunk)) of its link.
STATS_WARPS = 4          # kStatsWarps: one item per warp, 4 warps per CTA
STATS_MAX_UNITS = 64     # kStatsMaxUnits
STATS_ITEMS_PER_SM = 48  # kStatsItemsPerSm
PROD_MIN_UNITS = 16      # kProdMinUnits
PROD_MAX_UNITS = 64      # kProdMaxUnits
PROD_ITEMS_PER_SM = 8    # kProdItemsPerSm
SEGMENT_UNITS = {"wibeth": 1, "wib2": 4}  # Segment<WIB2>::kUnits: units per noise segment
SLAB_UNITS = {"wibeth": 1, "wib2": 8}     # ProductSlab<WIB2>::kUnits: units staged at once by a product CTA
GROUPS = {"wibeth": 1, "wib2": 4}         # 64-channel groups of a link (groups_per_link)


def cdiv(a, b):
    return -(-a // b)


def stats_geometry(fmt, n_links, stride, sms, spectra):
    """(parts, chunk) of launch_channel_stats; spectra: SWTPG_FLAG_NOISE_SPECTRA is set."""
    n = n_links * GROUPS[fmt]
    parts = max(1, min(max(cdiv(sms * STATS_ITEMS_PER_SM, n), cdiv(stride, STATS_MAX_UNITS)), stride))
    chunk = cdiv(stride, parts)
    if fmt == "wib2" and spectra:
        chunk = cdiv(chunk, SEGMENT_UNITS["wib2"]) * SEGMENT_UNITS["wib2"]
    return cdiv(stride, chunk), chunk


def products_geometry(fmt, n_links, stride, sms):
    """(parts, chunk) of launch_products."""
    n = n_links * GROUPS[fmt] * (GROUPS[fmt] + 1) // 2  # 64 x 64 block pairs
    parts = max(1, min(max(cdiv(sms * PROD_ITEMS_PER_SM, n), cdiv(stride, PROD_MAX_UNITS)), stride))
    slab = SLAB_UNITS[fmt]
    chunk = min(PROD_MAX_UNITS, cdiv(max(cdiv(stride, parts), PROD_MIN_UNITS), slab) * slab)
    return cdiv(stride, chunk), chunk


def pinned(src, line, count=1):
    """Asserts that the source holds `line` (any whitespace between its tokens) `count` times."""
    pattern = r"\s*".join(re.escape(tok) for tok in line.split())
    m = re.findall(pattern, src)
    assert len(m) == count, f"{line!r}: {len(m)} matches, expected {count}"


def body(src, head):
    """The text of the function that starts at `head`, up to its closing brace in column 0."""
    i = src.index(head)
    return src[i:src.index("\n}\n", i)]


def test_restated_split_rules_match_the_source():
    with open(os.path.join(CSRC, "swtpg_stats.cu")) as f:
        src = f.read()
    with open(os.path.join(CSRC, "swtpg_capi.cu")) as f:
        capi = f.read()
    for name, value in (("kStatsWarps", STATS_WARPS), ("kStatsMaxUnits", STATS_MAX_UNITS), ("kStatsItemsPerSm", STATS_ITEMS_PER_SM),
                        ("kProdMinUnits", PROD_MIN_UNITS), ("kProdMaxUnits", PROD_MAX_UNITS), ("kProdItemsPerSm", PROD_ITEMS_PER_SM)):
        pinned(src, f"constexpr uint32_t {name} = {value};")
    pinned(src, "static constexpr uint32_t kUnits = WIB2 ? SWTPG_WIB2_NOISE_SEGMENT_TICKS / SWTPG_WIB2_TICKS : 1;")
    assert F.NOISE_SEGMENT_TICKS["wib2"] // F.WIB2_SUPERCHUNK_FRAMES == SEGMENT_UNITS["wib2"]
    assert F.NOISE_SEGMENT_TICKS["wibeth"] == F.WIBETH_TICKS
    pinned(src, f"static constexpr uint32_t kUnits = WIB2 ? {SLAB_UNITS['wib2']} : {SLAB_UNITS['wibeth']};")
    pinned(capi, "h->groups_per_link = h->channels / 64;")
    # the items of both kernels
    pinned(src, "const uint32_t u0 = part * chunk;", 2)
    pinned(src, "const uint32_t u1 = min(units, u0 + chunk);", 2)
    stats = body(src, "swtpg_internal::launch_channel_stats(")
    for line in ("const uint32_t n = h->cfg.n_links * h->groups_per_link;",
                 "const uint32_t want = (uint32_t(sm_count[dev]) * kStatsItemsPerSm + n - 1) / n;",
                 "uint32_t parts = std::max(want, (units_stride + kStatsMaxUnits - 1) / kStatsMaxUnits);",
                 "parts = std::max(1u, std::min(parts, units_stride));",
                 "uint32_t chunk = (units_stride + parts - 1) / parts;",
                 "if (wib2 && h->d_noise_lags)",
                 "chunk = (chunk + Segment<true>::kUnits - 1) / Segment<true>::kUnits * Segment<true>::kUnits;",
                 "parts = (units_stride + chunk - 1) / chunk;",
                 "const unsigned grid = unsigned((items + kStatsWarps - 1) / kStatsWarps);"):
        pinned(stats, line)
    products = body(src, "launch_products(int sms,")
    for line in ("const uint32_t n = h->cfg.n_links * (kGroups * (kGroups + 1) / 2);",
                 "const uint32_t want = (uint32_t(sms) * kProdItemsPerSm + n - 1) / n;",
                 "uint32_t parts = std::max(want, (units_stride + kProdMaxUnits - 1) / kProdMaxUnits);",
                 "parts = std::max(1u, std::min(parts, units_stride));",
                 "uint32_t chunk = std::max((units_stride + parts - 1) / parts, kProdMinUnits);",
                 "chunk = std::min(kProdMaxUnits, (chunk + ProductSlab<WIB2>::kUnits - 1) / ProductSlab<WIB2>::kUnits * ProductSlab<WIB2>::kUnits);",
                 "parts = (units_stride + chunk - 1) / chunk;"):
        pinned(products, line)
    pinned(stats, "launch_products<true>(sm_count[dev],")  # the same SM count as the statistics
    pinned(stats, "launch_products<false>(sm_count[dev],")


# ---- the cases --------------------------------------------------------------------------------------------------------------
# name: (format, links as a function of the SM count, units_stride, noise spectra on). All three run the ADC statistics and the
# channel products as well. (parts, chunk) of the statistics and of the products, and the frames of one batch, at 148 SMs:
CASES = {
    "wibeth_40_per_sm_x64": ("wibeth", lambda s: 40 * s, 64, True),         # 5920 links, the bench workload: (2, 32), (1, 64); 2.7 GB
    "wib2_10_per_sm_x64": ("wib2", lambda s: 10 * s, 64, True),             # 1480: (2, 32), 8 segments an item; (1, 64); 0.54 GB
    "wib2_12_per_sm_x64": ("wib2", lambda s: 12 * s, 64, True),             # 1776, 48 statistics items per SM: (1, 64); (1, 64); 0.64 GB
    "wibeth_12_per_sm_x160": ("wibeth", lambda s: 12 * s, 160, True),       # 1776: (4, 40); (3, 54), the last of 52; 2.0 GB
    "wib2_6_per_sm_x130": ("wib2", lambda s: 6 * s, 130, True),             # 888: (3, 44) as 130 / 64 asks, the last of 42; (3, 48); 0.65 GB
    "wib2_400_x100": ("wib2", lambda s: 400, 100, True),                    # (5, 20); (2, 56), the last of 44; 0.23 GB
    "wib2_2_per_5_sm_x64": ("wib2", lambda s: cdiv(2 * s, 5), 64, True),    # 60: (16, 4), one segment an item; (2, 32)
    "wib2_stats_only_1_per_sm_x64": ("wib2", lambda s: s, 64, False),       # 148: (11, 6), no spectra; (1, 64)
}

REGIMES = (
    "statistics: one item of 64 units a link",
    "statistics: units_stride > 64 sets parts > 1, the last item shorter",
    "WIB2 spectra: 2 or more segments an item",
    "WIB2 statistics only: items of more than 1 unit, not whole segments",
    "WIBEth spectra: 32 or more frames an item",
    "products: items of 32 units",
    "products: one item of 64 units a link",
    "products: units_stride > 64 in 2-4 items, the last shorter",
)


def regimes(fmt, n_links, stride, spectra, sms):
    """The REGIMES a handle's launches take."""
    out = set()
    parts, chunk = stats_geometry(fmt, n_links, stride, sms, spectra)
    if (parts, chunk) == (1, 64):
        out.add(REGIMES[0])
    if stride > 64 and cdiv(stride, STATS_MAX_UNITS) > cdiv(sms * STATS_ITEMS_PER_SM, n_links * GROUPS[fmt]) and stride % chunk:
        out.add(REGIMES[1])
    if fmt == "wib2" and spectra and chunk // SEGMENT_UNITS["wib2"] >= 2:
        out.add(REGIMES[2])
    if fmt == "wib2" and not spectra and chunk > 1 and chunk % SEGMENT_UNITS["wib2"]:
        out.add(REGIMES[3])
    if fmt == "wibeth" and spectra and chunk >= 32:
        out.add(REGIMES[4])
    parts, chunk = products_geometry(fmt, n_links, stride, sms)
    if chunk == 32:
        out.add(REGIMES[5])
    if (parts, chunk) == (1, 64):
        out.add(REGIMES[6])
    if stride > 64 and 2 <= parts <= 4 and stride % chunk:
        out.add(REGIMES[7])
    return out


def test_cases_reach_every_regime():
    """At 148 SMs (a B200) and at the SM count of the GPU here, if there is one, the cases take every regime between them."""
    counts = [148]
    try:
        import torch

        if torch.cuda.is_available():
            counts.append(sms())
    except ImportError:
        pass
    for s in counts:
        got = set()
        for fmt, links, stride, spectra in CASES.values():
            got |= regimes(fmt, links(s), stride, spectra, s)
        assert got == set(REGIMES), f"{s} SMs: no case takes {sorted(set(REGIMES) - got)}"
    # the restatement against the table above
    assert [stats_geometry(f, l(148), st, 148, sp) for f, l, st, sp in CASES.values()] == [
        (2, 32), (2, 32), (1, 64), (4, 40), (3, 44), (5, 20), (16, 4), (11, 6)]
    assert [products_geometry(f, l(148), st, 148) for f, l, st, _ in CASES.values()] == [
        (1, 64), (1, 64), (1, 64), (3, 54), (3, 48), (2, 56), (2, 32), (1, 64)]


def ragged_counts(fmt, stride, stats_geo, products_geo):
    """Unit counts that put a link's end at every kind of place in its items: 0, 1, a chunk -1 / 0 / +1, two chunks +-1,
    units_stride - 1 and units_stride, for both geometries. WIB2 with spectra adds counts of 1, 2 and 3 modulo a segment on both
    sides of the edges after the first, a middle and the last-but-one item, so that the superchunks left out of a segment
    fall in a first, a middle and a last item."""
    out = {0, 1, stride - 1, stride}
    for _, chunk in (stats_geo, products_geo):
        out |= {chunk - 1, chunk, chunk + 1, 2 * chunk - 1, 2 * chunk + 1}
    parts, chunk = stats_geo
    if fmt == "wib2" and chunk % SEGMENT_UNITS["wib2"] == 0:
        out |= {1, 2, 3}
        for edge in {chunk, parts // 2 * chunk, (parts - 1) * chunk}:
            out |= {edge + d for d in (-3, -2, -1, 1, 2, 3)}
    return sorted(u for u in out if 0 <= u <= stride)


# ---- the host reference -----------------------------------------------------------------------------------------------------
_SHIFTS = np.array([0, 14, 28, 42], dtype=np.uint64)


def adc_rows(fmt, units):
    """(samples, channels) raw ADC values of a link's units, as adc_of returns them: every 7 bytes of a row are 4 packed 14-bit
    values, read as one little-endian word (numpy's bit unpacking, which adc_of uses, is too slow for every link of these
    batches; test_adc_rows_equals_adc_of ties the two)."""
    if fmt == "wib2":
        rows = units.reshape(-1, F.WIB2_FRAME_BYTES)[:, F.WIB2_ADC_OFFSET:F.WIB2_ADC_OFFSET + F.WIB2_CHANNELS * 14 // 8]
    else:
        rows = units.reshape(-1, F.WIBETH_FRAME_BYTES)[:, F.WIBETH_HEADER_BYTES:]
    words = np.zeros((rows.shape[0], rows.shape[1] // 7, 8), dtype=np.uint8)
    words[..., :7] = rows.reshape(words.shape[:2] + (7,))
    return ((words.view("<u8") >> _SHIFTS) & np.uint64(0x3FFF)).astype(np.uint16).reshape(-1, channels(fmt))


@pytest.mark.parametrize("fmt", ["wibeth", "wib2"])
def test_adc_rows_equals_adc_of(fmt):
    rng = np.random.default_rng(len(fmt))
    units = rng.integers(0, 256, (5, unit_bytes(fmt)), dtype=np.uint8)
    units[1] = 0xFF
    units[2] = 0
    assert (adc_rows(fmt, units) == adc_of(fmt, units)).all()
    assert adc_rows(fmt, units[:0]).shape == (0, channels(fmt))
    gen = S.gen_wib2_host if fmt == "wib2" else S.gen_wibeth_host
    units = gen(S.gen_params(3, 0.3), 1, 9)[0]
    assert (adc_rows(fmt, units) == adc_of(fmt, units)).all()


class Reference:
    """Host sums of a handle's batches, link by link (a thread pool over links: the products release the GIL)."""

    def __init__(self, fmt, n_links, v, sample):
        c = channels(fmt)
        self.fmt, self.v, self.sample = fmt, v, sample
        self.stats = np.zeros((n_links, c), dtype=F.ADC_STATS_DTYPE)
        self.proj = np.zeros((n_links, c, v.shape[1]), dtype=np.int64)  # X^T (X v)
        self.seg_sq = np.zeros((n_links, c), dtype=np.int64)            # squares summed over whole segments
        self.segments = np.zeros(n_links, dtype=np.int64)
        self.words = {l: np.zeros(F.channel_products_words(fmt), dtype=np.uint64) for l in sample}
        self.lags = {l: np.zeros(c, dtype=F.NOISE_LAGS_DTYPE) for l in sample}

    def add(self, frames, nu):
        """frames [n_links, stride, unit bytes] of one batch, nu its valid units per link (None: all)."""
        fmt, stride = self.fmt, frames.shape[1]

        def one(l):
            n = stride if nu is None else int(nu[l])
            a = adc_rows(fmt, frames[l, :n])
            self.stats[l] = combine(self.stats[l], stats_of(a))
            x = a.astype(np.int64)
            self.proj[l] += np.ascontiguousarray(x.T) @ (x @ self.v)
            segs = n // SEGMENT_UNITS[fmt]
            xs = x[: segs * SEGMENT_UNITS[fmt] * ticks_per_unit(fmt)]
            self.seg_sq[l] += (xs * xs).sum(axis=0)
            self.segments[l] += segs
            if l in self.words:
                b = adc_of(fmt, frames[l, :n])
                assert (b == a).all(), f"link {l}: adc_rows differs from adc_of"
                self.words[l] += words_of(fmt, b)
                lags = lags_of(fmt, b)
                self.lags[l]["segments"] += lags["segments"]
                self.lags[l]["lag"] += lags["lag"]

        with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
            list(ex.map(one, range(frames.shape[0])))


def first_bad(what, bad, got, want):
    """Fails with the count and the first (link, ...) index where `bad` is set."""
    idx = np.argwhere(bad)
    if idx.size:
        i = tuple(int(x) for x in idx[0])
        pytest.fail(f"{what}: {len(idx)} differ, on {len(np.unique(idx[:, 0]))} links; first at {i}: got {got[i]}, want {want[i]}")


def mark(fmt, buf, n_links, stride, nu, high, low):
    """On the device: ADC values of links `high` at 16383 and of links `low` at 0, every byte past a link's n_units 0xFF."""
    import torch

    v = buf.view(n_links, stride, unit_bytes(fmt))
    if fmt == "wib2":
        adc = v.view(n_links, stride * F.WIB2_SUPERCHUNK_FRAMES, F.WIB2_FRAME_BYTES)[..., F.WIB2_ADC_OFFSET:F.WIB2_ADC_OFFSET + 448]
    else:
        adc = v[..., F.WIBETH_HEADER_BYTES:]
    adc[torch.as_tensor(high, device="cuda")] = 0xFF
    adc[torch.as_tensor(low, device="cuda")] = 0
    if nu is not None:
        past = torch.arange(stride, device="cuda")[None, :] >= torch.as_tensor(nu.astype(np.int64), device="cuda")[:, None]
        v[past] = 0xFF


def assert_matches(case, stats, lags, words, ref):
    """The device's statistics, lags (None: not on) and products of every link against the host Reference."""
    fmt, v, sample = ref.fmt, ref.v, ref.sample
    n, c = stats.shape
    for f in ("samples", "sum", "sum_sq", "min", "max"):
        first_bad(f"{case}: ADC statistics, {f}", stats[f] != ref.stats[f], stats[f], ref.stats[f])
    assert not stats["reserved"].any()

    def products(l):  # (samples, sums, diagonal, P v) of one link's device words
        samples, sums, p = F.unpack_channel_products(words[l], fmt)
        return samples, sums, np.diag(p).copy(), p.astype(np.int64) @ v

    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        got = list(ex.map(products, range(n)))
    samples = np.array([g[0] for g in got], dtype=np.uint64)
    sums, diag, proj = (np.stack([g[i] for g in got]) for i in (1, 2, 3))
    first_bad(f"{case}: products, samples", samples != stats["samples"][:, 0], samples, stats["samples"][:, 0])
    first_bad(f"{case}: products, channel sums", sums != stats["sum"], sums, stats["sum"])
    first_bad(f"{case}: products, diagonal", diag != stats["sum_sq"], diag, stats["sum_sq"])
    first_bad(f"{case}: products, P v", proj != ref.proj, proj, ref.proj)
    for l in sorted(sample):
        first_bad(f"{case}: products of link {l}", (words[l] != ref.words[l])[None], words[l][None], ref.words[l][None])

    if lags is not None:
        segs = np.broadcast_to(ref.segments[:, None], (n, c)).astype(np.uint64)
        first_bad(f"{case}: lags, segments", lags["segments"] != segs, lags["segments"], segs)
        first_bad(f"{case}: lags, lag[0]", lags["lag"][..., 0] != ref.seg_sq, lags["lag"][..., 0], ref.seg_sq)
        if fmt == "wibeth":
            assert (lags["lag"][..., 0] == stats["sum_sq"]).all() and (lags["segments"] * 64 == stats["samples"]).all()
        else:
            assert not lags["lag"][..., F.NOISE_SEGMENT_TICKS["wib2"] // 2 + 1:].any()
        for l in sorted(sample):
            for f in ("segments", "lag"):
                first_bad(f"{case}: lags of link {l}, {f}", (lags[f][l] != ref.lags[l][f])[None], lags[f][l][None], ref.lags[l][f][None])


# ---- the GPU runs -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_statistics_at_production_geometry(case):
    import torch

    fmt, links, stride, spectra = CASES[case]
    s = sms()
    n = links(s)
    c, tpu = channels(fmt), ticks_per_unit(fmt)
    sgeo, pgeo = stats_geometry(fmt, n, stride, s, spectra), products_geometry(fmt, n, stride, s)
    seed = 900 + list(CASES).index(case)
    rng = np.random.default_rng(seed)
    v = rng.integers(0, 1 << 10, (c, 4))
    # the largest term of X^T (X v) over both batches: ticks x 16383 x (channels x 16383 x 1023)
    assert 2 * stride * tpu * 16383 * c * 16383 * 1023 < 2 ** 63
    counts = ragged_counts(fmt, stride, sgeo, pgeo)
    nus = [ragged_units(seed, n, stride, counts), None]
    rails = rng.choice(n, 6, replace=False)
    high, low = rails[:3], rails[3:]
    sample = {0, n - 1, *(int(l) for l in rails)}
    for u in counts:  # one link of each ragged count
        at = np.nonzero(nus[0] == u)[0]
        assert at.size, f"no link of {u} units"
        sample.add(int(at[0]))
    sample |= {int(l) for l in rng.permutation(n)[: max(0, 64 - len(sample))]}
    ref = Reference(fmt, n, v, sample)

    gen = S.gen_wib2_device if fmt == "wib2" else S.gen_wibeth_device
    buf = torch.empty(n * stride * unit_bytes(fmt), dtype=torch.uint8, device="cuda")
    try:
        with S.TPGenerator(n, stride, fmt=fmt, tp_capacity=1 << 24, adc_stats=True, noise_spectra=spectra, channel_covariance=True) as g:
            g.start()
            for k, nu in enumerate(nus):
                gen(S.gen_params(seed, 0.05), buf.data_ptr(), n, stride, unit0=k * stride)
                mark(fmt, buf, n, stride, nu, high, low)
                torch.cuda.synchronize()  # the generator and torch run on the legacy stream, the handle on its own
                g.process_device(buf.data_ptr(), stride, n_units=nu)
                g.fetch_count()
                g.sync()  # the statistics kernels too: the buffer is free to be read and rewritten
                ref.add(buf.view(n, stride, unit_bytes(fmt)).cpu().numpy(), nu)
            stats = g.read_adc_stats()
            lags = g.read_noise_lags() if spectra else None
            words = g.read_channel_products()
    finally:
        del buf
        torch.cuda.empty_cache()

    assert (nus[0] == 0).any() and (nus[0] == stride).any()
    assert (ref.stats["min"][high] == 16383).all() and (ref.stats["max"][low] == 0).all()
    assert_matches(case, stats, lags, words, ref)
