"""The dictionary table leaves each record's table slot with a creator bit, and the words are then
numbered by one scan over the records (pfp_phrase.cu: table_insert_k, table_compact_k, uid_words_k).
Each case is compared with the oracle at its extremes: every phrase a different word, one slot
taking nearly every occurrence, a table sized from a misleading previous parse (the rerun path),
and the occurrence counts of the weighted dictionary merge at the 2^32-1 limit."""
import numpy as np
import pytest
import torch

from conftest import assert_same_files
from oracle import pfp_oracle as orc

pytestmark = pytest.mark.gpu


def periodic_one_trigger(pkg, period=150):
    """A block whose repetition has exactly one trigger (w=10, p=100) per period: the parse of
    block * k is one word k-1 times plus the two border phrases."""
    for seed in range(1, 1000):
        b = pkg.synth.random_dna(period, seed).numpy().tobytes()
        t = orc.triggers(b * 6, 10, 100)
        if sum(1 for x in t if 2 * period <= x < 3 * period) == 1:
            return b
    raise AssertionError("no block with one trigger per period")


def test_every_phrase_distinct(pkg):
    text = np.random.default_rng(91).integers(3, 256, 2_000_000, dtype=np.uint8).tobytes()
    want = orc.parse(text, 10, 100)
    occ = np.frombuffer(want.occ, np.uint32)
    assert occ.max() == 1 and occ.size == len(want.parse) // 4 > 10_000
    s = pkg.pfp.Scanner(0)
    try:
        for rep in range(2):                 # fresh context, then a table sized from the first parse
            got = s.parse_host(text, 10, 100)
            assert_same_files(got, want, f"all distinct, parse {rep}")
            assert got.stats["n_distinct"] == occ.size
    finally:
        s.close()


def test_one_word_takes_every_count(pkg):
    block = periodic_one_trigger(pkg)
    text = block * 40_000
    want = orc.parse(text, 10, 100)
    occ = np.frombuffer(want.occ, np.uint32)
    assert occ.size <= 3 and occ.max() >= 39_990
    s = pkg.pfp.Scanner(0)
    try:
        for rep in range(2):
            assert_same_files(s.parse_host(text, 10, 100), want, f"one word, parse {rep}")
        # the same through the device entry and with the verify pass
        dev = torch.from_numpy(np.frombuffer(text, np.uint8).copy()).cuda()
        assert_same_files(s.fetch(s.parse_device(dev, 10, 100, verify=True)), want, "one word, verify")
    finally:
        s.close()


def test_repetitive_then_random_reruns_with_safe_table(pkg):
    """The first parse leaves a distinct/phrase ratio near 0 on the context; the random text after
    it overflows the table sized from that ratio (or crosses 0.85 of it) and the stage reruns."""
    block = periodic_one_trigger(pkg)
    rep = block * 20_000
    rnd = pkg.synth.random_dna(3_000_000, 92).numpy().tobytes()
    s = pkg.pfp.Scanner(0)
    try:
        got = s.parse_host(rep, 10, 100)
        assert got.stats["n_distinct"] <= 3
        want = orc.parse(rnd, 10, 100)
        got = s.parse_host(rnd, 10, 100)
        assert_same_files(got, want, "random after one-word text")
        assert got.stats["n_distinct"] == len(want.occ) // 4
        assert_same_files(s.parse_host(rep, 10, 100), orc.parse(rep, 10, 100), "one-word text again")
    finally:
        s.close()


def shard_words_of(pkg, text, w=10, p=100):
    """The local dictionary of one shard holding the whole text."""
    be = pkg.shards.CudaBackend(0)
    buf = torch.from_numpy(np.frombuffer(text, np.uint8).copy()).cuda()
    n = len(text)
    be.shard_scan(buf, 0, 0, n, n, True, w, p, True)
    return be, be.shard_words(-1)


def merge_twice(be, wd, count_a, count_b, w=10):
    """Every word of wd merged from two entries with the given per-entry counts."""
    cat = {k: torch.cat([wd[k], wd[k]]) for k in ("fpa", "fpb", "len", "uwords", "pool")}
    cnt = torch.cat([count_a, count_b]).contiguous()
    return be.dict_merge(cat["fpa"].contiguous(), cat["fpb"].contiguous(), cat["len"].contiguous(), cnt,
                         cat["uwords"].contiguous(), cat["pool"].contiguous(), w)


def test_weighted_merge_counts_at_the_limit(pkg):
    text = pkg.synth.pangenome_text(30_000, 6, 93).numpy().tobytes()
    want = orc.parse(text, 10, 100)
    occ_want = np.frombuffer(want.occ, np.uint32).astype(np.uint64)
    be, wd = shard_words_of(pkg, text)
    try:
        d = wd["n_words"]
        assert d == occ_want.size
        # the largest count the format allows: 2^32-1 on word 0 (its two entries add up exactly)
        big = (1 << 32) - 1
        ca = wd["count"].clone()
        c0 = int(ca[0].item()) & 0xFFFFFFFF
        v = big - c0
        ca[0] = v - (1 << 32) if v >= (1 << 31) else v          # the same 32 bits as an int32
        m = merge_twice(be, wd, ca, wd["count"])
        assert m["n_distinct"] == d
        assert m["dict"].cpu().numpy().tobytes() == want.dict
        occ = m["occ"].cpu().numpy().view(np.uint32).astype(np.uint64)
        # word 0's rank: where its entry went
        r0 = int(m["rank_of_entry"][0].item()) - 1
        assert occ[r0] == big
        rest = np.ones(d, bool)
        rest[r0] = False
        assert np.array_equal(occ[rest], 2 * occ_want[rest])
        ranks = m["rank_of_entry"].cpu().numpy()
        assert np.array_equal(ranks[:d], ranks[d:])
        # one occurrence more does not fit a 32-bit count
        cb = wd["count"].clone()
        cb[0] = cb[0] + 1
        with pytest.raises(pkg.pfp.PfpError) as e:
            merge_twice(be, wd, ca, cb)
        assert e.value.code == -5
    finally:
        be.scanner.close()
