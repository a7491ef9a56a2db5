"""CPU tests of the host side: formats, C-ABI surface, sharding + gather (gloo, world_size 2)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as ol
from fastga_b200 import formats, shard, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import fastga_b200
    lib = fastga_b200.load_library()
    hdr = open(os.path.join(ROOT, "include", "fastga_b200.h")).read()
    names = set(re.findall(r"\b(fgb_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) > 35
    for n in sorted(names):
        assert hasattr(lib, n), "libfastga_b200.so does not export %s" % n


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    import fastga_b200
    monkeypatch.setattr(fastga_b200, "_lib", None)
    monkeypatch.setattr(fastga_b200, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(fastga_b200.LibraryMissing):
        fastga_b200.load_library()


def test_no_product_module_touches_the_oracle():
    pk = os.path.join(ROOT, "fastga_b200")
    for f in os.listdir(pk):
        if f.endswith(".py") and f != "smoke.py":
            src = open(os.path.join(pk, f)).read()
            assert "oracle" not in src.replace("oracle/_ref", ""), f


def test_fasta_roundtrip_and_contig_split(tmp_path):
    rng = np.random.default_rng(1)
    c1, c2, c3 = (rng.integers(0, 4, n, dtype=np.uint8) for n in (1001, 37, 4000))
    scaf = [("s1 first", np.concatenate([c1, np.full(7, 4, np.uint8), c2])), ("s2", c3)]
    p = str(tmp_path / "x.fasta.gz")
    formats.write_fasta(p, scaf, width=60)
    g = formats.genome_from_fasta(p)
    assert list(g.clen) == [1001, 37, 4000]
    assert list(g.scaf) == [0, 0, 1] and list(g.sbeg) == [0, 1008, 0]
    assert g.names == ["s1 first", "s2"]
    for i, c in enumerate((c1, c2, c3)):
        assert np.array_equal(g.contig(i), c)
    assert list(g.boff) == [0, 251, 261]
    assert abs(float(g.freq.sum()) - 1.0) < 1e-6


def test_gix_file_roundtrip(tmp_path):
    rng = np.random.default_rng(2)
    n, pb, cb = 1000, 3, 1
    E = 9 + pb + cb
    ent = rng.integers(0, 256, n * E, dtype=np.uint8)
    index = np.sort(rng.integers(0, n + 1, 1 << 24)).astype(np.int64)
    p = str(tmp_path / "g.gix")
    formats.write_gix(p, 40, index, pb, cb, 123, np.arange(5, dtype=np.int32), ent, [400, 600])
    g = formats.read_gix(p)
    assert (g.kmer, g.nparts, g.post_bytes, g.cont_bytes, g.maxpre, g.marker) == (40, 2, pb, cb, 123, -1)
    assert np.array_equal(g.entries, ent) and np.array_equal(g.index, index) and g.part_n == [400, 600]


def test_ktab_lcp_and_canonical_form():
    tab = np.array([[0x0001 << 48 | 5, 0x10], [0x0001 << 48 | 9, 0x10], [0x0002 << 48 | 1, 0x10],
                    [3, 0x4000000000000011]], dtype=np.uint64)
    lcp = formats.table_lcp(tab, [0])
    assert list(lcp) == [0, 40, 39, 0]


def test_kmer_space_ownership_covers_everything_once():
    """the sharded path's two ownership maps: k-mer prefix ranges (by the first four bases) tile the
    prefix space, contigs are spread by length"""
    for world in (1, 2, 3, 4, 8):
        cuts = shard.top_byte_cuts(world)
        assert cuts[0] == 0 and cuts[-1] == 256 and all(a <= b for a, b in zip(cuts, cuts[1:]))
        assert max(b - a for a, b in zip(cuts, cuts[1:])) - min(b - a for a, b in zip(cuts, cuts[1:])) <= 1
        lens = [50, 10, 40, 30, 20, 60, 5, 33]
        own = shard.owner_of_contigs(lens, world)
        assert set(own.tolist()) <= set(range(world))
        loads = [sum(l for l, o in zip(lens, own) if o == r) for r in range(world)]
        assert max(loads) - min(loads) <= max(lens)


_XWORKER = r'''
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch, torch.distributed as dist
from fastga_b200 import shard
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
rng = np.random.default_rng(7)                       # same stream on every rank: everybody knows every block
send = rng.integers(0, 50, (world, world))           # send[src][dst] rows
send[0, 1] = 0                                       # an empty block
blocks = [[rng.integers(-2**62, 2**62, (int(send[s, d]), 2)) for d in range(world)] for s in range(world)]
mine = np.concatenate(blocks[rank]) if send[rank].sum() else np.zeros((0, 2), np.int64)
got = shard.exchange_rows(dist, torch.from_numpy(mine.astype(np.int64)), [int(v) for v in send[rank]])
want = np.concatenate([blocks[s][rank] for s in range(world)])
assert got.shape == want.shape and np.array_equal(got.numpy(), want), (rank, got.shape, want.shape)
# the pipelined form the sharded path uses: two exchanges in flight, waited for in issue order
src = torch.from_numpy(mine.astype(np.int64))
g1, w1 = shard.exchange_rows(dist, src, [int(v) for v in send[rank]], async_op=True)
g2, w2 = shard.exchange_rows(dist, src * 3, [int(v) for v in send[rank]], async_op=True)
w1.wait(); w2.wait()
assert np.array_equal(g1.numpy(), want) and np.array_equal(g2.numpy(), want * 3)
print("XCHG_OK", rank)
dist.destroy_process_group()
'''


def test_record_exchange_gloo_world2(tmp_path):
    """the all-to-all of 16-byte records that moves k-mer records and seeds between ranks (N > 1 path)"""
    script = tmp_path / "xworker.py"
    script.write_text(_XWORKER % {"root": ROOT})
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29583", str(script)],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.count("XCHG_OK") == 2, r.stdout[-3000:]


_WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r); sys.path.insert(0, os.path.join(%(root)r, "tests"))
import numpy as np, torch, torch.distributed as dist
from fastga_b200 import lib, shard
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
rng = np.random.default_rng(100 + rank)
n = 5 + 3 * rank
fields = rng.integers(0, 1000, (n, 9)).astype(np.int32)
fields[:, 1] = rng.integers(0, 2, n)          # local contig numbers
fields[:, 8] = 2 * rng.integers(1, 6, n)      # tlen
toff = np.concatenate([[0], np.cumsum(fields[:-1, 8])]).astype(np.int64)
pool = rng.integers(0, 256, int(fields[:, 8].sum()), dtype=np.uint8)
al = lib.Alignments(fields, toff, pool, n)
cmap = np.array([10 * rank, 10 * rank + 1], dtype=np.int32)
merged = shard.gather_alignments(al, cmap, dist, torch.device("cpu"))
np.save(os.path.join(%(out)r, "lines_%%d.npy" %% rank), np.array(
    [l.replace("A %%d " %% int(f[1]), "A %%d " %% int(cmap[f[1]]), 1) for l, f in zip(
        lib.Alignments(fields, toff, pool, n).canonical_lines_unsorted(), fields)], dtype=object), allow_pickle=True)
if rank == 0:
    assert len(merged) == sum(5 + 3 * r for r in range(world))
    key = merged.fields[:, [1, 3, 2, 0]]
    assert all(tuple(key[i]) <= tuple(key[i + 1]) for i in range(len(key) - 1))
    np.save(os.path.join(%(out)r, "merged.npy"), np.array(merged.canonical_lines(), dtype=object), allow_pickle=True)
dist.destroy_process_group()
'''


def test_gather_alignments_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % {"root": ROOT, "out": str(tmp_path)})
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29581")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29581", str(script)],
                       env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:]
    merged = list(np.load(tmp_path / "merged.npy", allow_pickle=True))
    want = sorted(list(np.load(tmp_path / "lines_0.npy", allow_pickle=True)) +
                  list(np.load(tmp_path / "lines_1.npy", allow_pickle=True)))
    assert merged == want


# ---- the hit-group rule of fgb_extend (host code of the library, no device) ----

from fastga_b200 import lib  # noqa: E402  (ctypes mirror; this rule needs no device)

INF = np.iinfo(np.int64).max


def _groups(hrange, tinfo, hits, **kw):
    items, nxt = lib.hit_groups_host(hrange, tinfo, hits, **kw)
    # per triple: list of (first hit number in the triple, hits) in chain order
    out = {}
    for (w, h0, hn, g), (na, nh) in zip(items.tolist(), nxt.tolist()):
        out.setdefault(w, []).append((g, hn, na, nh))
    return {w: sorted(v) for w, v in out.items()}, items


def test_hit_groups_far_apart_chains_of_one_triple_are_independent():
    hits = [(0, 5000), (200_000, 260_000), (900_000, 910_000)]
    g, items = _groups([(0, 3)], [(7, 100)], hits)
    assert g == {0: [(0, 1, 200_000, 260_000), (1, 1, 900_000, 910_000), (2, 1, INF, INF)]}
    # launch order: longest component first
    assert items[:, 3].tolist() == [1, 2, 0]


def test_hit_groups_chains_bridged_by_the_neighbouring_band_pair_stay_together():
    # triple 0 (band 100): two chains 40 kbp apart; triple 1 (band 101, same contig pair) holds one
    # chain that overlaps both (the block's path drifted into the next band and back)
    hits = [(0, 50_000), (90_000, 150_000),          # triple 0
            (45_000, 95_000)]                          # triple 1
    g, _ = _groups([(0, 2), (2, 1)], [(7, 100), (7, 101)], hits)
    assert g[0] == [(0, 2, INF, INF)] and g[1] == [(0, 1, INF, INF)]
    # another contig pair (key) or a band pair further away does not bridge
    g, _ = _groups([(0, 2), (2, 1)], [(7, 100), (8, 101)], hits)
    assert [x[:2] for x in g[0]] == [(0, 1), (1, 1)]
    g, _ = _groups([(0, 2), (2, 1)], [(7, 100), (7, 103)], hits)
    assert [x[:2] for x in g[0]] == [(0, 1), (1, 1)]
    g, _ = _groups([(0, 2), (2, 1)], [(7, 100), (7, 103)], hits, bands=3)
    assert [x[:2] for x in g[0]] == [(0, 2)]


def test_hit_groups_a_foreign_chain_between_two_of_one_block_is_not_cut_out():
    # triple 0: X1, Y, X2 in chain order; X1 and X2 are joined through triple 1's long chain, Y is on
    # its own: a group must be a contiguous run, so all three stay in one group (cutting Y out would
    # leave X2 to run as if X1's alignment had not covered it)
    hits = [(0, 30_000), (40_000, 45_000), (60_000, 90_000),     # triple 0: X1 Y X2
            (25_000, 65_000)]                                      # triple 1 bridges X1 and X2 ... and Y
    g, _ = _groups([(0, 3), (3, 1)], [(1, 10), (1, 11)], hits)
    assert g[0] == [(0, 3, INF, INF)]
    # a Y that really is foreign: X1 and X2 are joined through band 11 (B1, B2) and band 12 (C, which
    # overlaps B1 and B2 but is two bands from triple 0, so it does not reach Y): components
    # {X1, B1, C, B2, X2} and {Y}, chain order X Y X in triple 0 -> still one contiguous group
    hits = [(0, 30_000), (40_000, 45_000), (60_000, 90_000),     # triple 0, band 10: X1 Y X2
            (25_000, 32_000), (58_000, 65_000),                  # triple 1, band 11: B1 B2
            (30_000, 60_000)]                                    # triple 2, band 12: C
    g, _ = _groups([(0, 3), (3, 2), (5, 1)], [(1, 10), (1, 11), (1, 12)], hits)
    assert g[0] == [(0, 3, INF, INF)]
    assert g[1] == [(0, 2, INF, INF)] and g[2] == [(0, 1, INF, INF)]
    # without the bridge Y and the X's are three components and three groups
    g, _ = _groups([(0, 3)], [(1, 10)], hits[:3])
    assert [x[:2] for x in g[0]] == [(0, 1), (1, 1), (2, 1)]


def test_hit_groups_gap_rule_and_triples_without_a_list():
    hits = [(0, 10), (5_000, 5_010), (100_000, 100_010)]
    g, _ = _groups([(0, 3), (0, 0x80000000), (0, 0)], [(1, 1), (1, 50), (1, 90)], hits, gap=0)
    assert [x[:2] for x in g[0]] == [(0, 1), (1, 1), (2, 1)]
    assert g[1] == [(0, 0x80000000, INF, INF)] and 2 not in g
    g, _ = _groups([(0, 3)], [(1, 1)], hits, gap=50_000)
    assert [x[:2] for x in g[0]] == [(0, 2), (2, 1)]
    g, _ = _groups([(0, 3)], [(1, 1)], hits, gap=10**9)
    assert [x[:2] for x in g[0]] == [(0, 3)]
