"""GPU parity at store sizes where 32-bit quantities fill up: base positions, occurrence slots and group batch offsets past
2^31 and 2^32, and 4-byte level-1 remainders that use all 32 bits.  The full oracle cannot run at these sizes, so the
sampled-partition oracle (oracle_sample_prefix_pos) scans every read, keeps the instances of a few leading-bit
partitions with their positions, and those partitions are compared record by record; whole-store identities (the count
of invalid windows, windows per frequency = f * spectrum[f]) cover the rest of the store.

Two contexts, built one after the other (the first is closed before the second is built):
  A  the benchmark store: K = 25, 60 M x 100 bp reads (6.0 G bases, 4.56 G instances), automatic geometry (REM = 30).
     The records pack remainder and position into one word at exactly 64 bits (30 + 34, 2 * 6.0 G < 2^34).
  B  K = 26, prefix_bits = 20 (REM = 32), 22 M x 100 bp reads (2.2 G bases): 32 + 33 > 64, so the records keep
     remainders and positions in two arrays.

Each assertion names, in a comment, the 32-bit quantity it guards.

Measured on one NVIDIA B200 (1000 W power limit, 177.7 GiB free at the start): context A used 159.8 GiB of device
memory at its peak (the low point of free memory seen after each large call), context B 44.8 GiB; the module took 56 s,
26 s of it in the two set-ups (device count, the reads generated again on the host, the sampled oracle's scan and sort).
The card is shared, so the module skips, saying why, when less than MIN_FREE_BYTES is free."""
import concurrent.futures
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MIN_FREE_BYTES = 165 << 30   # context A's 159.8 GiB peak and some room
PBITS = 8
NONE32 = -1   # 0xFFFFFFFF read back as int32


class _CudaView:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def _device_array(ptr, n, typestr):
    import torch

    return torch.as_tensor(_CudaView(ptr, n, typestr), device="cuda")


def _revcomp(x, K):
    t, rc = x.copy(), np.zeros(len(x), dtype=np.uint64)
    for _ in range(K):
        rc = (rc << np.uint64(2)) | (np.uint64(3) - (t & np.uint64(3)))
        t >>= np.uint64(2)
    return rc


def _forward_kmers(words, q, K):
    """forward k-mer of the window starting at each base q, rebuilt from the packed reads (base q at bits [2q, 2q+2))"""
    fw = np.zeros(len(q), dtype=np.uint64)
    for j in range(K):
        b = q + np.uint64(j)
        fw = (fw << np.uint64(2)) | ((words[b >> np.uint64(5)] >> ((b & np.uint64(31)) << np.uint64(1))) & np.uint64(3))
    return fw


class _Memory:
    """Free device memory seen at checkpoints after each large call: the library allocates with cudaMalloc and keeps
    its buffers until the context closes, so the lowest value seen bounds what the module used."""

    def __init__(self):
        import torch

        self.start = torch.cuda.mem_get_info()[0]
        self.low = self.start

    def mark(self):
        import torch

        self.low = min(self.low, torch.cuda.mem_get_info()[0])


_STATE = {}


def _close_current():
    kc = _STATE.pop("kc", None)
    if kc is not None:
        kc.close()


def _setup(oracle, K, prefix_bits, n_reads, genome, parts_fn, rem, elem):
    import torch

    from allpathslg_b200 import KmerCounter, synth_params

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _close_current()
    torch.cuda.empty_cache()
    free = torch.cuda.mem_get_info()[0]
    if free < MIN_FREE_BYTES:
        pytest.skip("needs %.0f GiB of free device memory, %.1f GiB free (the card is shared)" % (MIN_FREE_BYTES / 2**30, free / 2**30))
    mem = _Memory()
    print("\n%s: %.1f GiB free of %.1f GiB" % (torch.cuda.get_device_name(), free / 2**30,
                                            torch.cuda.mem_get_info()[1] / 2**30))
    L = 100
    kc = KmerCounter(K, want_counts=True, prefix_bits=prefix_bits)
    _STATE["kc"] = kc
    kc.synth_reads(synth_params(genome, L), 0, n_reads)
    kc.finish()
    mem.mark()
    g = kc.geometry()
    assert (g["REM"], g["elem_bytes"]) == (rem, elem)           # remainder width: the layout this context names
    tb, _ = kc.read_store_info()
    ni, nd = kc.totals()
    assert tb == n_reads * L and ni == n_reads * (L - K + 1)
    host, _ = oracle.synth_reads(oracle.synth_params(genome, L), 0, n_reads)
    exported = kc.export_reads()
    assert len(exported) == len(host) and np.array_equal(exported, host)   # base position: the store past 2^32 bases
    del exported
    parts = parts_fn(kc)
    n_threads = os.cpu_count() or 1
    keys, pos, nw = oracle.sample_prefix_pos(host, None, K, PBITS, parts, n_reads=n_reads, read_len=L, n_threads=n_threads)
    assert nw == ni == n_reads * (L - K + 1)                   # base position: every window of the store was scanned
    keys = keys[:, 0]
    # sort by (k-mer, position): the oracle returns ascending positions, so a stable sort by k-mer per partition
    top = 2 * K - PBITS
    pre = (keys >> np.uint64(top)).astype(np.int64)
    sel = [np.nonzero(pre == p)[0] for p in parts]

    def sort_part(ix):
        return ix[np.argsort(keys[ix], kind="stable")]

    with concurrent.futures.ThreadPoolExecutor(len(parts)) as ex:
        order = np.concatenate(list(ex.map(sort_part, sel)))
    keys, pos = keys[order], pos[order]
    sk, sc = oracle.count_keys(keys[:, None], K, n_threads=n_threads)
    sk = sk[:, 0]
    assert int(sc.sum()) == len(keys)
    return dict(kc=kc, K=K, L=L, tb=tb, ni=ni, nd=nd, host=host, parts=parts, keys=keys, pos=pos, sk=sk, sc=sc,
                top=top, mem=mem)


def _part_bounds(S, part):
    lo = np.searchsorted(S["keys"], np.uint64(part << S["top"]))
    hi = np.searchsorted(S["keys"], np.uint64((part + 1) << S["top"]))
    dlo = np.searchsorted(S["sk"], np.uint64(part << S["top"]))
    dhi = np.searchsorted(S["sk"], np.uint64((part + 1) << S["top"]))
    return lo, hi, dlo, dhi


def _check_counts(S):
    """table records of every sampled partition, and lookups of present and absent k-mers"""
    kc, K = S["kc"], S["K"]
    n_rec = 0
    for part in S["parts"]:
        _, _, dlo, dhi = _part_bounds(S, part)
        first, n = kc.prefix_range(PBITS, part)
        gk, gc = kc.counts(first, n)
        assert n == dhi - dlo                                         # remainder width: no k-mer lost or merged
        assert (gk[:, 0] == S["sk"][dlo:dhi]).all()                   # remainder width: keys rebuilt from 32-bit elements
        assert (gc.astype(np.uint64) == S["sc"][dlo:dhi]).all()       # base position: every instance counted once
        n_rec += n
    rng = np.random.default_rng(K)
    idx = rng.integers(0, len(S["sk"]), size=100_000)
    q, exp = S["sk"][idx], S["sc"][idx]
    assert (kc.lookup(q[:, None], canonicalise=False).astype(np.uint64) == exp).all()              # remainder width
    assert (kc.lookup(_revcomp(q, K)[:, None], canonicalise=True).astype(np.uint64) == exp).all()  # remainder width
    # random k-mers of the sampled partitions that the oracle did not see must be absent
    parts = np.asarray(S["parts"], dtype=np.uint64)
    r = (parts[rng.integers(0, len(parts), size=200_000)] << np.uint64(S["top"])) | \
        rng.integers(0, 1 << S["top"], size=200_000, dtype=np.int64).astype(np.uint64)
    canon = np.minimum(r, _revcomp(r, K))
    absent = ~np.isin(r, S["sk"])
    assert absent.sum() > 100_000
    assert (kc.lookup(r[absent][:, None], canonicalise=False) == 0).all()                         # remainder width
    mine = np.isin(canon >> np.uint64(S["top"]), parts) & ~np.isin(canon, S["sk"])
    assert mine.sum() > 10_000
    assert (kc.lookup(r[mine][:, None], canonicalise=True) == 0).all()                            # remainder width
    return n_rec


def _check_freqs_bulk(S, out):
    """read_freqs_device output: the sampled positions and two identities over the whole store"""
    import torch

    kc = S["kc"]
    q = torch.from_numpy((S["pos"] >> np.uint64(1)).astype(np.int64)).cuda()
    got = out[q].cpu().numpy().view(np.uint32)
    del q
    exp = np.repeat(S["sc"], S["sc"].astype(np.int64))
    assert (got.astype(np.uint64) == exp).all()                       # base position: the answer lands on its own base
    tb, ni = S["tb"], S["ni"]
    assert int((out == NONE32).sum()) == tb - ni                      # base position: no window lost or written twice
    spec = kc.spectrum()
    hist = torch.zeros(len(spec), dtype=torch.int64, device="cuda")
    step = 1 << 28
    for a in range(0, tb, step):
        v = out[a:a + step]
        h = torch.bincount(v[v != NONE32].to(torch.int64), minlength=len(spec))
        assert len(h) == len(spec)                                    # base position: no count above the spectrum's
        hist += h
        del v, h
    hist = hist.cpu().numpy().astype(np.uint64)
    f = np.arange(len(spec), dtype=np.uint64)
    assert (hist == f * spec).all()                                   # base position: f windows for each k-mer of count f


def _check_records(S):
    """occurrence records of every sampled partition, record by record, and run offsets = scan of the counts"""
    import torch

    kc, L = S["kc"], S["L"]
    info = kc.build_occurrences()
    S["mem"].mark()
    assert info["n_occ"] == S["ni"]                                   # occurrence slot: one slot per instance
    d_off, _, n_occ = kc.occurrences_device()
    assert n_occ == S["ni"]
    kp, cp, nd = kc.counts_device()
    assert nd == S["nd"]
    run_off = _device_array(d_off, nd + 1, "<i8")
    scan = _device_array(cp, nd, "<i4").to(torch.int64).cumsum(0)
    assert int(run_off[0]) == 0 and int(run_off[-1]) == S["ni"]       # occurrence slot: the last run ends at n_instances
    assert torch.equal(run_off[1:], scan)                             # occurrence slot: every run starts at the scan
    del scan
    torch.cuda.empty_cache()
    n_rec = 0
    for part in S["parts"]:
        lo, hi, dlo, dhi = _part_bounds(S, part)
        first, n = kc.prefix_range(PBITS, part)
        ro, rid, pos = kc.occurrences(first, n)
        g = (S["pos"][lo:hi] >> np.uint64(1)).astype(np.int64)
        p1 = (g % L + 1).astype(np.int32)
        erid = (g // L).astype(np.uint32)
        epos = np.where(S["pos"][lo:hi] & np.uint64(1), -p1, p1)
        exp_ro = np.concatenate([[0], np.cumsum(S["sc"][dlo:dhi].astype(np.int64))]).astype(np.uint64)
        assert (ro == exp_ro).all()                                   # occurrence slot: run offsets inside the partition
        assert (rid == erid).all()                                    # read id: through the rank directory past 2^31 bases
        assert (pos == epos).all()                                    # base position: position in the read and strand
        n_rec += len(rid)
    return n_rec, run_off


# ---------------------------------------------------------------- context A: the benchmark store
A_READS, A_GENOME, A_K = 60_000_000, 100_000_000, 25
SLOT32 = 1 << 32


def _a_parts(kc):
    """partitions 0 (poly-A, the densest), 5, 77, 130, 201 and the one whose run holds occurrence slot 2^32"""
    import torch

    kp, cp, nd = kc.counts_device()
    scan = _device_array(cp, nd, "<i4").to(torch.int64).cumsum(0)
    row = int(torch.searchsorted(scan, torch.tensor([SLOT32], device="cuda"), right=True)[0])
    del scan
    torch.cuda.empty_cache()
    k, _ = kc.counts(row, 1)
    _STATE["slot32_row"] = row
    return sorted({0, 5, 77, 130, 201, int(k[0, 0]) >> (2 * A_K - PBITS)})


@pytest.fixture(scope="module")
def ctx_a(oracle):
    S = _setup(oracle, A_K, 0, A_READS, A_GENOME, _a_parts, rem=30, elem=4)
    # records: remainder and position share one word exactly when REM + bit length of 2 * total_bases <= 64
    pack_bits = int(2 * S["tb"]).bit_length()
    assert pack_bits == 34 and 30 + pack_bits == 64                   # remainder width + base position: all 64 bits used
    yield S
    _close_current()


def test_a_counts_and_lookups(ctx_a):
    S = ctx_a
    n_rec = _check_counts(S)
    print("\n[A] sampled instances %d, table records compared %d, partitions %s" % (len(S["keys"]), n_rec, S["parts"]))


def test_a_occurrence_records(ctx_a):
    import torch

    S = ctx_a
    kc, K, L = S["kc"], S["K"], S["L"]
    n_rec, run_off = _check_records(S)
    row = _STATE["slot32_row"]
    assert int(run_off[row]) <= SLOT32 < int(run_off[row + 1])     # occurrence slot: a sampled run holds slot 2^32
    assert S["ni"] > SLOT32
    # the reads that straddle base 2^31 and base 2^32: every window is in the run of its k-mer with its signed position
    words = S["host"].view(np.uint64)
    kp, _, nd = kc.counts_device()
    table = _device_array(kp, nd, "<i8")
    for r in (21_474_836, 42_949_672):
        assert r * L < (1 << 31 if r < 30_000_000 else 1 << 32) < (r + 1) * L
        q = np.arange(r * L, r * L + L - K + 1, dtype=np.uint64)
        fw = _forward_kmers(words, q, K)
        rc = _revcomp(fw, K)
        canon = np.minimum(fw, rc)
        rows = torch.searchsorted(table, torch.from_numpy(canon.astype(np.int64)).cuda()).cpu().numpy()
        for j in range(len(q)):
            k, _ = kc.counts(int(rows[j]), 1)
            assert k[0, 0] == canon[j]
            _, rid, pos = kc.occurrences(int(rows[j]), 1)
            want = -(j + 1) if rc[j] < fw[j] else j + 1
            assert ((rid == r) & (pos == want)).sum() == 1           # read id + base position across 2^31 / 2^32
    del table, run_off
    torch.cuda.empty_cache()
    print("\n[A] occurrence records compared %d (record layout: packed, %d + %d = 64 bits)"
          % (n_rec, 30, int(2 * S["tb"]).bit_length()))


def test_a_read_freqs_and_group(ctx_a):
    import torch

    from allpathslg_b200 import KmerGroup

    S = ctx_a
    kc, K, L, tb = S["kc"], S["K"], S["L"], S["tb"]
    kc.release_temp()
    torch.cuda.empty_cache()
    out = torch.empty(tb, dtype=torch.int32, device="cuda")
    kc.read_freqs_device(out.data_ptr())
    S["mem"].mark()
    _check_freqs_bulk(S, out)
    words = S["host"].view(np.uint64)
    n = 10_000
    for first in (0, (1 << 31) - 5000, (1 << 32) - 5000, tb - n):
        bulk = out[first:first + n].cpu().numpy().view(np.uint32)
        assert (kc.read_freqs(first, n) == bulk).all()              # base position: bulk and per-window forms agree
        q = np.arange(first, first + n, dtype=np.uint64)
        valid = (q % np.uint64(L)) <= np.uint64(L - K)
        assert ((bulk == 0xFFFFFFFF) == ~valid).all()               # base position: read ends found past 2^31 / 2^32
        fw = _forward_kmers(words, q[valid], K)
        assert (kc.lookup(fw[:, None], canonicalise=True) == bulk[valid]).all()   # base position: the window's own k-mer
    # the group lookups with one rank: batches of at most 2^31 bases, so later batches start past 2^31 and 2^32
    kc.release_temp()
    out2 = torch.empty(tb, dtype=torch.int32, device="cuda")
    with KmerGroup.local([kc]) as grp:
        grp.count()
        st = grp.read_freqs_device([out2.data_ptr()])
        S["mem"].mark()
        assert st["n_batches"] >= 3                                 # batch offset: batches start past 2^31 and 2^32
        assert st["n_queries"] == S["ni"]
        assert torch.equal(out, out2)                               # batch offset: every base of every batch in place
    print("\n[A] group read_freqs: n_batches %d; module device memory %.1f GiB (free at start %.1f GiB)"
          % (st["n_batches"], (S["mem"].start - S["mem"].low) / 2**30, S["mem"].start / 2**30))
    del out, out2
    _close_current()
    torch.cuda.empty_cache()


# ---------------------------------------------------------------- context B: 32-bit remainders, records in two arrays
B_READS, B_GENOME, B_K, B_P = 22_000_000, 100_000_000, 26, 20


@pytest.fixture(scope="module")
def ctx_b(oracle):
    S = _setup(oracle, B_K, B_P, B_READS, B_GENOME, lambda kc: [0, 77, 250], rem=32, elem=4)
    pack_bits = int(2 * S["tb"]).bit_length()
    assert pack_bits == 33 and 32 + pack_bits > 64                    # remainder width + base position: two arrays
    yield S
    _close_current()


def test_b_full_width_remainders(ctx_b):
    import torch

    S = ctx_b
    n_tab = _check_counts(S)
    n_rec, run_off = _check_records(S)
    del run_off
    S["kc"].release_temp()
    out = torch.empty(S["tb"], dtype=torch.int32, device="cuda")
    S["kc"].read_freqs_device(out.data_ptr())
    S["mem"].mark()
    _check_freqs_bulk(S, out)
    del out
    print("\n[B] sampled instances %d, table records %d, occurrence records %d (record layout: two arrays, 32 + 33 > 64); "
          "device memory %.1f GiB" % (len(S["keys"]), n_tab, n_rec, (S["mem"].start - S["mem"].low) / 2**30))
