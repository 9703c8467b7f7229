"""Multi-GPU k-mer spectrum: one process per GPU, sharded by canonical k-mer.

`sharded_count` is a thin caller of the library's group API (include/apgk.h, csrc/group.cuh): every rank runs
levels 0 and 1 of the single-GPU pipeline on ITS reads, the ranks all-gather the bucket histogram, cut the bucket
space into `world` contiguous ranges of (nearly) equal cost (keys + a charge per bucket), every rank gathers the ranges it owns
straight from the peers' partition buffers over NVLink peer memory (the exchange is fused into the gather kernel)
and sorts + counts them; the per-rank spectra -- disjoint sets of k-mers, so plain integer sums -- are all-reduced.
A k-mer's owner depends on the canonical k-mer alone, so counts are final without a merge (SURVEY.md section 8e).
When a rank's k-mers do not fit its device at once the library runs the same pipeline in k-mer-space rounds.
torch.distributed is used for one thing only: handing rank 0's group id to the other ranks.

The rest of this module is the HOST mirror of the exchange (numpy + gloo/nccl all_to_all), which the CPU test-suite
runs at world size 2 and 3: the splitter rule (`balanced_splitters`: the rule of the device's k_splitters, here on
instance counts), the round planning (`plan_rounds`) and the sparse-spectrum merge, so the host logic of the N-rank
path is covered without a GPU.
"""
import numpy as np
import torch
import torch.distributed as dist


def _splitters_tensor(bucket_totals, world):
    """bounds as an int64 tensor [world+1] on the device of bucket_totals (no host round trip)."""
    t = bucket_totals.to(torch.int64)
    nb = int(t.numel())
    dev = t.device
    if nb == 0:
        return torch.zeros(world + 1, dtype=torch.int64, device=dev)
    cum = torch.cumsum(t, 0)
    total = cum[-1]
    r = torch.arange(1, world, dtype=torch.int64, device=dev)
    targets = torch.div(total * r, world, rounding_mode="floor")
    inner = torch.searchsorted(cum, targets, right=True).clamp(max=nb)
    return torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), inner,
                      torch.full((1,), nb, dtype=torch.int64, device=dev)])


def balanced_splitters(bucket_totals, world):
    """Cut buckets [0, nb) into `world` contiguous ranges with (nearly) equal instance counts.
    bucket_totals: 1-D integer torch tensor or numpy array (instances per bucket, summed over ranks).
    -> list of world+1 bucket indices, bounds[0] = 0, bounds[world] = nb, non-decreasing: range r ends
    after the first bucket whose cumulative count exceeds total * (r+1) / world.
    Deterministic in its input, so every rank derives the same ownership."""
    if not isinstance(bucket_totals, torch.Tensor):
        bucket_totals = torch.from_numpy(np.ascontiguousarray(np.asarray(bucket_totals)).astype(np.int64))
    return [int(x) for x in _splitters_tensor(bucket_totals, world).cpu()]


def plan_rounds(level0_max, capacity):
    """Cut the level-0 buckets [0, len(level0_max)) into consecutive ranges whose summed entries stay within
    `capacity` (a single bucket above it gets a range of its own).  level0_max: per bucket, the largest count any
    rank holds.  Deterministic in its input, so every rank derives the same rounds.  -> list of (lo, hi)."""
    rounds, lo, acc = [], 0, 0
    for d, t in enumerate(int(x) for x in level0_max):
        if acc and acc + t > capacity:
            rounds.append((lo, d))
            lo, acc = d, 0
        acc += t
    rounds.append((lo, len(level0_max)))
    return rounds


def sharded_count(kc, rank, world, group=None, timings=None):
    """Run the sharded pipeline on this rank's KmerCounter `kc` (reads already in its store): one call into the
    library (apgk_group_count); torch.distributed only carries the 128-byte group id once.

    Returns (spectrum uint64 array summed over all ranks, n_instances_global, n_distinct_global).
    The rank's own shard table stays queryable in `kc`: the counts of ALL the k-mers it owns, every k-mer-space
    round appended."""
    grp = _group_of(kc, rank, world, group)
    grp.count()
    ni, nd = grp.totals()
    if timings is not None:
        st = grp.stats()
        ms = kc.stage_ms()
        timings.update({k: float(v) for k, v in ms.items() if v})
        timings["path"] = "partition-first/" + ("peer" if st["peer_exchange"] else "nccl") + ("" if st["n_rounds"] == 1 else "/rounds")
        timings["n_rounds"] = st["n_rounds"]
        timings["n_outer_rounds"] = st["n_outer_rounds"]
        timings["prefix_bits"] = st["prefix_bits"]
        timings["split_bits"] = st["split_bits"]
        timings["shard_instances"] = st["shard_instances"]
        timings["remote_bytes"] = st["remote_bytes"]
        timings["gather_ms"] = st["gather_ms"]
        timings["gather_remote_GBps"] = (st["remote_bytes"] / (st["gather_ms"] * 1e-3) / 1e9) if st["gather_ms"] > 0 else 0.0
        timings["step_ms"] = st["step_ms"]
    return grp.spectrum(), ni, nd


def sharded_read_freqs(kc, rank, world, first_base=0, n_bases=None, group=None, stats=None):
    """After `sharded_count`: the GLOBAL count of the canonical k-mer at every base of [first_base, first_base +
    n_bases) of this rank's read store (default: to its end), as a host uint32 array (0xFFFFFFFF where the window
    leaves its read).  Collective: every rank calls it, each with its own range (apgk_group_read_freqs_device)."""
    grp = _group_of(kc, rank, world, group)
    return grp.read_freqs([first_base], None if n_bases is None else [n_bases], stats=stats)[0]


def _group_of(kc, rank, world, group=None):
    """The library-side group of this counter (made once: rank 0's id is broadcast over torch.distributed)."""
    from .kmers import KmerGroup

    grp = getattr(kc, "_group", None)
    if grp is not None and grp._h:
        return grp
    if world == 1:
        grp = KmerGroup.local([kc])
    else:
        uid = KmerGroup.unique_id() if rank == 0 else np.zeros(128, dtype=np.uint8)
        t = torch.from_numpy(uid.copy())
        if dist.get_backend(group) == "nccl":
            t = t.cuda()
        src = dist.get_global_rank(group, 0) if group is not None else 0
        dist.broadcast(t, src=src, group=group)
        grp = KmerGroup.join(kc, t.cpu().numpy(), rank, world)
    kc._group = grp
    return grp


def merge_sparse_spectra(spec, ni, nd, world, dev, group=None):
    """Sum per-rank sparse spectra {frequency: n_kmers} (disjoint k-mer sets, so plain sums) and the totals over
    the ranks: frequencies below 65536 and the totals in one all-reduce, the (rare) larger ones gathered.
    -> (dense uint64 spectrum up to the largest frequency, n_instances, n_distinct).  Works on gloo and nccl."""
    DENSE = 65536
    dense = np.zeros(DENSE + 2, dtype=np.int64)
    far = {}
    for x, y in spec.items():
        if x < DENSE:
            dense[x] = y
        else:
            far[int(x)] = int(y)
    dense[DENSE], dense[DENSE + 1] = ni, nd
    td = torch.from_numpy(dense).to(dev)
    dist.all_reduce(td, op=dist.ReduceOp.SUM, group=group)
    dense = td.cpu().numpy()
    far_all = [None] * world
    dist.all_gather_object(far_all, far, group=group)
    far = {}
    for d_ in far_all:
        for x, y in d_.items():
            far[x] = far.get(x, 0) + y
    nz = np.nonzero(dense[:DENSE])[0]
    top = max([int(nz.max()) if len(nz) else 0] + list(far.keys()))
    out = np.zeros(top + 1, dtype=np.uint64)
    out[: min(top + 1, DENSE)] = dense[: min(top + 1, DENSE)].astype(np.uint64)
    for x, y in far.items():
        out[x] = y
    return out, int(dense[DENSE]), int(dense[DENSE + 1])


# ---------------------------------------------------------------------------
# Host-side logic of the shuffle, separated so it can be tested on CPU with gloo:
# the same ownership rule and the same exchange, with numpy doing what the kernels do.
# ---------------------------------------------------------------------------
def host_shuffle(kmers, K, rank, world, group=None):
    """kmers: uint64[n, W] canonical k-mer instances held by this rank (host).  Routes every
    instance to its owner with all_to_all (gloo or nccl) and returns the instances this rank owns."""
    from .kmers import owner_of, words_per_kmer

    W = words_per_kmer(K)
    kmers = np.ascontiguousarray(kmers, dtype=np.uint64).reshape(-1, W)
    own = owner_of(K, kmers, world) if len(kmers) else np.zeros(0, dtype=np.uint32)
    order = np.argsort(own, kind="stable")
    send_counts = np.bincount(own, minlength=world).astype(np.int64)
    send = torch.from_numpy(kmers[order].astype(np.int64).reshape(-1))
    t_recv_counts = torch.empty(world, dtype=torch.int64)
    dist.all_to_all_single(t_recv_counts, torch.from_numpy(send_counts), group=group)
    recv_counts = t_recv_counts.numpy()
    recv = torch.empty(int(recv_counts.sum()) * W, dtype=torch.int64)
    dist.all_to_all_single(recv, send, output_split_sizes=[int(c) * W for c in recv_counts],
                           input_split_sizes=[int(c) * W for c in send_counts], group=group)
    return recv.numpy().astype(np.uint64).reshape(-1, W)


def host_partition_shuffle(kmers, K, prefix_bits, rank, world, group=None):
    """Host mirror of the partition-first exchange (gloo or nccl): kmers uint64[n, W] canonical k-mer
    instances held by this rank.  Buckets = leading prefix_bits of the 2K-bit k-mer; bucket ranges are
    cut by `balanced_splitters` from the all-gathered histogram; returns (the instances this rank owns,
    (bucket_lo, bucket_hi))."""
    from .kmers import words_per_kmer

    W = words_per_kmer(K)
    kmers = np.ascontiguousarray(kmers, dtype=np.uint64).reshape(-1, W)
    top = 2 * K - 64 * (W - 1)  # bits in word 0
    if prefix_bits > 2 * K:
        raise ValueError("prefix longer than the k-mer")
    if prefix_bits <= top:
        bucket = (kmers[:, 0] >> np.uint64(top - prefix_bits)).astype(np.int64) if len(kmers) else np.zeros(0, np.int64)
    else:  # the prefix reaches into word 1
        r = prefix_bits - top
        bucket = ((kmers[:, 0] << np.uint64(r)) | (kmers[:, 1] >> np.uint64(64 - r))).astype(np.int64)
    nb = 1 << prefix_bits
    sizes = torch.from_numpy(np.bincount(bucket, minlength=nb).astype(np.int64))
    all_sizes = [torch.empty(nb, dtype=torch.int64) for _ in range(world)]
    dist.all_gather(all_sizes, sizes, group=group)
    all_sizes = torch.stack(all_sizes)
    bounds = balanced_splitters(all_sizes.sum(0), world)
    order = np.argsort(bucket, kind="stable")
    cum = np.concatenate([[0], np.cumsum(all_sizes.numpy(), axis=1)[rank]])
    send_counts = np.array([cum[bounds[r + 1]] - cum[bounds[r]] for r in range(world)], dtype=np.int64)
    send = torch.from_numpy(kmers[order].astype(np.int64).reshape(-1))
    t_recv_counts = torch.empty(world, dtype=torch.int64)
    dist.all_to_all_single(t_recv_counts, torch.from_numpy(send_counts), group=group)
    recv_counts = t_recv_counts.numpy()
    recv = torch.empty(int(recv_counts.sum()) * W, dtype=torch.int64)
    dist.all_to_all_single(recv, send, output_split_sizes=[int(c) * W for c in recv_counts],
                           input_split_sizes=[int(c) * W for c in send_counts], group=group)
    return recv.numpy().astype(np.uint64).reshape(-1, W), (bounds[rank], bounds[rank + 1])
