"""Multi-GPU sharding of the path: subbands (IFs) are independent from VDIF bytes to
requantised bytes -- the reference already runs one process per IF
(/root/reference/base2fil.sh:60-66) -- so ranks take disjoint groups of IFs with no data-path
collective.  The single exchange is the frequency splice (/root/reference/base2fil.sh:422):
each rank's finished [rows, tile] bytes are gathered into the owner's band-ordered rows.
torch.distributed is plumbing only (NCCL on GPUs, gloo in the CPU tests).
"""
from __future__ import annotations


def shard_ifs(nif_total: int, world: int, rank: int) -> list[int]:
    """1-based IF numbers owned by `rank`: contiguous groups, rank 0 lowest in frequency."""
    per = (nif_total + world - 1) // world
    lo = rank * per + 1
    return list(range(lo, min(nif_total, lo + per - 1) + 1))


def rank_if_plan(nif_total: int, world: int, rank: int, freq_lsb0: float, bw: float):
    """(if numbers, signed bandwidths, centre frequencies) of one rank, following base2fil's plan
    (/root/reference/base2fil.sh:54,65,254,407-414): IF i at freqLSB_0+(i-1)*bw, odd LSB, even USB."""
    ifs = shard_ifs(nif_total, world, rank)
    bws = [bw if i % 2 == 0 else -bw for i in ifs]
    freqs = [freq_lsb0 + (i - 1) * bw for i in ifs]
    return ifs, bws, freqs


def band_reference_mhz(nif_total: int, freq_lsb0: float, bw: float, nchan: int) -> float:
    """Centre of the highest channel of base2fil's whole band (the spliced file's fch1): the delay_ref_mhz every rank of an
    IF-sharded scan passes with remove_delays, so that all ranks align their channels to the same frequency."""
    top = max(freq_lsb0 + (i - 1) * bw for i in range(1, nif_total + 1))
    return top + abs(bw) / 2 - abs(bw) / (2 * nchan)


def gather_splice(local_rows, world: int, rank: int, dst: int = 0, group=None, out=None):
    """Gather every rank's [rows, tile_bytes] uint8 tensor to `dst` and lay the tiles out in
    splice order: highest sky frequency first, i.e. rank world-1's tile leftmost
    (/root/reference/base2fil.sh:350,367).  Returns [rows, world*tile_bytes] on dst, None elsewhere."""
    import torch
    import torch.distributed as dist

    if world == 1:
        return local_rows
    rows, tile = local_rows.shape
    if rank == dst:
        if out is None:
            out = torch.empty((world, rows, tile), dtype=local_rows.dtype, device=local_rows.device)
        parts = [out[r] for r in range(world)]
    else:
        parts = None
    dist.gather(local_rows.contiguous(), parts, dst=dst, group=group)
    if rank != dst:
        return None
    # [world, rows, tile] -> [rows, world(descending), tile]
    return out.flip(0).permute(1, 0, 2).reshape(rows, world * tile)


class PeerSplice:
    """In-GPU splice across ranks without a collective on the data path: the owner's spliced rows
    [rows, world*tile_bytes] live in symmetric memory, every rank gets the owner's device pointer
    (NVLink-mapped) and its requantise kernel stores its tile there at column
    (world-1-rank)*tile_bytes -- highest sky frequency first, like base2fil's splice_list
    (/root/reference/base2fil.sh:350,367,422).  torch only provides the mapping."""

    def __init__(self, rows: int, tile_bytes: int, world: int, rank: int, device, owner: int = 0, group=None):
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm

        self.rows, self.tile, self.world, self.rank, self.owner = rows, tile_bytes, world, rank, owner
        self.pitch = world * tile_bytes
        self.col = (world - 1 - rank) * tile_bytes
        self.buf = symm.empty((rows, self.pitch), dtype=torch.uint8, device=device)
        self.handle = symm.rendezvous(self.buf, group if group is not None else dist.group.WORLD)
        self.owner_ptr = int(self.handle.buffer_ptrs[owner])

    def dst(self, row: int) -> int:
        """device pointer of this rank's tile in output row `row` of the owner's buffer"""
        return self.owner_ptr + row * self.pitch + self.col

    def result(self):
        """the spliced rows (valid on the owner after every rank has synchronised)"""
        return self.buf if self.rank == self.owner else None


# ---------------------------------------------------------------------------------------------
# Time sharding: one long scan (BASELINE config 5: 3600 s) cut into consecutive segments, one per
# rank.  Segments start where frames, FFT blocks and output samples coincide, so every rank's rows
# are exactly the rows a single GPU would produce for that stretch, and each rank writes them at
# their final offset of the same file.  The one thing the segments share is digifil's `-c` rescale
# (/root/reference/process_vdif.py:181-182: mean and sigma of the first 10 s, then frozen): the rank
# that holds the head of the scan measures it and broadcasts 2 * nif * npol * nchan floats.
def broadcast_rescale(plan, rank: int, src: int = 0, group=None, device=None):
    """Every rank ends up with src's measured (mean, scale) set on its plan."""
    import torch
    import torch.distributed as dist

    n = plan.nif * plan.nprod * plan.cfg.nchan
    buf = torch.empty(2 * n, dtype=torch.float32, device=device or "cpu")
    if rank == src:
        mean, scale = plan.rescale()
        buf[:n] = torch.from_numpy(mean.reshape(-1))
        buf[n:] = torch.from_numpy(scale.reshape(-1))
    dist.broadcast(buf, src=src, group=group)
    host = buf.cpu().numpy()
    plan.set_rescale(host[:n], host[n:])
    return host[:n].copy(), host[n:].copy()


def measure_first_interval(plan, paths, **scan_kw):
    """digifil -c statistics of THIS scan: drop any preset first (it survives b2f_reset and would end the
    stats_only pass after one chunk with the previous scan's numbers), then measure."""
    plan.set_rescale(None)
    plan.run_scan(paths, None, stats_only=True, **scan_kw)
    return plan.rescale()


def run_scan_time_sharded(plan, paths, out_path: str, world: int, rank: int, *, group=None, device=None,
                          **scan_kw) -> dict:
    """Rank `rank` of `world` processes its time segment of the scan into `out_path` (shared file system).
    Collective: call on every rank with the same arguments.  Returns this rank's b2f_run_scan result."""
    import os

    import torch.distributed as dist

    if world == 1:
        return plan.run_scan(paths, out_path, **scan_kw)
    keep_bp = bool(plan.cfg.keep_bandpass)
    # a preset left over from an earlier scan survives b2f_reset and would make the stats_only pass stop at once
    # and hand out the OLD scan's mean/scale: every rank returns to measuring first
    plan.set_rescale(None)
    if rank == 0:
        if os.path.exists(out_path):
            os.remove(out_path)                 # parts never truncate: start from nothing
        if not keep_bp:
            measure_first_interval(plan, paths, **scan_kw)
    if not keep_bp:
        broadcast_rescale(plan, rank, 0, group, device)
    else:
        dist.barrier(group=group)               # nobody writes before the stale file is gone
    try:
        res = plan.run_scan(paths, out_path, part=(rank, world), **scan_kw)
    finally:
        plan.set_rescale(None)                  # the plan goes back to measuring: a later plain run_scan is a new scan
    dist.barrier(group=group)
    return res
