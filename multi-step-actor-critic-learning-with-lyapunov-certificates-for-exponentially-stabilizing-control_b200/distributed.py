"""Multi-GPU plumbing: env instances shard across ranks with NO collective on the step path
(every env is independent; RNG is keyed by the global env id, so results do not depend on the
number of GPUs).  Collectives (NCCL on GPUs, gloo in the CPU tests) are used only for the
per-chunk episode statistics and for assembling a global replay batch from per-rank
sub-batches (SURVEY.md section 8e).
"""
import struct

import torch
import torch.distributed as dist


def shard_env_range(total_envs, rank, world):
    """Contiguous env-id range [lo, hi) owned by `rank`; sizes differ by at most one."""
    base, rem = divmod(int(total_envs), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def all_reduce_stats(stats):
    """Sum the [8] float64 rollout statistics vector (episodes, sum return, sum length,
    terminated, truncated, ...) over ranks."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        stats = stats.clone()
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    return stats


def all_gather_replay_batch(sub_batch):
    """Concatenate per-rank replay sub-batches {field: [B/G, n, ...]} along the batch axis in
    rank order -> {field: [B, n, ...]} on every rank."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return sub_batch
    world = dist.get_world_size()
    out = {}
    for k in sorted(sub_batch):
        t = sub_batch[k].contiguous()
        full = torch.empty((world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(full, t)
        out[k] = full
    return out


def exchange_batch_and_stats(sub_batch, stats):
    """One collective per chunk instead of eight: the per-rank replay sub-batch {field: [B/G, n, ...]} (float32) and
    the [8] float64 statistics vector are packed into one buffer, all-gathered once, and unpacked into the global
    batch {field: [B, n, ...]} (rank order, as `all_gather_replay_batch`) and the rank-summed statistics (as
    `all_reduce_stats`; summed in rank order, so the result is identical on every rank).  NVSwitch makes the cost of
    these small exchanges launch latency, not bandwidth, hence the single bucket."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return sub_batch, stats
    world = dist.get_world_size()
    keys = sorted(sub_batch)
    parts = [sub_batch[k].contiguous().float().reshape(-1) for k in keys]
    st32 = stats.detach().to(torch.float64).contiguous().view(torch.float32)         # 8 doubles -> 16 floats, bit-exact
    packed = torch.cat(parts + [st32.to(parts[0].device)])
    flat = torch.empty(world * packed.numel(), dtype=torch.float32, device=packed.device)
    dist.all_gather_into_tensor(flat, packed)
    full = flat.view(world, packed.numel())
    out, off = {}, 0
    for k, p in zip(keys, parts):
        shape = tuple(sub_batch[k].shape)
        out[k] = full[:, off:off + p.numel()].reshape((world * shape[0],) + shape[1:])
        off += p.numel()
    stats_all = full[:, off:off + st32.numel()].contiguous().view(torch.float64)      # [world, 8]
    return out, stats_all.sum(dim=0)


class BatchExchange:
    """Per-chunk exchange of the replay sub-batches and the episode statistics, overlapped with the next rollout.

    One preallocated packed float32 buffer per rank holds the 7 batch fields ([B/G, n, .] each; `views()` hands them out
    so that the buffer's gather kernel writes the sampled windows straight into it -- no torch.cat) followed by the [8]
    float64 statistics bit-cast to 16 floats.  `exchange()` issues ONE all-gather of that buffer on a side stream and
    returns the result of the call `depth` calls earlier (default 1: the PREVIOUS call): the learner's batch is one iteration stale (as it already is in the
    reference loop, where the batch is drawn before the current chunk's windows matter), so the collective's latency hides
    behind the next rollout launch instead of blocking it.  Buffers are double-buffered; the first call returns its own
    result.  On CPU tensors (gloo tests) the same protocol runs synchronously."""

    def __init__(self, fields, sub_batch, n_step, device, group=None, depth=1):
        self.depth = max(1, int(depth))      # calls between issuing a gather and consuming it (1: next call; 2 absorbs rank skew)
        self.world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
        self.group, self.device = group, torch.device(device)
        self.keys = sorted(fields)
        self.shapes = {k: (int(sub_batch), int(n_step)) + tuple(fields[k]) for k in self.keys}
        self.offsets, off = {}, 0
        for k in self.keys:
            numel = 1
            for d in self.shapes[k]:
                numel *= d
            self.offsets[k] = (off, numel)
            off += (numel + 3) // 4 * 4                 # keep every field 16-byte aligned
        self.stats_off, self.P = off, off + 16
        self.nbuf = self.depth + 2                # one spare: a consumer may still be copying a returned buffer to the host
        self.send = [torch.zeros(self.P, dtype=torch.float32, device=self.device) for _ in range(self.nbuf)]
        self.recv = [torch.zeros(self.world, self.P, dtype=torch.float32, device=self.device) for _ in range(self.nbuf)]
        self.side = torch.cuda.Stream(self.device) if self.device.type == "cuda" else None
        self.done = [None] * self.nbuf
        self.reuse_guard = [None] * self.nbuf     # events a consumer recorded after reading recv[i] on ANOTHER stream (see guard_reuse)
        self.last_take = 0
        self.t = 0

    def views(self):
        """{field: [B/G, n, .]} views of the CURRENT send buffer: pass as `out=` to buffer.sample_batch."""
        buf = self.send[self.t % self.nbuf]
        return {k: buf[o:o + m].view(self.shapes[k]) for k, (o, m) in self.offsets.items()}

    def _unpack(self, recv):
        out = {}
        for k, (o, m) in self.offsets.items():
            shp = self.shapes[k]
            out[k] = recv[:, o:o + m].reshape((self.world * shp[0],) + shp[1:])
        stats = recv[:, self.stats_off:self.stats_off + 16].contiguous().view(torch.float64).sum(dim=0)    # rank order
        return out, stats

    def exchange(self, sub_batch, stats, unpack=True):
        """sub_batch: `views()` already filled by the gather kernel, or any {field: tensor} (copied in).  Returns the
        previous call's (global batch {field: [B, n, .]}, rank-summed statistics [8] float64) -- with unpack=False the raw
        gathered [G, P] buffer instead (one contiguous D2H copy; unpack on the host with `host_views`)."""
        cur = self.t % self.nbuf
        mine = self.views()
        for k in self.keys:
            if sub_batch[k].data_ptr() != mine[k].data_ptr():
                mine[k].copy_(sub_batch[k])
        self.send[cur][self.stats_off:].view(torch.float64).copy_(stats.detach().to(torch.float64))
        guard, self.reuse_guard[cur] = self.reuse_guard[cur], None
        if guard is not None:                         # recv[cur] is about to be overwritten: its last reader must be done
            (self.side if (self.side is not None and self.world > 1) else torch.cuda.current_stream()).wait_event(guard)
        if self.world == 1:
            self.recv[cur].copy_(self.send[cur][None])
        elif self.side is None:                       # CPU tensors (gloo), or in-stream on request
            dist.all_gather_into_tensor(self.recv[cur].view(-1), self.send[cur], group=self.group)
        else:
            ready = torch.cuda.Event()
            ready.record()
            self.side.wait_event(ready)
            with torch.cuda.stream(self.side):
                dist.all_gather_into_tensor(self.recv[cur].view(-1), self.send[cur], group=self.group)
                ev = torch.cuda.Event()
                ev.record()
            self.done[cur] = ev
        take = (self.t - min(self.t, self.depth)) % self.nbuf      # the first `depth` calls return the oldest result there is
        if self.side is not None and self.done[take] is not None:
            torch.cuda.current_stream().wait_event(self.done[take])
        self.t += 1
        self.last_take = take
        return self._unpack(self.recv[take]) if unpack else self.recv[take]

    def guard_reuse(self, event):
        """`event` (recorded on whatever stream reads the buffer the last exchange() returned, e.g. a D2H copy stream) must
        complete before that buffer is gathered into again."""
        self.reuse_guard[self.last_take] = event

    def host_views(self, host_packed):
        """Unpack a host copy [G, P] of a gathered buffer: ({field: [B, n, .]}, statistics [8] float64); the batch fields are
        strided views when G > 1 (rank-major rows), plain views when G == 1."""
        return self._unpack(host_packed)


def broadcast_parameters(module_or_tensors, src=0):
    """Learner -> rollout ranks: broadcast a module's parameters (e.g. `networks.policy`, 285 KB) from rank `src`
    in ONE collective (flattened bucket) and copy them back in place, so that every rank samples with the same actor."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    tensors = [p.data for p in module_or_tensors.parameters()] if hasattr(module_or_tensors, "parameters") else list(module_or_tensors)
    flat = torch.cat([t.reshape(-1) for t in tensors])
    dist.broadcast(flat, src=src)
    off = 0
    for t in tensors:
        t.copy_(flat[off:off + t.numel()].view_as(t))
        off += t.numel()


def mean_std_over_ranks(*per_instance):
    """Mean and population std of per-instance values whose instances are sharded over ranks (evaluator: one value per
    evaluation episode).  One all-reduce of the float64 moments [N, sum x_j, sum x_j^2 ...]; single-process: two-pass
    torch mean/std.  Returns [(mean, std), ...] as Python floats, identical on every rank."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return [(float(x.mean()), float(x.std(unbiased=False))) for x in per_instance]
    dev = per_instance[0].device
    m = [torch.tensor(float(per_instance[0].numel()), dtype=torch.float64, device=dev)]
    for x in per_instance:
        x = x.double()
        m += [x.sum(), (x * x).sum()]
    m = torch.stack(m)
    dist.all_reduce(m, op=dist.ReduceOp.SUM)
    n = m[0]
    out = []
    for j in range(len(per_instance)):
        mean = m[1 + 2 * j] / n
        var = torch.clamp(m[2 + 2 * j] / n - mean * mean, min=0.0)
        out.append((float(mean), float(var.sqrt())))
    return out


def episode_summary(stats):
    """Host dict from a (reduced) statistics vector."""
    s = stats.detach().cpu().tolist()
    ep = max(s[0], 1.0)
    return {"episodes": int(s[0]), "mean_return": s[1] / ep, "mean_length": s[2] / ep, "terminated": int(s[3]),
            "truncated": int(s[4])}


def float_order_key(x):
    """Order-preserving uint32 key of a float32 (as the certificate verifier's atomicMin uses): bits | 0x80000000 for sign 0,
    ~bits for sign 1.  Returns a Python int."""
    b = struct.unpack("<I", struct.pack("<f", float(x)))[0]
    return (~b & 0xFFFFFFFF) if b & 0x80000000 else (b | 0x80000000)


def float_from_order_key(key):
    """Inverse of `float_order_key`."""
    key = int(key) & 0xFFFFFFFF
    b = (key & 0x7FFFFFFF) if key & 0x80000000 else (~key & 0xFFFFFFFF)
    return struct.unpack("<f", struct.pack("<I", b))[0]


CERT_CSTAR_KEY, CERT_ROA = 9, 10        # MSACL_CERT_SUM_CSTAR_KEY / MSACL_CERT_SUM_ROA of include/msacl_b200.h


def combine_certificate(summary, count_below):
    """Combine the per-rank certificate summaries (int64 [11 + horizon], layout MSACL_CERT_SUM_* of include/msacl_b200.h) of
    states sharded over ranks: counters and histogram are summed, the c_star key is all-reduced with MIN, and then
    `count_below(c_star)` -- this rank's #{i : V_0,i < c_star} -- is summed into the ROA slot.  Returns (summary, c_star) with
    the same values on every rank; single process: the local summary with its own c_star."""
    s = summary.detach().to(torch.int64).clone()
    key = s[CERT_CSTAR_KEY:CERT_CSTAR_KEY + 1].clone()
    s[CERT_CSTAR_KEY] = 0
    s[CERT_ROA] = 0
    sharded = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    if sharded:
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
        dist.all_reduce(key, op=dist.ReduceOp.MIN)
    c_star = float_from_order_key(int(key.item()))
    roa = torch.tensor([int(count_below(c_star))], dtype=torch.int64, device=s.device)
    if sharded:
        dist.all_reduce(roa, op=dist.ReduceOp.SUM)
    s[CERT_CSTAR_KEY] = key[0]
    s[CERT_ROA] = roa[0]
    return s, c_star
