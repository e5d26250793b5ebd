"""Chain sharding for the multi-GPU SAPG run (SURVEY.md section 8e).

One process per GPU.  `total_chains` independent MYULA chains are split into
contiguous blocks, rank r owning chains [r*n_local, (r+1)*n_local).  At every
outer iteration each rank contributes the per-chain sums of its chains; all
ranks receive all of them IN GLOBAL CHAIN ORDER and reduce them in that fixed
order, so the theta / sigma^2 / PSF-parameter updates are bit-identical on every
rank and independent of the number of GPUs.  This generalises the reference's
size-1 mini-batch average `G_b = mean(g_b)` (SAPG_algorithm_moffat.m:170-173).

On the GPU the exchange is an ncclAllGather enqueued on the compute stream by
libsbd (`sbd_comm_init`); this module holds the host-side logic - the
partition, the NCCL unique-id rendezvous through torch.distributed, and the
same gather-in-chain-order combine for CPU (gloo) tests.
"""
import ctypes as C

import numpy as np

from ._lib import lib, SbdError, SBD_NCCL_ID_BYTES


class ChainShard:
    def __init__(self, total_chains, world_size=1, rank=0):
        if total_chains % world_size != 0:
            raise ValueError("total_chains must be a multiple of world_size (equal shards)")
        self.total_chains, self.world_size, self.rank = int(total_chains), int(world_size), int(rank)
        self.n_local = self.total_chains // self.world_size
        self.chain_offset = self.rank * self.n_local

    def local_chains(self):
        return range(self.chain_offset, self.chain_offset + self.n_local)

    def owner(self, chain):
        return chain // self.n_local

    # -- rendezvous ---------------------------------------------------------
    def init_engine_comm(self, engine):
        """Create the NCCL communicator inside libsbd for this rank.  The unique
        id is generated on rank 0 and broadcast with torch.distributed."""
        if self.world_size == 1:
            return
        import torch
        import torch.distributed as dist
        buf = C.create_string_buffer(SBD_NCCL_ID_BYTES)
        if self.rank == 0:
            rc = lib.sbd_comm_unique_id(buf)
            if rc != 0:
                raise SbdError(rc, lib.sbd_last_error(None).decode())
        t = torch.tensor(list(buf.raw), dtype=torch.uint8)
        if dist.get_backend() == "nccl":
            t = t.cuda()
        dist.broadcast(t, src=0)
        raw = bytes(t.cpu().tolist())
        rc = lib.sbd_comm_init(engine._h, self.world_size, self.rank, raw)
        if rc != 0:
            raise SbdError(rc, lib.sbd_last_error(engine._h).decode())

    # -- host-side combine (same semantics as the device all-gather) -------
    def combine(self, local_vectors):
        """local_vectors: list (length n_local) of equal-length 1-D arrays, one
        per local chain.  Returns the sum over ALL chains, accumulated in global
        chain order."""
        local = np.stack([np.asarray(v, dtype=np.float64) for v in local_vectors], 0)
        if self.world_size == 1:
            allv = local
        else:
            import torch
            import torch.distributed as dist
            mine = torch.from_numpy(np.ascontiguousarray(local))
            parts = [torch.empty_like(mine) for _ in range(self.world_size)]
            dist.all_gather(parts, mine)
            allv = torch.cat(parts, 0).numpy()
        tot = np.zeros(allv.shape[1])
        for ch in range(allv.shape[0]):          # fixed order
            tot = tot + allv[ch]
        return tot

    def combine_posterior(self, stats):
        """Merge the posterior statistics of every rank's chains (Engine.sapg(..., post_levels=L)["posterior"]: one
        dict per block size with scale, n, chains, mean, within, between) into those of all chains.  Each rank's
        (C_r, mean_r, within_r, between_r) is all-gathered and merged in rank order:
            mean = sum_r C_r mean_r / C,  within = sum_r within_r,  between = sum_r [between_r + C_r (mean_r - mean)^2]
        This is exact algebra, but it sums in another order than one context running all C chains, so the result
        equals a one-GPU run to rounding (~1e-13 relative), not bit for bit.  Returns the same list of dicts with
        var, std and Rhat recomputed from the merged statistics.
        With the diagnostics (Engine.sapg(..., post_batch=b)) the batch statistics are merged the same way with
        weights C_r and the half statistics with weights 2 C_r, and ESS, MCSE and Rhat_split are recomputed; the
        ranks must agree in n, batch_len and n_batches.
        Quantiles (Engine.sapg(..., post_ci=alpha)) do not merge: each rank's P^2 markers summarise the stream of its
        own chains, and marker states of different streams give no estimator of the pooled one.  One rank passes them
        through; with more than one, results that carry them raise ValueError on every rank."""
        from .host import posterior_moments, posterior_diagnostics
        out = []
        for st in stats:
            diag = "batch_mean" in st
            keys = ("mean", "within", "between") + (DIAG_KEYS if diag else ())
            local = np.stack([np.asarray(st[k], dtype=np.float64) for k in keys])
            quant = "median" in st
            meta = [int(st["chains"]), int(st["n"]), int(diag)]
            if diag:
                meta += [int(st["batch_len"]), int(st["n_batches"]), int(st["half_n"])]
            if self.world_size == 1:
                parts, metas = [local], [meta]
            else:
                import torch
                import torch.distributed as dist
                mt = torch.tensor(meta + [0] * (6 - len(meta)) + [int(quant)], dtype=torch.int64)
                mts = [torch.empty_like(mt) for _ in range(self.world_size)]
                dist.all_gather(mts, mt)
                metas = [[int(v) for v in m] for m in mts]
                if any(m[6] for m in metas):
                    raise ValueError("combine_posterior: posterior quantiles (post_ci) cannot be merged across ranks: "
                                     "the P^2 markers of each rank's chains give no estimator of the pooled stream; "
                                     "hold all chains on one context (one rank) to get credible intervals")
                if len({m[2] for m in metas}) != 1:
                    raise ValueError("combine_posterior: some ranks have diagnostics and some do not")
                mine = torch.from_numpy(np.ascontiguousarray(local))
                gathered = [torch.empty_like(mine) for _ in range(self.world_size)]
                dist.all_gather(gathered, mine)
                parts = [g.numpy() for g in gathered]
            counts = [m[0] for m in metas]
            ns = [m[1] for m in metas]
            if len(set(ns)) != 1:
                raise ValueError(f"combine_posterior: ranks differ in samples per chain {ns}")
            C_ = sum(counts)
            m, within, between = _merge(counts, [p[0:3] for p in parts])
            var, std, rhat = posterior_moments(m, within, between, ns[0], C_)
            d = dict(scale=st["scale"], n=ns[0], chains=C_, mean=m, within=within, between=between, var=var,
                     std=std, Rhat=rhat)
            if diag:
                bs = {tuple(mm[3:6]) for mm in metas}
                if len(bs) != 1:
                    raise ValueError(f"combine_posterior: ranks differ in (batch_len, n_batches, half_n) {sorted(bs)}")
                b, B, h = bs.pop()
                merged = _merge(counts, [p[3:6] for p in parts]) + _merge([2 * c for c in counts], [p[6:9] for p in parts])
                d.update(zip(DIAG_KEYS, merged))
                d.update(batch_len=b, n_batches=B, half_n=h)
                d["ESS"], d["MCSE"], d["Rhat_split"] = posterior_diagnostics(
                    var, d["batch_within"], d["batch_between"], d["half_within"], d["half_between"], ns[0], C_, b, B, h)
            if quant:                           # one rank (more were refused above)
                d.update({k: st[k] for k in QUANT_KEYS})
            out.append(d)
        return out


DIAG_KEYS = ("batch_mean", "batch_within", "batch_between", "half_mean", "half_within", "half_between")
QUANT_KEYS = ("ci_alpha", "ci_count", "lower", "median", "upper", "ci_width")


def _merge(counts, parts):
    """(mean, within, between) of groups of counts[r] members each, from their own (mean_r, within_r, between_r),
    summed in rank order"""
    tot = np.zeros_like(parts[0][0])
    for cr, pr in zip(counts, parts):
        tot = tot + cr * pr[0]
    m = tot / sum(counts)
    within = np.zeros_like(m)
    between = np.zeros_like(m)
    for cr, pr in zip(counts, parts):
        within = within + pr[1]
        between = between + (pr[2] + cr * (pr[0] - m) ** 2)
    return m, within, between
