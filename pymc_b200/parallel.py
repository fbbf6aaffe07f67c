"""Multi-GPU: chains are the unit of sharding (one process per GPU, torch.distributed for plumbing).

The reference never exchanges anything between NUTS chains (per-chain adaptation,
hmc/quadpotential.py:335-355; one OS process per chain, sampling/parallel.py:477-589), so the data path
has NO collective: rank r runs a contiguous block of chains with streams derived on every rank from the
same ``SeedSequence`` spawn (sampling/mcmc.py:907), which makes results independent of the number of
GPUs.  The only communication is the final gather of draws and sampler stats (all_gather over
NCCL/NVLink, or gloo on CPU in tests).
"""
from __future__ import annotations

import numpy as np


def _dist():
    try:
        import torch.distributed as dist
    except Exception:  # pragma: no cover
        return None
    return dist if dist.is_available() and dist.is_initialized() else None


def world_size() -> int:
    d = _dist()
    return d.get_world_size() if d else 1


def rank() -> int:
    d = _dist()
    return d.get_rank() if d else 0


def chain_range(chains: int, r: int, world: int) -> tuple[int, int]:
    """Contiguous block of chains owned by rank r: sizes differ by at most one."""
    base, extra = divmod(chains, world)
    lo = r * base + min(r, extra)
    return lo, lo + base + (1 if r < extra else 0)


def my_chain_range(chains: int) -> tuple[int, int]:
    return chain_range(chains, rank(), world_size())


def gather_chains(draws, stats: dict, chains: int, dst: int | None = 0):
    """Gather per-rank shards [c_r, T, ...] into [chains, T, ...] on rank ``dst`` (other ranks get ``(None, None)``);
    ``dst=None`` all-gathers to every rank (N x the traffic and memory: 24 GB per rank for the Radon bench at 8 GPUs --
    only when every rank really needs every draw).

    NCCL needs device tensors and equal shard shapes: shards are padded to the largest block."""
    import torch

    d = _dist()
    world = d.get_world_size()
    backend = d.get_backend()
    dev = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
    sizes = [chain_range(chains, r, world) for r in range(world)]
    cmax = max(hi - lo for lo, hi in sizes)

    def gather(a):
        was_np = isinstance(a, np.ndarray)
        t = torch.as_tensor(a).to(dev)
        if t.shape[0] < cmax:
            pad = torch.zeros((cmax - t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
            t = torch.cat([t, pad], dim=0)
        if dst is None:
            outs = [torch.empty_like(t) for _ in range(world)]
            d.all_gather(outs, t.contiguous())
        else:
            outs = [torch.empty_like(t) for _ in range(world)] if d.get_rank() == dst else None
            d.gather(t.contiguous(), outs, dst=dst)
            if outs is None:
                return None
        full = torch.cat([o[: hi - lo] for o, (lo, hi) in zip(outs, sizes)], dim=0)
        return full.cpu().numpy() if was_np else full

    g = gather(draws)
    st = {k: gather(v) for k, v in stats.items()}
    return (g, st) if g is not None else (None, None)


def max_over_ranks(x: float) -> float:
    """Device-side timing rule: a multi-GPU time is the max over ranks."""
    d = _dist()
    if not d:
        return x
    import torch

    dev = torch.device("cuda", torch.cuda.current_device()) if d.get_backend() == "nccl" else torch.device("cpu")
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    d.all_reduce(t, op=d.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x: float) -> float:
    d = _dist()
    if not d:
        return x
    import torch

    dev = torch.device("cuda", torch.cuda.current_device()) if d.get_backend() == "nccl" else torch.device("cpu")
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    d.all_reduce(t, op=d.ReduceOp.SUM)
    return float(t.item())


# ------------------------------------------------------------------------------------------------------------------------
# Pooled warm-up (north_star: "NCCL used only to gather draws and pooled warmup statistics at tuning-window boundaries").
# An OPT-IN extension: the reference adapts every chain's mass matrix from its own draws only (quadpotential.py:335-355).
# With thousands of chains the per-chain estimate (~100 draws per window) is the noisy part of warm-up and makes step sizes
# -- hence tree depths and run times -- differ between chains; pooling the Welford statistics of all chains (and all GPUs)
# at the window boundaries gives every chain the same, far better, estimate.
# ------------------------------------------------------------------------------------------------------------------------
def pool_welford(count, mean, m2):
    """Combine per-chain Welford triples (count[C], mean[C, n], m2[C, n]) over the chains of ALL ranks (Chan et al.):
    returns (N, mean[n], M2[n]).  One all-reduce of 2n + 1 doubles when torch.distributed is initialised."""
    count = np.asarray(count, dtype=np.float64)
    s0 = count.sum()
    s1 = (count[:, None] * mean).sum(axis=0)
    s2 = (m2 + count[:, None] * mean * mean).sum(axis=0)
    d = _dist()
    if d:
        import torch

        dev = torch.device("cuda", torch.cuda.current_device()) if d.get_backend() == "nccl" else torch.device("cpu")
        t = torch.as_tensor(np.concatenate([[s0], s1, s2]), device=dev)
        d.all_reduce(t, op=d.ReduceOp.SUM)
        t = t.cpu().numpy()
        n = len(s1)
        s0, s1, s2 = t[0], t[1 : 1 + n], t[1 + n :]
    mu = s1 / s0
    return float(s0), mu, s2 - s0 * mu * mu


def pooled_warmup_run(cm, q0, rng_states, *, tune, draws, mean0=None, window=101, discard_window=50, chain_offset=0,
                      philox_seed=0, **kw):
    """NUTS/HMC run whose diagonal mass matrix is adapted from the POOLED draws of all chains of all ranks.

    The tuning phase runs in slices that end at the reference's window boundaries (every ``window`` draws); inside a
    slice the kernel only accumulates the per-chain estimators (draws after ``discard_window``, like the reference); at a
    boundary the foreground estimators are pooled (``pool_welford``: one small all-reduce over NCCL), every chain's
    inverse mass becomes the pooled variance, and foreground <- background as in the reference.  Chains are carried
    between slices by ``engine.ChainState`` (the kernel continues them bit-exactly).  Returns the ``NutsResult`` of the
    sampling phase with ``summary['final_var']`` = the pooled mass matrix."""
    from . import engine

    q0 = np.ascontiguousarray(q0, dtype=np.float64)
    C, n = q0.shape
    never = 1 << 30  # no in-kernel refresh / estimator switch: the host does both at the boundaries
    common = dict(tune=tune, draws=draws, mass="diag_adapt", adaptation_window=never, discard_window=discard_window,
                  chain_offset=chain_offset, philox_seed=philox_seed, **kw)
    bounds = list(range(window + 1, tune, window)) + [tune] if tune > 0 else []
    state, begin = None, 0
    for b in bounds:
        nxt = engine.ChainState(C, n)
        cm.nuts_run(q0, rng_states, mean0=mean0, store_warmup=False, iter_begin=begin, iter_count=b - begin, resume=state,
                    save=nxt, stats=False, **common)
        state, begin = nxt, b
        if state.fg_n.min() > 0:
            N, mu, M2 = pool_welford(state.fg_n, state.fg_mean, state.fg_m2)
            state.var[:] = np.clip(M2 / N, 1e-12, 1e12)[None, :]
        # foreground <- background, background starts empty (QuadPotentialDiagAdapt.update, quadpotential.py:350-354)
        state.fg_n[:], state.fg_mean[:], state.fg_m2[:] = state.bg_n, state.bg_mean, state.bg_m2
        state.bg_n[:], state.bg_mean[:], state.bg_m2[:] = 0.0, 0.0, 0.0
    res = cm.nuts_run(q0, rng_states, mean0=mean0, store_warmup=False, iter_begin=begin, iter_count=tune + draws - begin,
                      resume=state, **common)
    return res


# ------------------------------------------------------------------------------------------------------------------------
# Host memory next to the GPU.  The sampling kernel writes draws straight into page-locked host memory (b200nuts.cu:
# stage_in, `direct`); on a two-socket box those writes cross the inter-socket link when the buffer was allocated on the
# other socket, and the kernel then runs at the speed of that link.  Page-locked allocations follow the allocating thread's
# NUMA policy, so binding the thread to the CPUs of the GPU's node WHILE the buffers are allocated is enough.
# ------------------------------------------------------------------------------------------------------------------------
def gpu_numa_cpus(device: int) -> tuple[int, set[int]]:
    """(NUMA node of the GPU or -1, the CPUs local to it -- empty when the platform does not say)."""
    import torch

    pr = torch.cuda.get_device_properties(device)
    try:
        dom, bus, dev = int(getattr(pr, "pci_domain_id", 0)), int(pr.pci_bus_id), int(pr.pci_device_id)
        base = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0"
        node = int(open(base + "/numa_node").read().strip())
        cpus: set[int] = set()
        for part in open(base + "/local_cpulist").read().strip().split(","):
            if not part:
                continue
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        return node, cpus
    except (OSError, ValueError, AttributeError):
        return -1, set()


class near_gpu:
    """``with near_gpu(device): allocate pinned buffers`` -- restricts the calling thread to the GPU-local CPUs for the
    duration (restored on exit); a no-op where the platform reports no locality or the local CPUs are outside the cgroup."""

    def __init__(self, device: int):
        self.device, self.saved, self.info = device, None, {"numa_node": -1, "bound": False}

    def __enter__(self):
        import os

        node, cpus = gpu_numa_cpus(self.device)
        self.info["numa_node"] = node
        try:
            cur = os.sched_getaffinity(0)
            want = cpus & cur
            if want and want != cur:
                self.saved = cur
                os.sched_setaffinity(0, want)
                self.info["bound"] = True
                self.info["cpus"] = len(want)
        except (AttributeError, OSError):
            pass
        return self

    def __exit__(self, *exc):
        import os

        if self.saved is not None:
            try:
                os.sched_setaffinity(0, self.saved)
            except OSError:
                pass
        return False
