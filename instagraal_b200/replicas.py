"""Replica chains (SURVEY section 8e: a single chain is sequential, so the only natural sharding of the 8 x B200 box is
independent chains with different seeds, one or more per GPU).

``ReplicaSet`` owns the chains of ONE process / GPU: the first one is a normal ``sampler`` (uploads the level), the others
are ``ig_clone``s that share its contacts in device memory.  ``run_cycle`` advances all of them together
(``ig_run_cycles_device_multi``: steps enqueued round-robin on the chains' streams, so a GPU that one yeast-scale chain
keeps < 25 % busy is filled by eight); ``allgather`` is the per-cycle exchange of {likelihood, n_contigs, p(s) parameters,
validity list, live scaffold} across the GPUs: ``ncclAllGather`` INSIDE the library, straight from device memory over NVLink
(``ig_allgather_best``).  ``adopt`` / ``exchange`` restart every chain from the gathered best one on the device
(``ig_adopt_gathered``), so the set searches as one population instead of N unrelated runs.
No PyTorch here: the launcher only has to hand every rank the 128-byte NCCL id created by rank 0
(``nccl_unique_id`` -> file / environment / any broadcast).
The live path of the reference has no temperature (fragment moves are an argmax, CL:1435-1446): by default the chains differ
by their seeds only, and every rank takes the same decision (best chain) from the gathered table.

Tempering (DESIGN.md 4e, 6b): ``set_ladder`` gives every chain of the whole set a temperature (``sampler.set_chain_temperature``;
T = 0 is the argmax, a hot chain also takes worse moves), and ``swap_temperatures`` exchanges the temperatures of adjacent
rungs after a gather with the replica-exchange rule, decided identically on every rank (``swap_decisions``).  Temperatures
move and scaffolds stay, so a swap copies nothing on the device.  Like the seeds, the ladder is a run setting: checkpoints do
not hold it.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L


def best_chain(likelihoods):
    """Deterministic on every rank: highest likelihood, lowest global chain index on ties (what ig_allgather_best returns)."""
    lik = np.asarray(likelihoods, dtype=np.float64)
    return int(np.flatnonzero(lik == lik.max())[0])


def swap_decisions(temperatures, ladder, likelihoods, round_index, swap_seed=0):
    """One round of temperature swaps between adjacent rungs; a pure function, so every rank decides the same.

    temperatures[k] = the temperature of rung k, ladder[k] = the global chain at rung k, likelihoods[g] = the live
    log-likelihood of global chain g.  Round r tries the pairs (k, k + 1) with k = r (mod 2), with the uniforms of
    np.random.default_rng([swap_seed, r]) (uniform k for pair k), and accepts with probability
    min(1, exp((beta_k - beta_k+1) (L_k+1 - L_k))), beta = 1 / T.  A rung at T = 0 takes the limit: the swap is accepted iff
    it does not lower the likelihood the colder rung holds (ties accepted); two rungs at T = 0 always swap.
    -> (pairs tried, pairs accepted, new ladder)."""
    T = np.asarray(temperatures, dtype=np.float64)
    lad = np.array(ladder, dtype=np.int64)
    lik = np.asarray(likelihoods, dtype=np.float64)
    u = np.random.default_rng([int(swap_seed), int(round_index)]).random(max(len(T) - 1, 0))
    tried, accepted = [], []
    for k in range(int(round_index) % 2, len(T) - 1, 2):
        tried.append((k, k + 1))
        t0, t1 = T[k], T[k + 1]
        l0, l1 = lik[lad[k]], lik[lad[k + 1]]
        if t0 == 0.0 and t1 == 0.0:
            ok = True
        elif t0 == 0.0 or t1 == 0.0:
            ok = (l1 >= l0) if t0 == 0.0 else (l0 >= l1)   # the colder rung would then hold the other chain's likelihood
        else:
            log_a = (1.0 / t0 - 1.0 / t1) * (l1 - l0)
            ok = bool(log_a >= 0.0 or u[k] < np.exp(log_a))
        if ok:
            accepted.append((k, k + 1))
            lad[k], lad[k + 1] = lad[k + 1], lad[k]
    return tried, accepted, lad


def nccl_unique_id():
    """128-byte id for ncclCommInitRank (call on rank 0, distribute to the other ranks)."""
    buf = (C.c_char * 128)()
    L.check(None, L.lib().ig_nccl_unique_id(buf), "ig_nccl_unique_id")
    return bytes(buf)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class ReplicaSet:
    def __init__(self, first_sampler, n_chains, seeds=None):
        """first_sampler: a constructed ``sampler`` (parameters already set); n_chains - 1 clones are made from it."""
        from .cuda_lib_gl_single import sampler
        self.chains = [first_sampler] + [sampler.clone_of(first_sampler) for _ in range(n_chains - 1)]
        self.n = n_chains
        self.seeds = np.ascontiguousarray(seeds if seeds is not None else np.arange(n_chains), dtype=np.uint64)
        self._handles = (C.c_void_p * n_chains)(*[c._h for c in self.chains])
        self.rank, self.n_ranks = 0, 1
        self._nccl = False
        self.nf = int(first_sampler.n_new_frags)
        self.gather_ms = 0.0
        self.n_gathers = 0
        self._gathered_nc = None   # n_contigs of every chain in the last all-gather
        self.temperatures = None   # set_ladder: temperature of every rung of the whole set, the chain at every rung
        self.ladder = None
        self.swap_seed = 0
        self.swap_round = 0
        self.swap_stats = None
        # several chains on this GPU: each takes a share of the SMs so that their (latency-bound) kernels overlap
        self.gpu_share = min(n_chains, 4)
        for c in self.chains:
            c.set_gpu_share(self.gpu_share)

    def init_comm(self, rank=0, n_ranks=1, nccl_id=None):
        lead = self.chains[0]
        idbuf = C.create_string_buffer(nccl_id, 128) if nccl_id is not None else None
        L.check(lead._h, L.lib().ig_nccl_init(lead._h, int(rank), int(n_ranks), self.n, idbuf), "ig_nccl_init")
        self.rank, self.n_ranks, self._nccl = int(rank), int(n_ranks), True

    def bomb(self, seed0=0):
        for i, c in enumerate(self.chains):
            np.random.seed(int(seed0) + i)
            c.bomb_the_genome()

    def run_cycle(self, frags_per_chain, n_neighbours=5, cycle=0, nuisance=False):
        """frags_per_chain: int32[n_chains, n_steps] visiting orders, n_neighbours <= IG_MAX_NEIGHBOURS (64).  Returns the structured per-step records
        [n_chains, n_steps] (same fields as sampler.run_cycle_device).  nuisance=True: every chain samples the p(s)
        parameters after every step, on the device with its own seed (sampler.run_cycle_device(nuisance=True)); returns
        (steps, nuis) with nuis [n_chains, n_steps] of sampler.NUIS_STEP_DTYPE."""
        frags = np.ascontiguousarray(frags_per_chain, dtype=np.int32)
        assert frags.ndim == 2 and frags.shape[0] == self.n
        for c in self.chains:
            c._upload_neighbour_weights()
            c.set_device_nuisance(nuisance)
        n_steps = frags.shape[1]
        out = np.zeros((self.n, n_steps), dtype=L.CYCLE_DTYPE)
        rc = L.lib().ig_run_cycles_device_multi(self._handles, self.n, n_steps, _ptr(frags), int(n_neighbours), _ptr(self.seeds),
                                                int(cycle), _ptr(out))
        L.check(None, rc, "ig_run_cycles_device_multi")
        for i, c in enumerate(self.chains):
            c._after_cycle(out[i], max(L.IG_MAX_CANDS, int(n_neighbours)))
        if not nuisance:
            return out
        return out, np.stack([c._after_nuisance(n_steps) for c in self.chains])

    def allgather(self):
        """-> (best global chain index, likelihood[n_ranks * n], n_contigs[n_ranks * n]); device ms accumulated in gather_ms"""
        if not self._nccl:
            self.init_comm()
        n_all = self.n_ranks * self.n
        lik = np.zeros(n_all, dtype=np.float64)
        nc = np.zeros(n_all, dtype=np.int32)
        best, ms = C.c_int32(0), C.c_float(0.0)
        lead = self.chains[0]
        L.check(lead._h, L.lib().ig_allgather_best(lead._h, self._handles, self.n, _ptr(lik), _ptr(nc), C.byref(best), C.byref(ms)),
                "ig_allgather_best")
        self.gather_ms += float(ms.value)
        self.n_gathers += 1
        self._gathered_nc = nc
        return int(best.value), lik, nc

    def adopt(self, index):
        """Every local chain other than global chain ``index`` restarts from that chain's state in the last all-gather, on the
        device (ig_adopt_gathered): scaffold, p(s) parameters and validity list; each keeps its own seed, and its next step
        is a full refresh.  Chain ``index``, if it is local, is not touched.  -> (p8, valid, likelihood) of chain ``index``."""
        from .cuda_lib_gl_single import PARAM_SIMU_RIPPE
        p8 = np.zeros(8, dtype=np.float32)
        valid = np.zeros(12, dtype=np.int32)
        lik = C.c_double(0.0)
        lead = self.chains[0]
        L.check(lead._h, L.lib().ig_adopt_gathered(lead._h, self._handles, self.n, int(index), _ptr(p8), _ptr(valid), C.byref(lik)),
                "ig_adopt_gathered")
        for c, ch in enumerate(self.chains):
            if self.rank * self.n + c == int(index):
                continue
            ch.param_simu = np.array([tuple(p8.tolist())], dtype=PARAM_SIMU_RIPPE)
            ch.param_simu_test = ch.param_simu
            ch.likelihood_t = ch.o = np.float64(lik.value)
            ch.n_contigs = np.int32(self._gathered_nc[int(index)])
        return p8, valid, float(lik.value)

    def exchange(self):
        """allgather() followed by adopt(best): every chain continues from the best chain of the whole set.
        -> (best, likelihood[n_ranks * n], n_contigs[n_ranks * n]) as allgather returns them."""
        best, lik, nc = self.allgather()
        self.adopt(best)
        return best, lik, nc

    def gathered_live_likelihood(self):
        """the live log-likelihood (likelihood_t) of every chain [n_ranks * n] in the last all-gather"""
        out = np.zeros(self.n_ranks * self.n, dtype=np.float64)
        lead = self.chains[0]
        L.check(lead._h, L.lib().ig_get_gathered_live_likelihood(lead._h, _ptr(out)), "ig_get_gathered_live_likelihood")
        return out

    def set_ladder(self, temperatures, swap_seed=0):
        """The temperatures of the whole set's n_ranks * n rungs, assigned rank-major at first (global chain g at rung g);
        every rank passes the same list.  Resets the swap rounds and swap_stats (tried / accepted per adjacent rung pair)."""
        T = np.array(temperatures, dtype=np.float64)
        if T.shape != (self.n_ranks * self.n,):
            raise ValueError("set_ladder: %d temperatures for %d chains" % (T.size, self.n_ranks * self.n))
        if not np.all(np.isfinite(T)) or np.any(T < 0):
            raise ValueError("set_ladder: temperatures must be finite and >= 0")
        self.temperatures, self.ladder = T, np.arange(T.size, dtype=np.int64)
        self.swap_seed, self.swap_round = int(swap_seed), 0
        self.swap_stats = {"tried": np.zeros(max(T.size - 1, 0), np.int64), "accepted": np.zeros(max(T.size - 1, 0), np.int64)}
        self._apply_ladder()

    def _apply_ladder(self):
        rung = np.empty_like(self.ladder)
        rung[self.ladder] = np.arange(self.ladder.size)
        for c, ch in enumerate(self.chains):
            T = float(self.temperatures[rung[self.rank * self.n + c]])
            if T != ch.chain_temperature:
                ch.set_chain_temperature(T)

    def swap_temperatures(self):
        """One all-gather, then one round of swap_decisions on the gathered live likelihoods; the local chains take their
        rungs' new temperatures.  -> (pairs tried, pairs accepted, ladder: rung -> global chain)."""
        if self.ladder is None:
            raise RuntimeError("swap_temperatures: no ladder (set_ladder)")
        self.allgather()
        lik = self.gathered_live_likelihood()
        tried, accepted, self.ladder = swap_decisions(self.temperatures, self.ladder, lik, self.swap_round, self.swap_seed)
        for k, _ in tried:
            self.swap_stats["tried"][k] += 1
        for k, _ in accepted:
            self.swap_stats["accepted"][k] += 1
        self.swap_round += 1
        self._apply_ladder()
        return tried, accepted, self.ladder.copy()

    def gathered_state(self, index):
        out = np.zeros((13, self.nf), dtype=np.int32)
        lead = self.chains[0]
        L.check(lead._h, L.lib().ig_get_gathered_state(lead._h, int(index), _ptr(out)), "ig_get_gathered_state")
        return out

    def free(self):
        for c in reversed(self.chains):
            c.free_gpu()
