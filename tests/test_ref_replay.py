"""The restated HOST sequence of the reference step (oracle/ref_replay.py) driving the reference's own
kernels: on the CPU backend it must reproduce the golden vectors recorded from the unmodified
reference class exactly (same kernels, same order) -- this validates the GPU baseline harness
(same code, backend "gpu") that bench.py times as "B-ref"."""
import numpy as np
import pytest

from conftest import load_golden
from instagraal_b200.synth import WORKLOADS, make_level
from oracle import ref_kernels as rk
from parity_common import OracleTeacher, replay, score_tol


class ReplayImpl:
    def __init__(self, level, p8, backend):
        from oracle.ref_replay import RefReplaySampler
        if backend == "oracle":   # the reference's NumPy port, where its kernels are not built
            self.r = OracleTeacher(level, p8)
        else:
            self.r = RefReplaySampler(level, p8, backend=backend, canonical_slice_order=(backend == "gpu"))  # GPU: atomic order varies run to run

    def set_state(self, st):
        self.r.set_state(st)

    def set_valid(self, v):
        self.r.set_valid(v)

    def set_params(self, p8):
        self.r.set_params(p8)

    def get_state(self):
        return self.r.get_state()

    def step(self, a, cands):
        o, dist, op, b, ml, nc = self.r.step_sampler(a, cands)
        return dict(scores=self.r.all_scores, op=op, B=b, o=o, dist=dist, mean_len=ml, n_contigs=nc)


@pytest.mark.skipif(not rk.available(), reason="oracle/_ref/libref_cpu.so not built")
def test_replay_cpu_backend_matches_golden_exactly():
    g = load_golden("micro_bomb_seed1")
    level = make_level(WORKLOADS["micro"])
    impl = ReplayImpl(level, g["params8"], "cpu")
    res = replay(g, impl, max_steps=25, check_nuis=False)
    assert not res.errors, res.errors[:3]
    assert res.same_choice == res.steps  # identical kernels, identical order: no tie can break differently
    assert res.max_rel == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("d_exp", [None, 2.37])
def test_reference_kernels_on_gpu_vs_product(built, d_exp):
    """GPU-vs-GPU: the reference's own kernels (cubin) and the product agree on every score to 1e-9
    relative (same libdevice powf/log10) over a replayed trajectory.  Where the cubin is not built, the teacher is the
    reference's NumPy port and every score is held to parity_common.score_tol."""
    import os
    from oracle.ref_replay import _HERE
    kernels = os.path.exists(os.path.join(_HERE, "_ref", "ref_kernels.cubin"))
    from test_gpu_parity import GpuImpl
    g = load_golden("toy_bomb_seed2")
    level = make_level(WORKLOADS["toy"])
    ref = ReplayImpl(level, g["params8"], "gpu" if kernels else "oracle")
    mine = GpuImpl(level)
    worst = 0.0
    n = 60
    for t in range(n):
        nc = int(g["step_ncand"][t])
        cands = [int(c) for c in g["step_cands"][t][:nc]]
        st = g["state0"] if t == 0 else g["step_states"][t - 1]
        for impl in (ref, mine):
            impl.set_state(st)
            impl.set_valid(g["step_valid_before"][t])
            p8 = np.array(g["step_params_before"][t], dtype=np.float32)
            if d_exp is not None:
                p8[4] = d_exp   # expf branch of rippe_contacts
            impl.set_params(p8)
        a = ref.step(int(g["step_A"][t]), cands)
        b = mine.step(int(g["step_A"][t]), cands)
        sa, sb = np.asarray(a["scores"]), np.asarray(b["scores"])
        assert np.array_equal(sa != 0, sb != 0), t
        nz = sa != 0
        worst = max(worst, float(np.max(np.abs(sa[nz] - sb[nz]) / np.abs(sa[nz]))))
        if not kernels:
            assert np.all(np.abs(sa[nz] - sb[nz]) <= score_tol(sa[nz])), t
    assert worst < 1e-9 or not kernels, worst
    mine.s.free_gpu()
