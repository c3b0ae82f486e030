"""TEST INFRASTRUCTURE ONLY — CPU oracle for the CFM/DiT hot path.

Nothing under ``oracle/`` is product code.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs may import it, and there only as the checker / reported CPU
baseline — never as the thing measured or shipped.  The product path
(``stabletts_b200``) never imports this package and fails loudly when its CUDA
library is missing.

Parity pinning: the restatement in ``estimator_ref.py`` is checked against
the committed fixtures under ``tests/golden/``, produced by
``oracle/make_golden.py`` and ``oracle/make_golden_modules.py`` from the
unmodified reference's own ``models.estimator.Decoder``.  The ODE
stepping arithmetic belongs to the third-party ``torchdiffeq`` (unpinned in the
reference's requirements.txt:14, absent here): fixed-grid tableaux are restated
from the published algorithm — "parity unpinned" for solver behaviour.
"""


def usable_cpus() -> int:
    """Host threads actually usable: min(affinity mask, cgroup CPU quota).  The GPU boxes report 128 CPUs
    under a 16-CPU cgroup quota; torch's default of 128 intra-op threads there slows the oracle ~50x."""
    import os
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def _limit_threads() -> None:
    try:
        import torch
        if torch.get_num_threads() > usable_cpus():
            torch.set_num_threads(usable_cpus())
    except Exception:
        pass


_limit_threads()
