"""run.plan_step: every decision of a dense step, field by field, for a cut without virtual gates (syc-32 d1) and two
with (hwe-16 d5, syc-16 d5), exact and at ACCURACY = 1e-5, on one, two and four ranks, with the label-sharding
threshold (dist.SHARD_MIN_WORK) on either side of the cut's simulation work.  Host only: no device is touched."""
import dataclasses
from importlib import import_module

import pytest

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
cutting = import_module(f"{PKG}.cutting")
vcm = import_module(f"{PKG}.virtual_circuit")
runm = import_module(f"{PKG}.run")
qdist = import_module(f"{PKG}.dist")

# cut -> (K, labels, innermost radix, output bits)
CUTS = {"syc32d1": (0, 1, None, 32), "hwe16d5": (5, 7776, 6, 16), "syc16d5": (4, 1296, 6, 16)}


def _expected(cfg: str, accuracy: float, rank: int, world: int, sharded_labels: bool) -> dict:
    """The plan of one case, written out from the rules in ``run.plan_step`` and ``dist.py``."""
    K, L, radix, n_out = CUTS[cfg]
    faithful = accuracy > 0.0
    want = dict(K=K, faithful=faithful, fold=not faithful, union=(1 << n_out) - 1, n_out=n_out, mode="single",
                label_range=None, y_range=None, part=(0, 1), collective=None, knit_stats=K == 0 and not faithful,
                accuracy=accuracy if faithful else 0.0)
    if world == 1:
        return want
    if K == 0 and faithful:                  # the full output on every rank (no y_range), nothing exchanged
        want["mode"] = "replicated"
    elif K == 0:
        span = (1 << n_out) // world
        want.update(mode="output index by top bits", y_range=(rank * span, (rank + 1) * span),
                    collective="allreduce_stats")
    elif faithful:
        want.update(mode="output entries + all-reduce", part=(rank, world), collective="allreduce_sum")
    elif sharded_labels:
        want.update(mode="label range + all-reduce", collective="allreduce_sum",
                    label_range=qdist.shard_range(L, rank, world, align=radix))
    else:
        want["mode"] = "replicated (below the sharding threshold)"
    return want


@pytest.mark.parametrize("cfg", list(CUTS))
def test_plan_step_fields(cfg, monkeypatch):
    circ, cut = cutting.make_baseline(cfg, seed=0)
    virt = vcm.VirtualCircuit(cut)
    work = qdist.simulation_work(virt)
    assert work > 0.0
    K, L, radix, n_out = CUTS[cfg]
    assert len(virt.vgates) == K and virt.num_global_labels() == L
    assert (virt.global_radices()[-1] if K else None) == radix
    for min_work, sharded_labels in ((work * 2.0, False), (work / 2.0, True)):
        monkeypatch.setattr(qdist, "SHARD_MIN_WORK", min_work)
        for accuracy in (0.0, 1e-5):
            for world in (1, 2, 4):
                for rank in sorted({0, world - 1}):
                    plan = runm.plan_step(virt, rank, world, accuracy)
                    got = dataclasses.asdict(plan)
                    want = _expected(cfg, accuracy, rank, world, sharded_labels)
                    assert got == want, (cfg, accuracy, world, rank, min_work)
                    if plan.label_range is not None:
                        lo, hi = plan.label_range
                        assert lo % radix == 0 and (hi % radix == 0 or hi == L)
                        assert (rank != 0 or lo == 0) and (rank != world - 1 or hi == L)
    with pytest.raises(dataclasses.FrozenInstanceError):
        plan.mode = "single"

