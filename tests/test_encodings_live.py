"""The deterministic encoders (``single``, ``repeat``, ``rank_order``) and the ``Encoder`` wrappers against the
reference (encodings.py:6-47, 159-191; encoders.py; its outputs stored under tests/golden/live): equal outputs on the
same data; ``poisson(approx=True)`` draws from torch's generator like the reference, so the same seed gives the same
spikes.  CPU only."""
import pytest
import torch

from live import REF, stored


def _data(seed, shape=(1, 12, 12), zeros=0.3):
    g = torch.Generator().manual_seed(seed)
    x = 128.0 * torch.rand(*shape, generator=g)
    return x * (torch.rand(*shape, generator=g) > zeros)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("time,dt", [(50, 1.0), (40, 0.5), (7, 1.0)])
def test_rank_order_single_repeat_equal_the_live_reference(seed, time, dt):
    from bindsnet_b200 import encoding as E

    x = _data(seed)
    keep = x.clone()
    a = stored("rank_order", lambda: REF.encoding.rank_order(x.clone(), time=time, dt=dt))
    b = E.rank_order(x, time=time, dt=dt)
    assert a.dtype == b.dtype and torch.equal(a, b) and int(b.sum()) > 0
    assert torch.equal(x, keep)                                  # ours leaves the caller's tensor alone
    assert int(b.sum(0).max()) == 1                              # at most one spike per feature
    for sparsity in (0.5, 0.1):
        a = stored(f"single/{sparsity}", lambda: REF.encoding.single(x.clone(), time=time, dt=dt, sparsity=sparsity))
        b = E.single(x, time=time, dt=dt, sparsity=sparsity)
        assert a.dtype == b.dtype and torch.equal(a, b) and int(b[0].sum()) > 0 and int(b[1:].sum()) == 0
    assert torch.equal(stored("repeat", lambda: REF.encoding.repeat(x, time=time, dt=dt)), E.repeat(x, time=time, dt=dt))


def test_encoder_classes_equal_the_live_reference():
    from bindsnet_b200 import encoding as E

    x = _data(9)
    for name, kw in (("SingleEncoder", dict(sparsity=0.2)), ("RepeatEncoder", {}), ("RankOrderEncoder", {})):
        a = stored(name, lambda: getattr(REF.encoding, name)(time=30, dt=1.0, **kw)(x.clone()))
        b = getattr(E, name)(time=30, dt=1.0, **kw)(x.clone())
        assert torch.equal(a, b), name
    assert E.NullEncoder()(x) is x
    for name, kw in (("PoissonEncoder", dict(approx=True)), ("PoissonEncoder", {}), ("BernoulliEncoder", dict(max_prob=0.5))):
        torch.manual_seed(3)
        a = stored(f"{name}/{sorted(kw)}", lambda: getattr(REF.encoding, name)(time=25, dt=1.0, **kw)(x.clone()))
        torch.manual_seed(3)
        b = getattr(E, name)(time=25, dt=1.0, **kw)(x.clone())
        assert a.shape == b.shape and a.dtype == b.dtype, name
        if kw.get("approx"):
            assert torch.equal(a, b)                             # same generator, same operations
        else:
            assert abs(float(a.float().mean()) - float(b.float().mean())) < 0.02, name


def test_loaders_equal_the_live_reference():
    from bindsnet_b200 import encoding as E

    data = torch.stack([_data(s) for s in (4, 5, 6)])
    a = stored("rank_order_loader", lambda: list(REF.encoding.rank_order_loader(data.clone(), time=20, dt=1.0)))
    b = list(E.rank_order_loader(data, time=20, dt=1.0))
    assert len(a) == len(b) == 3 and all(torch.equal(x, y) for x, y in zip(a, b))
    for name in ("poisson_loader", "bernoulli_loader"):
        out = list(getattr(E, name)(data, time=15, dt=1.0))
        ref = stored(name, lambda: list(getattr(REF.encoding, name)(data.clone(), time=15, dt=1.0)))
        assert [o.shape for o in out] == [r.shape for r in ref] and out[0].dtype == ref[0].dtype == torch.uint8
