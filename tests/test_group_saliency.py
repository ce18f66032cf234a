"""Group saliency maps on the host: the batching of ``cgcnn.saliency``, ``graph_saliency`` and ``adjacency_saliency``
with ``groups``, with the three gradient schedules replaced by fakes that return known per-window values and sum them
per group as the device does.  Checks the batch-local ids, the padding rows, the float64 accumulation in batch order,
the return shapes and counts, ``groups="target"`` and every refusal.  The device side is in
``test_gpu_group_saliency.py``."""
import numpy as np
import pytest
import scipy.sparse as sp

torch = pytest.importorskip("torch")

C_ = 5  # classes of the test network
BS = 16


def _per_window(x, width):
    """Known per-window values: a [B, width] float32 matrix that depends on each window only."""
    base = x.reshape(x.shape[0], -1)[:, :1].to(torch.float64)
    return (base * torch.linspace(-1.0, 1.0, width, dtype=torch.float64) + base ** 2).to(torch.float32)


def _target_of(x, t):
    return t if t is not None else (x[:, 0, 0].abs() * 100).long() % C_


class _Fake:
    """Records every call; grouped calls sum the per-window values per group in row order (float32), fill the rows of
    absent groups with NaN (the host must not read them) and zero them when grouped by target."""

    calls = []

    def __init__(self, model, *args, **kw):
        self.model = model

    def _values(self, x):
        raise NotImplementedError

    def __call__(self, x, target=None, gather=False, valid=None, absolute=False, group=None, n_groups=None):
        B = x.shape[0]
        valid = B if valid is None else valid
        t = _target_of(x, target)
        vals = self._values(x)
        _Fake.calls.append(dict(group=None if group is None or isinstance(group, str) else group.clone(),
                                mode=group if isinstance(group, str) else None, n_groups=n_groups, valid=valid))
        if group is None:
            return self._ungrouped(vals, valid, absolute), None, t
        if isinstance(group, str):
            assert group == "target"
            n_groups = C_
            group = torch.where(torch.arange(B) < valid, t, torch.full_like(t, -1)).to(torch.int32)
        assert group.dtype == torch.int32 and group.shape == (B,)
        outs = []
        for v in vals:
            out = torch.full((n_groups, v.shape[1]), float("nan"))
            if isinstance(self.calls[-1]["mode"], str):
                out.zero_()
            for g in range(n_groups):
                rows = (group == g).nonzero().flatten()
                if len(rows):
                    acc = torch.zeros(v.shape[1])
                    for r in rows:
                        acc += v[r].abs() if absolute else v[r]
                    out[g] = acc
            outs.append(out)
        return self._pack(outs, x), None, t


class FakeInputGradient(_Fake):
    def _values(self, x):
        return [_per_window(x, x[0].numel())]

    def _ungrouped(self, vals, valid, absolute):
        return vals[0].view(-1, *self.model._xshape)

    def _pack(self, outs, x):
        return outs[0].view(outs[0].shape[0], *x.shape[1:])

    def __call__(self, x, target=None, gather=False, group=None, n_groups=None, absolute=False, valid=None):
        self.model._xshape = tuple(x.shape[1:])
        return super().__call__(x, target, gather, valid, absolute, group, n_groups)


class FakeGraphGradient(_Fake):
    def _levels(self):
        m = self.model
        out = {}
        for i, lvl in enumerate(m._graph_levels):
            pl = m._plan(m.L[i])
            out.setdefault(lvl, (pl.nnz, pl.M))
        return sorted(out.items())

    def _values(self, x):
        vals = []
        for k, (lvl, (nnz, M)) in enumerate(self._levels()):
            v = _per_window(x, nnz + M) * (k + 1)
            vals += [v[:, :nnz], v[:, nnz:]]
        return vals

    def _ungrouped(self, vals, valid, absolute):
        out = {}
        for k, (lvl, _) in enumerate(self._levels()):
            v = torch.cat([vals[2 * k], vals[2 * k + 1]], 1)[:valid]
            out[lvl] = (v.abs() if absolute else v).sum(0)
        return out

    def _pack(self, outs, x):
        return {lvl: (outs[2 * k], outs[2 * k + 1]) for k, (lvl, _) in enumerate(self._levels())}


class FakeAdjacencyGradient(_Fake):
    def __init__(self, model, maps, *args, **kw):
        super().__init__(model)
        self.maps = maps

    def _values(self, x):
        return [_per_window(x, len(self.maps.rows))]

    def _ungrouped(self, vals, valid, absolute):
        v = vals[0][:valid]
        return (v.abs() if absolute else v).sum(0)

    def _pack(self, outs, x):
        return outs[0]


@pytest.fixture()
def model(graph_l4, monkeypatch):
    from gcn_fmri_decoding_b200 import saliency
    from gcn_fmri_decoding_b200.models import cgcnn

    monkeypatch.setattr(saliency, "InputGradient", FakeInputGradient)
    monkeypatch.setattr(saliency, "GraphGradient", FakeGraphGradient)
    monkeypatch.setattr(saliency, "AdjacencyGradient", FakeAdjacencyGradient)
    _Fake.calls = []
    return cgcnn(L=graph_l4["L"], F=[8, 8], K=[3, 3], p=[4, 4], M=[16, C_], channel=15, device="cpu", seed=1,
                 batch_size=BS, perm=graph_l4["perm"], n_input_vertices=360)


def _data(n, seed=0):
    rng = np.random.RandomState(seed)
    return rng.randn(n, 360, 15).astype(np.float32)


def _expected(x, ids, G, width_of, absolute=False, target=None):
    """Per batch: float32 row-order sums per group, added in float64 in batch order."""
    out = np.zeros((G, width_of))
    for begin in range(0, x.shape[0], BS):
        end = min(begin + BS, x.shape[0])
        xb = torch.as_tensor(x[begin:end])
        v = _per_window(xb, width_of)
        if absolute:
            v = v.abs()
        t = _target_of(xb, None if target is None else torch.as_tensor(target[begin:end])).numpy()
        gid = t if ids is None else ids[begin:end]
        for g in np.unique(gid):
            acc = torch.zeros(width_of)
            for r in np.flatnonzero(gid == g):
                acc += v[r]
            out[g] += acc.numpy().astype(np.float64)
    return out


def test_saliency_grouped_ids_padding_and_float64_batch_order(model):
    x = _data(40)
    ids = np.random.RandomState(1).choice([3, 7, 100], 40)
    for absolute in (False, True):
        _Fake.calls = []
        sums, counts, targets = model.saliency(x, gather=True, groups=ids, absolute=absolute)
        assert sums.dtype == np.float64 and sums.shape == (101, 360, 15)
        assert counts.dtype == np.int64 and counts.tolist() == np.bincount(ids, minlength=101).tolist()
        assert targets.dtype == np.int64 and targets.shape == (40,)
        want = _expected(x, ids, 101, 360 * 15, absolute).reshape(101, 360, 15)
        assert np.array_equal(sums, want)  # bit for bit: float64 accumulation in batch order
        assert not np.isnan(sums).any()
        assert len(_Fake.calls) == 3
        for j, call in enumerate(_Fake.calls):
            begin, end = j * BS, min(j * BS + BS, 40)
            uniq, dense = np.unique(ids[begin:end], return_inverse=True)
            g = call["group"].numpy()
            assert call["n_groups"] == BS
            assert g[: end - begin].tolist() == dense.tolist()
            assert (g[end - begin:] == -1).all()


def test_saliency_grouped_by_target(model):
    x = _data(37, seed=2)
    sums, counts, targets = model.saliency(x, gather=True, groups="target")
    want_t = _target_of(torch.as_tensor(x), None).numpy()
    assert sums.shape == (C_, 360, 15) and np.array_equal(targets, want_t)
    assert counts.tolist() == np.bincount(want_t, minlength=C_).tolist()
    assert np.array_equal(sums, _expected(x, None, C_, 360 * 15).reshape(C_, 360, 15))
    assert all(c["mode"] == "target" for c in _Fake.calls)
    given = np.arange(37) % C_
    sums, counts, targets = model.saliency(x, target=given, gather=True, groups="target")
    assert np.array_equal(targets, given) and counts.tolist() == np.bincount(given, minlength=C_).tolist()
    assert np.array_equal(sums, _expected(x, None, C_, 360 * 15, target=given).reshape(C_, 360, 15))


def test_graph_saliency_grouped(model):
    from gcn_fmri_decoding_b200.saliency import edge_matrix, to_input_order

    x = _data(35, seed=3)
    ids = np.random.RandomState(4).randint(0, 4, 35)
    got, counts = model.graph_saliency(x, gather=True, groups=ids, absolute=True)
    assert counts.tolist() == np.bincount(ids, minlength=4).tolist()
    levels = FakeGraphGradient(model)._levels()
    assert sorted(got) == [lvl for lvl, _ in levels]
    perm = model.perm.numpy()
    for k, (lvl, (nnz, M)) in enumerate(levels):
        mats = got[lvl]
        assert len(mats) == 4
        pl = model._plan(model.L[model._graph_levels.index(lvl)])
        for g in range(4):
            ref = np.zeros(nnz + M)
            for begin in range(0, 35, BS):
                end = min(begin + BS, 35)
                v = (_per_window(torch.as_tensor(x[begin:end]), nnz + M) * (k + 1)).abs()
                sel = np.flatnonzero(ids[begin:end] == g)
                acc = torch.zeros(nnz + M)
                for r in sel:
                    acc += v[r]
                if len(sel):
                    ref += acc.numpy().astype(np.float64)
            R = edge_matrix(pl, ref)
            if lvl == 0:
                R = to_input_order(R, perm, 360)
            assert isinstance(mats[g], sp.csr_matrix) and mats[g].dtype == np.float64
            assert mats[g].shape == R.shape and (mats[g] != R).nnz == 0


def test_adjacency_saliency_grouped(model, graph_l4):
    x = _data(20, seed=5)
    ids = np.random.RandomState(6).randint(0, 3, 20)
    got, counts = model.adjacency_saliency(x, graph_l4["A"], gather=True, groups=ids)
    assert len(got) == 3 and counts.tolist() == np.bincount(ids, minlength=3).tolist()
    maps = model.__dict__["_adjacency_saliency"][2].maps
    want = _expected(x, ids, 3, len(maps.rows))
    for g in range(3):
        assert isinstance(got[g], sp.csr_matrix) and (got[g] != got[g].T).nnz == 0
        assert (got[g] != maps.matrix(want[g])).nnz == 0
    by_target, counts = model.adjacency_saliency(x, graph_l4["A"], gather=True, groups="target")
    assert len(by_target) == C_ and counts.sum() == 20


def test_ungrouped_calls_are_unchanged(model, graph_l4):
    x = _data(20, seed=7)
    grads, targets = model.saliency(x, gather=True)
    assert grads.shape == (20, 360, 15) and grads.dtype == np.float32
    assert all(c["group"] is None and c["mode"] is None for c in _Fake.calls)
    assert isinstance(model.graph_saliency(x, gather=True), dict)
    assert isinstance(model.adjacency_saliency(x, graph_l4["A"], gather=True), sp.csr_matrix)


@pytest.mark.parametrize("call", ["saliency", "graph_saliency", "adjacency_saliency"])
def test_refusals(model, graph_l4, call):
    x = _data(10, seed=8)
    run = (lambda **kw: getattr(model, call)(x, graph_l4["A"], gather=True, **kw)) if call == "adjacency_saliency" \
        else (lambda **kw: getattr(model, call)(x, gather=True, **kw))
    for groups, msg in ((np.zeros(9, np.int64), "shape"), (np.zeros((10, 1), np.int64), "shape"),
                        (np.full(10, -1), "non-negative"), (np.zeros(10, np.float64), "integer"),
                        (np.array([0.5] * 10), "integer"), ("labels", "'target'")):
        with pytest.raises(ValueError, match="cgcnn.%s: groups.*%s" % (call, msg)):
            run(groups=groups)
    assert _Fake.calls == []


def test_saliency_absolute_needs_groups(model):
    with pytest.raises(ValueError, match="absolute needs groups"):
        model.saliency(_data(4), gather=True, absolute=True)


def test_graph_calls_refuse_fourier_with_groups(graph_l4):
    from gcn_fmri_decoding_b200.models import cgcnn

    four = cgcnn(L=graph_l4["L"], F=[8, 8], K=[0, 0], p=[4, 4], M=[16, C_], filter="fourier", channel=15, device="cpu",
                 seed=1, batch_size=BS, perm=graph_l4["perm"], n_input_vertices=360)
    with pytest.raises(ValueError, match="fourier"):
        four.graph_saliency(_data(4), gather=True, groups=np.zeros(4, np.int64))
    with pytest.raises(ValueError, match="fourier"):
        four.adjacency_saliency(_data(4), graph_l4["A"], gather=True, groups="target")
