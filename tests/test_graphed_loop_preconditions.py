"""CPU-side checks of the graphed steps' training-loop features: per-term losses, silhouette cameras, batches smaller
than the captured one, and HostPipeline with a short last batch.  There is no device here, so the step's kernels and the
CUDA-graph capture are replaced by CPU stand-ins: `_capture` runs the warm-up and the captured call eagerly and its
"replay" reruns the captured call into the static outputs, and PrimitiveLoss.__call__ computes its terms with torch.
What is checked is the step layer itself: which buffers, shapes, cameras and uniforms each batch size's graph gets, when
after_backward runs, and what is refused before any copy."""
import pytest
import torch


@pytest.fixture(scope="module")
def step_mod():
    from vpn_b200 import step
    return step


class Log(list):
    state: dict


class FakeGraph:
    def __init__(self, run, outs, pool, log):
        self.run, self.outs, self._pool, self.log = run, outs, pool if pool is not None else object(), log

    def pool(self):
        return self._pool

    def replay(self):
        self.log.append(("replay",))
        new = self.run()
        for o, n in zip(self.outs[:-1], new[:-1]):
            o.copy_(n)
        for k, o in self.outs[-1].items():
            o.copy_(new[-1][k])


@pytest.fixture
def fake(monkeypatch, step_mod):
    """Replaces _capture and PrimitiveLoss.__call__; returns the event log."""
    log = Log()
    state = {"capturing": False}

    def capture(run, device, warmup, warm=None, pool=None):
        log.append(("capture", pool))
        for _ in range(warmup):
            (warm or run)()
        state["capturing"] = True
        try:
            outs = run()
            # static output buffers of their own, as a captured graph's are
            outs = (*(o.detach().clone() for o in outs[:-1]), {k: o.detach().clone() for k, o in outs[-1].items()})
        finally:
            state["capturing"] = False
        return FakeGraph(run, outs, pool, log), outs, 7

    def call(self, v, q, t, uniforms, targets, silhouettes=None, canonical_points=None, dists=None, elevs=None,
             azims=None, angles=None, sil_cameras=None):
        shapes = None if uniforms is None else ([tuple(u.shape) for u in uniforms] if isinstance(uniforms, tuple)
                                                else tuple(uniforms.shape))
        log.append(("step", q.shape[0], shapes, None if sil_cameras is None else tuple(c.shape[0] for c in sil_cameras)))
        out = {"points": v, "view_cd": ((v * v).sum() + q.sum()) * targets.mean() * self.cfg.l_view_cd,
               "vp_div": (t * t).sum() * self.cfg.l_vp_div}
        if self.cfg.l_sil:
            scale = 1.0 if sil_cameras is None else sil_cameras[0].sum()
            out["sil"] = (q * silhouettes.mean()).sum() * scale * self.cfg.l_sil
        total = None
        for k in self.TERMS:
            if k in out:
                total = out[k] if total is None else total + out[k]
        out["total"] = total
        return out

    monkeypatch.setattr(step_mod, "_capture", capture)
    monkeypatch.setattr(step_mod.PrimitiveLoss, "__call__", call)
    log.state = state
    return log


def batch(b, k=4, res=8, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(b, k, 3, generator=g), torch.rand(b, k, 4, generator=g), torch.rand(b, k, 3, generator=g),
            torch.rand(b, 16, 3, generator=g), torch.rand(b, 1, res, res, generator=g))


def cams(b, seed):
    g = torch.Generator().manual_seed(seed)
    return 1.0 + torch.rand(b, generator=g), 30 * torch.rand(b, generator=g), 360 * torch.rand(b, generator=g)


def eager_terms(step_mod, cfg, v, q, t, tgt, sil, sc=None):
    v, q, t = (x.clone().requires_grad_() for x in (v, q, t))
    out = step_mod.PrimitiveLoss(cfg)(v, q, t, None, tgt, silhouettes=sil, sil_cameras=sc)
    gv, gq, gt = torch.autograd.grad(out["total"], (v, q, t))
    return out, (gv, gq, gt)


@pytest.mark.parametrize("kind", ["sphere", "mixed", "vertex"])
def test_short_batches_get_their_own_graph_and_rows(step_mod, fake, kind):
    cfg = step_mod.PrimitiveLossConfig(kind="mixed" if kind == "mixed" else "sphere", n_cuboids=1 if kind == "mixed" else 0,
                                       l_sil=1.0, vertex_chamfer=kind == "vertex")
    collectives = []
    ab = lambda: collectives.append(fake.state["capturing"])
    n = 0 if kind == "vertex" else 5
    v, q, t, tgt, sil = batch(4)
    g = step_mod.GraphedPrimitiveLoss(cfg, v, q, t, tgt, sil, n_samples=n, after_backward=ab)
    # construction: three eager warm-up steps run the collective (every rank constructs), the captured call records it
    assert collectives == [False, False, False, True]
    assert [e[0] for e in fake if e[0] in ("capture", "replay")] == ["capture"] and fake[0][1] is None
    full_pool = g.graph.pool()
    want_u = {"sphere": lambda b: (b, 4, 5, 2), "mixed": lambda b: [(b, 1, 5, 3), (b, 3, 5, 2)], "vertex": lambda b: None}[kind]
    for i, b in enumerate((3, 4, 3)):
        fake.clear(); collectives.clear()
        v, q, t, tgt, sil = batch(b, seed=10 + i)
        loss, gv, gq, gt = g(v, q, t, tgt, sil)
        steps = [e for e in fake if e[0] == "step"]
        captures = [e for e in fake if e[0] == "capture"]
        out, grads = eager_terms(step_mod, cfg, v, q, t, tgt, sil)
        assert torch.equal(loss, out["total"].detach())
        for got, want in zip((gv, gq, gt), grads):
            assert got.shape == want.shape and torch.equal(got, want)
        assert list(g.terms) == ["view_cd", "vp_div", "sil"]
        for k, val in g.terms.items():
            assert torch.equal(val, out[k].detach()), k
        assert all(e[1] == b and e[2] == want_u(b) for e in steps)
        if i == 0:
            # lazy capture into the full-size graph's pool; its warm-ups leave the collective out
            assert captures == [("capture", full_pool)] and len(steps) == 3 + 1 + 1
            assert collectives == [True, False]
        else:
            assert captures == [] and len(steps) == 1 and collectives == [False]
        assert torch.equal(g.v[:b], v) and torch.equal(g.targets[:b], tgt)         # staged into the leading rows
    assert g.graph is g._graphs[4].graph and len(g._graphs) == 2


def test_larger_batch_is_refused_before_any_copy(step_mod, fake):
    cfg = step_mod.PrimitiveLossConfig(vertex_chamfer=True, l_sil=1.0)
    g = step_mod.GraphedPrimitiveLoss(cfg, *batch(4))
    before = [x.clone() for x in (g.v, g.q, g.t, g.targets, g.sil)]
    fake.clear()
    with pytest.raises(AssertionError, match="at most 4"):
        g(*batch(5, seed=3))
    assert fake == []
    for x, y in zip(before, (g.v, g.q, g.t, g.targets, g.sil)):
        assert torch.equal(x, y)


def test_sil_cameras_reach_the_step(step_mod, fake):
    cfg = step_mod.PrimitiveLossConfig(vertex_chamfer=True, l_sil=1.0)
    v, q, t, tgt, sil = batch(4)
    g = step_mod.GraphedPrimitiveLoss(cfg, v, q, t, tgt, sil, sil_cameras=cams(4, 1))
    plain = step_mod.GraphedPrimitiveLoss(cfg, v, q, t, tgt, sil)
    for b, seed in ((4, 2), (3, 3)):
        fake.clear()
        v, q, t, tgt, sil = batch(b, seed=seed)
        sc = cams(b, seed)
        loss = g(v, q, t, tgt, sil, sil_cameras=sc)[0].clone()
        assert [e for e in fake if e[0] == "step"] and all(e[3] == (b, b, b) for e in fake if e[0] == "step")
        out, _ = eager_terms(step_mod, cfg, v, q, t, tgt, sil, sc)
        assert torch.equal(loss, out["total"].detach()) and torch.equal(g.terms["sil"], out["sil"].detach())
        fake.clear()
        assert not torch.equal(plain(v, q, t, tgt, sil)[0], loss)                 # the view-centred camera
        assert all(e[3] is None for e in fake if e[0] == "step")


def test_default_outputs_unchanged(step_mod, fake):
    """The return value is the 4-tuple of before; the full-size graph's outputs stay the object's attributes."""
    cfg = step_mod.PrimitiveLossConfig(vertex_chamfer=True)
    g = step_mod.GraphedPrimitiveLoss(cfg, *batch(4)[:4])
    outs = g(*batch(4, seed=5)[:4])
    assert isinstance(outs, tuple) and len(outs) == 4
    assert all(a is b for a, b in zip(outs, (g.loss, g.gv, g.gq, g.gt)))
    assert g.launches_per_step == 7 and list(g.terms) == ["view_cd", "vp_div"]


def test_term_names_follow_the_summation_order(step_mod):
    assert step_mod.PrimitiveLoss.TERMS == ("view_cd", "obj_cd", "vp_div", "emd", "sil")
    assert step_mod.MeshLoss.TERMS == ("cd", "emd", "sil")


def test_host_pipeline_takes_a_short_last_batch():
    """Five full batches, then one of 2 rows out of 4, with the step's 'terms' returned next to its results: results in
    order and equal to direct calls; full-size batches reuse their slot's host buffers, the short one gets its own; a
    batch larger than the example is refused before the step runs."""
    import vpn_b200
    seen = []

    def step(s):
        seen.append(tuple(s["x"].shape))
        x = s["x"]
        return x.sum(), x * 2, x.max(), s["y"][:, 0] + 1

    example = {"x": torch.zeros(4, 3), "y": torch.zeros(4, 2), "unused": None}
    g = torch.Generator().manual_seed(0)
    batches = [{"x": torch.rand(4, 3, generator=g), "y": torch.rand(4, 2, generator=g), "unused": None} for _ in range(5)]
    batches.append({"x": torch.rand(2, 3, generator=g), "y": torch.rand(2, 2, generator=g), "unused": None})
    want = [[o.clone() for o in step(bt)] for bt in batches]
    seen.clear()
    pipe = vpn_b200.HostPipeline(step, example, "cpu")
    got, objs = [], []
    pipe.submit(batches[0])
    for bt in batches[1:]:
        pipe.submit(bt)
        r = pipe.result()
        objs.append(r)
        got.append([o.clone() for o in r])
    r = pipe.result()
    objs.append(r)
    got.append([o.clone() for o in r])
    assert seen == [(4, 3)] * 5 + [(2, 3)]
    for w, gg in zip(want, got):
        assert [tuple(o.shape) for o in gg] == [tuple(o.shape) for o in w]
        for a, c in zip(w, gg):
            assert torch.equal(a, c)
    assert objs[0] is objs[2] is objs[4] and objs[1] is objs[3]                  # one set of buffers per slot
    assert objs[5] is not objs[3] and tuple(objs[5][1].shape) == (2, 3)
    with pytest.raises(AssertionError, match="example batch"):
        pipe.submit({"x": torch.rand(5, 3), "y": torch.rand(5, 2), "unused": None})
    assert len(seen) == 6
