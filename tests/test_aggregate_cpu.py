"""The aggregation entry points without a GPU: lkg_aggregate_fwd refuses bad arguments with the right status before it
touches a device, lkg_aggregate_supported describes the kernels' envelope, and the model only asks the layer for shapes
that envelope contains (refusing the others at construction)."""
import argparse
import ctypes

import pytest
import torch

import literalkg_oracle as O

INVALID, UNSUPPORTED = -1, -2
FAKE = 4096                      # a 16-byte aligned address that is never dereferenced: every call stops at validation


@pytest.fixture(scope="module")
def lib():
    from literalkg_b200 import _lib, build
    build.build(verbose=False)
    return _lib.load()


def _graph(**kw):
    from literalkg_b200 import _lib
    g = _lib.LkgGraph()
    g.n_entities, g.row_begin, g.row_end = 10, 0, 10
    g.rowptr = g.col = g.row_order = g.row_sched = FAKE
    for k, v in kw.items():
        setattr(g, k, v)
    return g


def _fwd(lib, g=None, d_in=300, d_out=32, ego=FAKE, pa=None, pb=FAKE, p2=None, z=None, ld_z=0, xn_planes=None,
         xn_rec=None):
    g = _graph() if g is None else g
    return lib.lkg_aggregate_fwd(ctypes.byref(g), FAKE, ego, d_in, d_in, d_out, pa, pb, p2, None, None, 0, FAKE, FAKE,
                                 None, FAKE, d_out, None, 0, xn_planes, 0, 0, xn_rec, 0, z, ld_z, None, 0, None, 0,
                                 FAKE, None)


def _refused(lib, rc, status, words):
    assert rc == status, (rc, lib.lkg_last_error())
    msg = lib.lkg_last_error().decode()
    assert all(w in msg for w in words), msg


def test_fwd_refuses_z_without_p2_or_with_pa_pb(lib):
    _refused(lib, _fwd(lib, pb=None, z=FAKE, ld_z=32), INVALID, ["p2"])
    _refused(lib, _fwd(lib, pb=FAKE, p2=FAKE, z=FAKE, ld_z=32), INVALID, ["no pa / pb"])
    _refused(lib, _fwd(lib, pa=FAKE, pb=None, p2=FAKE, z=FAKE, ld_z=32), INVALID, ["no pa / pb"])
    _refused(lib, _fwd(lib, d_in=64, pb=None, p2=FAKE, z=FAKE, ld_z=32), INVALID, ["wide rows"])
    _refused(lib, _fwd(lib, g=_graph(row_sched=None), pb=None, p2=FAKE, z=FAKE, ld_z=32), INVALID, ["row schedule"])


def test_fwd_refuses_two_sum_matrices_with_p2(lib):
    _refused(lib, _fwd(lib, pa=FAKE + 16, pb=FAKE, p2=FAKE), INVALID, ["one shared sum matrix"])


def test_fwd_refuses_d_in_not_multiple_of_4(lib):
    _refused(lib, _fwd(lib, d_in=302), INVALID, ["multiple of 4", "302"])
    _refused(lib, _fwd(lib, d_in=0), INVALID, ["multiple of 4"])


def test_fwd_refuses_widths_beyond_the_envelope(lib):
    _refused(lib, _fwd(lib, d_in=516), UNSUPPORTED, ["516 > 512"])
    _refused(lib, _fwd(lib, d_out=65), UNSUPPORTED, ["65 > 64"])


def test_fwd_refuses_shapes_no_kernel_runs_before_any_launch(lib):
    # without a device a launch would fail with LKG_ERR_CUDA: these are decided on the host first
    _refused(lib, _fwd(lib, d_in=128, d_out=36, pb=None, p2=FAKE, z=FAKE, ld_z=36), UNSUPPORTED, ["pre-projected", "128"])
    _refused(lib, _fwd(lib, d_in=300, d_out=64, pb=None, p2=FAKE, z=FAKE, ld_z=64), UNSUPPORTED, ["pre-projected"])
    _refused(lib, _fwd(lib, d_in=448, d_out=64, pa=FAKE + 16), UNSUPPORTED, ["shared memory", "448"])
    _refused(lib, _fwd(lib, d_in=404, d_out=61, p2=FAKE), UNSUPPORTED, ["shared memory"])


def test_fwd_refuses_unaligned_ego(lib):
    _refused(lib, _fwd(lib, ego=FAKE + 4), INVALID, ["ego rows"])


def test_fwd_refuses_narrow_segment_scratch(lib):
    g = _graph(n_sched=12, seg_tickets=FAKE, seg_scratch=FAKE, seg_stride=300 + 28)
    _refused(lib, _fwd(lib, g=g, d_in=300, d_out=32), INVALID, ["segment scratch", "300", "32"])
    g.seg_scratch = None
    _refused(lib, _fwd(lib, g=g, d_in=300, d_out=32), INVALID, ["segment scratch"])


def test_fwd_refuses_other_bad_arguments(lib):
    _refused(lib, _fwd(lib, g=_graph(row_begin=4, row_end=3)), INVALID, ["row range"])
    _refused(lib, _fwd(lib, xn_planes=FAKE), INVALID, ["scale record"])
    _refused(lib, _fwd(lib, pb=None), INVALID, ["null"])


def _sup(lib, d_in, d_out, mode):
    ok = ctypes.c_int32(-1)
    assert lib.lkg_aggregate_supported(d_in, d_out, mode, ctypes.byref(ok)) == 0
    assert ok.value in (0, 1)
    return bool(ok.value)


def test_supported_query_envelope(lib):
    from literalkg_b200 import _lib
    one, two, bi, biz = _lib.AGG_ONE_TERM, _lib.AGG_TWO_TERMS, _lib.AGG_BI, _lib.AGG_BI_Z
    ok = ctypes.c_int32(0)
    assert lib.lkg_aggregate_supported(300, 32, 4, ctypes.byref(ok)) == INVALID
    assert lib.lkg_aggregate_supported(300, 32, biz, None) == INVALID
    for d_out in range(4, 65, 4):
        # pre-projected z: only the wide-row stream kernel gathers it -- none for one or two 128-wide slots with two
        # channel chunks, and the 6-slot ring with z rows must fit next to the P2 tile
        assert _sup(lib, 128, d_out, biz) == (d_out <= 32)
        assert _sup(lib, 132, d_out, biz) == (d_out <= 32)
        assert _sup(lib, 256, d_out, biz) == (d_out <= 32)
        assert _sup(lib, 260, d_out, biz) and _sup(lib, 292, d_out, biz)
        assert _sup(lib, 300, d_out, biz) == (d_out <= 52)
        assert not _sup(lib, 64, d_out, biz) and not _sup(lib, 512, d_out, biz)
        for mode in (one, two, bi):                       # the generic kernel covers every width up to 400
            assert _sup(lib, 12, d_out, mode) and _sup(lib, 128, d_out, mode) and _sup(lib, 400, d_out, mode)
    assert not _sup(lib, 300, 30, biz)                   # z rows are gathered as float4
    # two combine matrices of [d_in, d_out] in shared memory: d_out <= 60 from d_in 404 on
    for mode in (two, bi):
        assert _sup(lib, 404, 60, mode) and not _sup(lib, 404, 61, mode) and not _sup(lib, 512, 64, mode)
        assert _sup(lib, 512, 32, mode)
    assert _sup(lib, 512, 64, one)
    for shape in ((302, 32), (516, 32), (300, 65), (0, 32), (300, 0)):
        assert not any(_sup(lib, *shape, m) for m in (one, two, bi, biz))


def _model(**kw):
    import literalkg_b200 as L
    cfg = O.OracleConfig(n_conv_layers=2, **kw)
    args = argparse.Namespace(**{k: getattr(cfg, k) for k in cfg.__dataclass_fields__})
    return L.LiteralKG(args, 10, 2, None, torch.zeros(10, cfg.num_lit_dim), torch.zeros(10, cfg.txt_lit_dim))


@pytest.mark.parametrize("agg,res,d,c,z", [
    ("bi-interaction", True, 300, 32, True), ("bi-interaction", True, 128, 32, True), ("bi-interaction", True, 128, 48, False),
    ("bi-interaction", True, 256, 48, False), ("bi-interaction", True, 300, 64, False),
    ("bi-interaction", False, 300, 32, False), ("gcn", True, 300, 64, True), ("graphsage", True, 128, 16, True),
    ("graphsage", True, 64, 16, False)])
def test_layer1_takes_z_only_where_it_runs(lib, agg, res, d, c, z):
    m = _model(embed_dim=d, relation_dim=d, conv_dim=c, aggregation_type=agg, use_residual=res)
    assert m._layer1_z_path() == z
    if res:
        with torch.no_grad():
            folds = [layer.folded(m.lamda, m.alpha, k + 1) for k, layer in enumerate(m.aggregator_layers)]
            wq, _, _, zcol = m._stack_q(folds)
        assert (zcol >= 0) == z
        assert wq.shape[0] == sum(f["q1"].shape[1] + (0 if f["q2"] is None else c) for f in folds) + (c if z else 0)


@pytest.mark.parametrize("agg,res,d,c", [("graphsage", False, 512, 64), ("bi-interaction", True, 404, 64),
                                         ("bi-interaction", False, 448, 60), ("gcn", False, 302, 32),
                                         ("gcn", False, 300, 68)])
def test_model_refuses_shapes_outside_the_kernels(lib, agg, res, d, c):
    with pytest.raises(ValueError, match="outside the aggregation kernels"):
        _model(embed_dim=d, relation_dim=d, conv_dim=c, aggregation_type=agg, use_residual=res)


@pytest.mark.parametrize("agg,res", [("gcn", False), ("gcn", True), ("graphsage", True)])
def test_model_accepts_wide_single_matrix_layers(lib, agg, res):
    _model(embed_dim=512, relation_dim=512, conv_dim=64, aggregation_type=agg, use_residual=res)
