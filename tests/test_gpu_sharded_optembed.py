"""Row sharding of the OptEmbed family: the supernet (`deepfm_optembed`, `deepfm_optembed_d`) and its retrain stage
(`deepfm_optembed_retrain`).

Kernel level: "virtual" shards on ONE GPU (the pointer table points at G tensors) must give the single-table OPTEMBED
kernels' results bit for bit - forward, chain-rule backward (including the per-lookup mask-E scalars) and the pushes
into the owners' gradient shards.  Module level: ShardedDeepFM / ShardedDCNMix at world 1 against the single-device
model (training, the eval cache, the plugin's bookkeeping, state-dict round trips, the retrain mask), and at world 2 over
NCCL + NVLink peer access when the box has two GPUs."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.helpers import assert_close

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
DIMS = [50, 7, 300, 11, 5, 1000, 3]
D = 16


@pytest.fixture(scope="module")
def env():
    import __graft_entry__ as G

    G.build()
    import recsys_benchmark_b200.functional as RF
    from recsys_benchmark_b200 import _lib as L
    from recsys_benchmark_b200 import sharded as S

    return RF, L, S


def _ids(b, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.stack([torch.randint(0, d, (b,), generator=g) for d in DIMS], 1)


def _ptr_table(tensors):
    return torch.tensor([t.data_ptr() for t in tensors], dtype=torch.int64, device=DEV)


def _offsets(dev):
    return torch.tensor([0] + DIMS[:-1]).cumsum(0).to(dev)


# ---------------------------------------------------------------- kernel level
@pytest.mark.parametrize("case", ["norm1", "norm2", "mask_e_off"])
@pytest.mark.parametrize("with_mask_d", [False, True])
@pytest.mark.parametrize("G", [1, 3])
def test_virtual_shards_match_the_single_table_optembed_kernels_bit_for_bit(env, case, with_mask_d, G):
    RF, L, S = env
    lib = L.load()
    torch.manual_seed(13)
    n = sum(DIMS)
    b, f = 97, len(DIMS)
    x = _ids(b, 4).to(DEV)
    offsets = _offsets(DEV)
    table = torch.rand(n, D, device=DEV) - 0.5
    norm = 2 if case == "norm2" else 1
    t = None
    if case != "mask_e_off":
        # per-field thresholds around the median row norm: about half the rows survive mask-E
        nrm = table.norm(p=norm, dim=1)
        t = (nrm.median() + 0.1 * torch.randn(f, device=DEV)).contiguous()
    mask_d = torch.randint(0, D, (b, f), device=DEV) if with_mask_d else None
    fc = torch.randn(n, 1, device=DEV)
    bias = torch.randn(1, device=DEV)

    def outputs():
        return (torch.empty(b, f, D, device=DEV), torch.empty(b, device=DEV), torch.empty(b, D, device=DEV),
                torch.empty(b, f, dtype=torch.int64, device=DEV))

    st = L.stream_ptr(torch.device(DEV))
    err = torch.zeros(1, dtype=torch.int32, device=DEV)
    emb0, y0, s0, rows0 = outputs()
    L.check(lib.rsb_lookup_fwd(L.KIND_OPTEMBED, L.ptr(x), 0, L.ptr(offsets), b, f, D, L.ptr(table), n, n, None, 0,
                               L.ptr(t), norm, L.ptr(mask_d), L.ptr(fc), L.ptr(bias), L.ptr(emb0), L.ptr(y0), L.ptr(s0),
                               L.ptr(rows0), L.ptr(err), None, st))
    shards = [S.shard_of_full(table, g, G).contiguous() for g in range(G)]
    tp = _ptr_table(shards)
    emb1, y1, s1, rows1 = outputs()
    L.check(lib.rsb_lookup_fwd_sharded_kind(L.KIND_OPTEMBED, L.ptr(x), 0, L.ptr(offsets), b, f, D, L.ptr(tp), G, n, n,
                                            None, 0, L.ptr(t), None, norm, L.ptr(mask_d), L.ptr(fc), L.ptr(bias),
                                            L.ptr(emb1), L.ptr(y1), L.ptr(s1), L.ptr(rows1), L.ptr(err), None, st))
    assert int(err.item()) == 0
    assert torch.equal(rows0, rows1) and torch.equal(emb0, emb1) and torch.equal(y0, y1) and torch.equal(s0, s1)
    if t is not None:
        zero_rows = (emb0.abs().sum(-1) == 0).float().mean().item()
        assert 0.1 < zero_rows < 0.9, "the thresholds should drop some rows and keep others"

    # chain-rule backward: per-lookup row gradients and (mask-E on) one g_z per lookup
    g_deep = torch.randn(b, f, D, device=DEV)
    g_y = torch.randn(b, device=DEV)
    rg0, rg1 = torch.zeros(b * f, D, device=DEV), torch.zeros(b * f, D, device=DEV)
    ra0 = torch.zeros(b, f, device=DEV) if t is not None else None
    ra1 = torch.zeros(b, f, device=DEV) if t is not None else None
    L.check(lib.rsb_lookup_bwd_rows(L.KIND_OPTEMBED, L.ptr(rows0), b, f, D, L.ptr(table), n, None, 0, L.ptr(t), norm,
                                    L.ptr(mask_d), L.ptr(emb0), L.ptr(s0), L.ptr(g_y), L.ptr(g_deep), L.ptr(rg0),
                                    L.ptr(ra0), None, st))
    L.check(lib.rsb_lookup_bwd_rows_sharded(L.KIND_OPTEMBED, L.ptr(rows0), b, f, D, L.ptr(tp), G, n, None, 0, L.ptr(t),
                                            None, norm, L.ptr(mask_d), L.ptr(emb0), L.ptr(s0), L.ptr(g_y),
                                            L.ptr(g_deep), L.ptr(rg1), L.ptr(ra1), st))
    assert torch.equal(rg0, rg1)
    if t is not None:
        assert torch.equal(ra0, ra1)
        assert bool((ra0 != 0).any()), "some lookups sit inside the BinaryStep surrogate's support"

    # pushes into the owners' gradient shards == the dense scatter-add, re-assembled
    pair = RF.sort_rows(rows0, n)
    dense = RF.dense_row_grad(rows0, rg0, n, sorted_pair=pair)
    gshards = [torch.zeros_like(s) for s in shards]
    ws = RF._ws(lib.rsb_segment_workspace_bytes(b * f, D), torch.device(DEV))
    L.check(lib.rsb_segment_scatter_shards(L.ptr(pair[0]), L.ptr(pair[1]), b * f, L.ptr(rg0), D, L.ptr(_ptr_table(gshards)),
                                           G, 1.0, None, f, None, L.ptr(ws), ws.numel(), st))
    assert torch.equal(S.full_from_shards(gshards, n), dense)


# ---------------------------------------------------------------- module level
CONFIGS = {"optembed": {"name": "deepfm_optembed"}, "optembed_d": {"name": "deepfm_optembed_d"},
           "optembed_l2": {"name": "deepfm_optembed", "norm": 2},
           "optembed_retrain": {"name": "deepfm_optembed_retrain"}}


def _models(R, S, name, model_kind, dev, group=None):
    cfg = CONFIGS[name]
    torch.manual_seed(5)
    if model_kind == "deepfm":
        full = R.get_ctr_model(DIMS, dict(num_factor=D, hidden_sizes=[32, 16], p_dropout=0.0, use_batchnorm=False,
                                          embedding_config=dict(cfg))).to(dev)
        torch.manual_seed(5)
        sh = S.ShardedDeepFM(DIMS, D, [32, 16], p_dropout=0.0, use_batchnorm=False, embedding_config=dict(cfg),
                             group=group).to(dev)
    else:
        full = R.get_ctr_model(DIMS, dict(name="dcn_mix", num_factor=D, hidden_sizes=[32], num_layers=2, num_experts=2,
                                          rank=8, p_dropout=0.0, embedding_config=dict(cfg))).to(dev)
        torch.manual_seed(5)
        sh = S.ShardedDCNMix(DIMS, D, [32], num_layers=2, num_experts=2, rank=8, p_dropout=0.0,
                             embedding_config=dict(cfg), group=group).to(dev)
    if name == "optembed_retrain":
        # RetrainOptEmbed leaves its weight uninitialised (the retrain script loads one): a seeded one here
        with torch.no_grad():
            full.embedding._weight.copy_(torch.randn(sum(DIMS), D, generator=torch.Generator().manual_seed(9)) * 0.2)
    _copy_state(full, sh)
    return full, sh


def _copy_state(full, sh):
    """The single-device model's parameters into the sharded one (replicated ones directly, the embedding through its
    full-state conversion)."""
    st = {k: v for k, v in full.state_dict().items() if not k.startswith("embedding.")}
    sh.load_state_dict(st, strict=False)
    sh.embedding.load_full_state_dict(full.embedding.state_dict())


def _retrain_masks(seed=21):
    g = torch.Generator().manual_seed(seed)
    mask_e = (torch.rand(sum(DIMS), generator=g) > 0.3).to(torch.int64)
    mask_d = torch.randint(0, D, (len(DIMS),), generator=g)
    return mask_e, mask_d


def _train(model, x, y, steps, sharded, seed=17, lr=1e-2):
    torch.manual_seed(seed)          # the same mask-D draws for both models
    opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=lr, weight_decay=1e-4)
    crit = torch.nn.BCEWithLogitsLoss()
    outs = []
    for _ in range(steps):
        logits = model(x)
        loss = crit(logits, y)
        opt.zero_grad()
        loss.backward()
        if sharded:
            model.sync_gradients()
        opt.step()
        if sharded:
            model.finish_step()
        outs.append(logits.detach().clone())
    return outs


def _check_state(full, sh, atol_scale):
    ref = full.embedding.state_dict()
    got = sh.embedding.full_state_dict()
    assert got.keys() == ref.keys()
    for k, v in ref.items():
        assert got[k].dtype == v.dtype, k
        if not v.is_floating_point():
            assert torch.equal(got[k].cpu(), v.cpu()), k
        else:
            assert_close(got[k].cpu().numpy(), v.detach().cpu().numpy(), what=f"{k}", atol_scale=atol_scale)


MODULE_CASES = [("deepfm", "optembed"), ("deepfm", "optembed_d"), ("deepfm", "optembed_l2"),
                ("deepfm", "optembed_retrain"), ("dcn", "optembed")]


@pytest.mark.parametrize("model_kind,name", MODULE_CASES)
def test_sharded_optembed_world1_matches_the_single_device_model(env, model_kind, name):
    RF, L, S = env
    import recsys_benchmark_b200 as R

    dev = torch.device(DEV)
    full, sh = _models(R, S, name, model_kind, dev)
    g = torch.Generator().manual_seed(1)
    x = _ids(64, 1).to(dev)
    y = torch.randint(0, 2, (64,), generator=g).float().to(dev)
    retrain = name == "optembed_retrain"
    if retrain:
        with pytest.raises(AssertionError):
            full(x)
        with pytest.raises(AssertionError):
            sh(x)
        mask_e, mask_d = _retrain_masks()
        full.embedding.init_mask(mask_e, mask_d)
        shard = sh.embedding.init_mask(mask_e, mask_d)
        assert shard.shape == (sh.embedding.shards.n_local, D) and shard.dtype == torch.bool
        ref_mask = full.embedding.state_dict()["_mask"]
        got_mask = sh.embedding.full_state_dict()["_mask"]
        assert got_mask.dtype == ref_mask.dtype and torch.equal(got_mask, ref_mask)

    a = _train(full, x, y, 3, False)
    b = _train(sh, x, y, 3, True)
    assert torch.equal(a[0], b[0]), "same rows, same mask-D draw, same kernel arithmetic"
    for s in range(3):
        assert_close(b[s].cpu().numpy(), a[s].cpu().numpy(), what=f"logits step {s}", atol_scale=5e-5)
    _check_state(full, sh, 5e-5)

    # evaluation on identical parameters: the eval shards are built by the single-device cache's kernel
    _copy_state(full, sh)
    full.eval()
    sh.eval()
    with torch.no_grad():
        assert torch.equal(sh(x), full(x)), "eval logits"
        x_off = x + _offsets(dev)
        md = torch.randint(0, D, (len(DIMS),), generator=torch.Generator().manual_seed(3))
        assert torch.equal(sh.embedding(x_off, md), full.embedding(x_off, md)), "forward(x, mask_d)"
        assert torch.equal(sh(x), full(x)), "eval logits after a mask-D rebuild"
        if retrain:
            assert torch.equal(sh.embedding.get_weight(), full.embedding.get_weight())
        else:
            assert torch.equal(sh.embedding.get_weight(md), full.embedding.get_weight(md)), "get_weight(mask_d)"
            assert torch.equal(sh.embedding.get_mask_e(), full.embedding.get_mask_e())
            assert torch.equal(sh.embedding.get_submask(), full.embedding.get_submask())
            l_s_sh, l_s_full = sh.embedding.get_l_s(), full.embedding.get_l_s()
            assert (torch.equal(l_s_sh, l_s_full) if torch.is_tensor(l_s_full) else l_s_sh == l_s_full)
        assert sh.embedding.get_sparsity() == full.embedding.get_sparsity()
        assert sh.embedding.get_sparsity(True) == full.embedding.get_sparsity(True)
        assert sh.embedding.get_num_params() == full.embedding.get_num_params()

    # the gathered state loads strictly into a fresh single-device module
    fresh = R.get_embedding(dict(CONFIGS[name]), DIMS, D).to(dev)
    if retrain:
        fresh.init_mask(*_retrain_masks(seed=99))
    fresh.load_state_dict(sh.embedding.full_state_dict(), strict=True)
    for k, v in full.embedding.state_dict().items():
        assert torch.equal(fresh.state_dict()[k], v), k
    if retrain:
        # a retrain checkpoint (with its mask) loads into a wrapper whose init_mask never ran
        sh2 = S.ShardedEmbedding(R.get_embedding(dict(CONFIGS[name]), DIMS, D))
        sh2.load_full_state_dict(full.embedding.state_dict())
        for k, v in sh2.full_state_dict().items():
            assert torch.equal(v, full.embedding.state_dict()[k]), k
        assert torch.equal(sh2.get_weight(), full.embedding.get_weight())


def test_sharded_optembed_eval_cache_follows_the_reference(env):
    """Fresh module in eval(): F.embedding on an empty weight raises (INTEGRATION 5); after get_weight() the cache
    exists; a training forward invalidates it and the next eval lookup rebuilds it."""
    RF, L, S = env
    import recsys_benchmark_b200 as R

    dev = torch.device(DEV)
    full, sh = _models(R, S, "optembed", "deepfm", dev)
    x = _ids(32, 6).to(dev)
    full.eval()
    sh.eval()
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="must be 2-D"):
            full(x)
        with pytest.raises(RuntimeError, match="must be 2-D"):
            sh(x)
        assert torch.equal(sh.embedding.get_weight(), full.embedding.get_weight())
        assert torch.equal(sh(x), full(x))
        assert sh.embedding.get_num_params() == full.embedding.get_num_params()
    y = torch.randint(0, 2, (32,), generator=torch.Generator().manual_seed(2)).float().to(dev)
    full.train()
    sh.train()
    _train(full, x, y, 1, False)
    _train(sh, x, y, 1, True)
    assert sh.embedding._eval_state == "stale" and sh.embedding.inner._submask_cache is None
    _copy_state(full, sh)
    full.eval()
    sh.eval()
    with torch.no_grad():
        assert torch.equal(sh(x), full(x))


def test_sharded_optembed_refuses_feature_thresholds(env):
    RF, L, S = env
    import recsys_benchmark_b200 as R

    inner = R.get_embedding({"name": "deepfm_optembed", "mode_threshold_e": "feature"}, DIMS, D)
    with pytest.raises(NotImplementedError):
        S.ShardedEmbedding(inner)
    with pytest.raises(NotImplementedError):
        S.ShardedDeepFM(DIMS, D, [32], embedding_config={"name": "deepfm_optembed", "mode_threshold_e": "feature"})


# ---------------------------------------------------------------- world 2
def _pin_mask_d(module, draws):
    """Replace the module's per-step mask-D draw by the given [B, F] arrays, one per training forward."""
    it = iter(draws)
    module._mask_d_for = lambda b, f, device: next(it).to(device).contiguous()


def _worker2(rank, world, port, ret, model_kind, name):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        import recsys_benchmark_b200 as R
        from recsys_benchmark_b200 import sharded as S

        full, sh = _models(R, S, name, model_kind, dev)
        for m in list(full.modules()) + list(sh.modules()):
            if isinstance(m, torch.nn.BatchNorm1d):
                m.eval()             # per-rank batch statistics: the global-batch run is not the reference for a slice
        steps, bsz = 3, 128
        g = torch.Generator().manual_seed(2)
        x = _ids(bsz, 2)
        y = torch.randint(0, 2, (bsz,), generator=g).float()
        if name == "optembed_retrain":
            mask_e, mask_d = _retrain_masks()
            full.embedding.init_mask(mask_e, mask_d)
            sh.embedding.init_mask(mask_e, mask_d)
        else:
            # each rank would draw its own [B_local, F] mask-D: pin both to one global draw and its slice
            md = torch.randint(0, D, (steps, bsz, len(DIMS)), generator=torch.Generator().manual_seed(8))
            _pin_mask_d(full.embedding, [md[s] for s in range(steps)])
            _pin_mask_d(sh.embedding.inner, [md[s][rank::world] for s in range(steps)])
        a = _train(full, x.to(dev), y.to(dev), steps, False)          # every rank: the single-GPU run on the global batch
        b = _train(sh, x[rank::world].to(dev), y[rank::world].to(dev), steps, True)
        assert torch.equal(a[0][rank::world], b[0]), "forward over peer shards differs from the single-GPU gather"
        for s in range(steps):
            assert_close(b[s].cpu().numpy(), a[s][rank::world].cpu().numpy(), what=f"logits step {s}", atol_scale=1e-4)
        _check_state(full, sh, 1e-4)
        # counts all-reduced over the shards; the two tables agree to rounding, so a few weights may sit on a threshold
        n_sh, n_full = sh.embedding.get_num_params(), full.embedding.get_num_params()
        assert abs(n_sh - n_full) <= 8, (n_sh, n_full)
        sp_sh, sp_full = sh.embedding.get_sparsity(True), full.embedding.get_sparsity(True)
        assert abs(sp_sh[1] - sp_full[1]) <= 8, (sp_sh, sp_full)
        # eval on identical parameters: the rebuilt eval shards, gathered over NVLink
        _copy_state(full, sh)
        full.eval()
        sh.eval()
        with torch.no_grad():
            ref = full(x.to(dev))
            got = sh(x[rank::world].to(dev))
            assert torch.equal(got, ref[rank::world]), "eval logits over the eval shards"
            if name != "optembed_retrain":
                md1 = torch.randint(0, D, (len(DIMS),), generator=torch.Generator().manual_seed(3))
                assert torch.equal(sh.embedding.get_weight(md1), full.embedding.get_weight(md1))
                assert torch.equal(sh.embedding.get_mask_e(), full.embedding.get_mask_e())
                assert torch.equal(sh.embedding.get_submask(), full.embedding.get_submask())
            assert sh.embedding.get_num_params() == full.embedding.get_num_params()
        sh.embedding.shards.close()          # collective: unmap the peers, barrier, free
        ret[rank] = 1
    finally:
        dist.destroy_process_group()


WORLD2_CASES = [("deepfm", "optembed"), ("deepfm", "optembed_retrain"), ("dcn", "optembed_d")]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("model_kind,name", WORLD2_CASES)
def test_sharded_optembed_world2_matches_single_gpu(model_kind, name):
    import __graft_entry__ as G

    G.build()
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 29850 + (os.getpid() % 40) * 4 + WORLD2_CASES.index((model_kind, name))
    mp.spawn(_worker2, args=(2, port, ret, model_kind, name), nprocs=2, join=True)
    assert dict(ret) == {0: 1, 1: 1}
