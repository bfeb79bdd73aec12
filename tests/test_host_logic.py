"""CPU: host-side behaviour of the reference-facing Python surface that needs no GPU --
constructor validation, error conventions, no silent fallback."""
import pytest
import torch

from nope_b200 import NopeError
from nope_b200.encoder import FeatureExtractor
from nope_b200.model import PoseConditional, score_topk
from nope_b200.unet import UNet


def _unet(**kw):
    args = dict(u_net_dim=192, rot_representation_dim=6, encoder=FeatureExtractor(descriptor_size=8),
                pose_mlp_name="single_layer", device="cuda:0")
    args.update(kw)
    return UNet(**args)


def test_unet_keeps_reference_attributes():
    u = _unet()
    assert u.channels == 8 and u.name == "template" and u.encoder.latent_dim == 8
    assert callable(u) and hasattr(u.encoder, "encode_image")


@pytest.mark.parametrize("kw", [dict(pose_mlp_name="two_layers"), dict(pose_mlp_name="posEncoding"),
                                dict(rot_representation_dim=4), dict(dim_mults=(1, 2, 4)),
                                dict(use_hard_up_down=False), dict(resnet_block_groups=4)])
def test_unsupported_unet_configurations_are_rejected(kw):
    with pytest.raises(ValueError):
        _unet(**kw)


def test_unknown_similarity_metric_raises_instead_of_returning_none():
    # the reference's retrieval() falls through and returns None (src/model/model.py:256)
    m = PoseConditional(_unet(), testing_config={"similarity_metric": "dot"})
    with pytest.raises(ValueError):
        m.retrieval(torch.zeros(1, 3, 256, 256), torch.zeros(1, 6, 8, 32, 32))
    with pytest.raises(ValueError):
        m.predict_pose(torch.zeros(1, 3, 256, 256), torch.zeros(1, 3, 256, 256), torch.zeros(1, 6, 6))
    with pytest.raises(ValueError):
        score_topk(torch.zeros(1, 8, 32, 32), torch.zeros(1, 6, 8, 32, 32), metric="dot")


def test_no_cpu_fallback_for_the_hot_path():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(NopeError):
        score_topk(torch.zeros(1, 8, 32, 32), torch.zeros(1, 6, 8, 32, 32))     # CPU tensors
    u = _unet()
    with pytest.raises(NopeError):
        u.sweep(torch.zeros(1, 8, 32, 32), torch.zeros(1, 3, 6))                 # not loaded / no GPU
    with pytest.raises(NopeError):
        FeatureExtractor(descriptor_size=8, backend="b200").encode_image(torch.zeros(1, 3, 256, 256))


def test_loss_type_and_compute_loss():
    m = PoseConditional(_unet(), optim_config={"loss_type": "l2"})
    a, b = torch.ones(2, 8, 32, 32), torch.zeros(2, 8, 32, 32)
    assert float(m.compute_loss(a, b)) == 1.0
    m1 = PoseConditional(_unet(), optim_config={"loss_type": "l1"})
    assert float(m1.compute_loss(a * 3, b)) == 3.0


def test_scripts_have_no_undefined_names():
    """bench.py / __graft_entry__.py paths that only run on a multi-GPU box (torchrun legs) cannot be exercised
    here; at least every name a function loads must be bound in it, at module level, or be a builtin."""
    import ast
    import builtins
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for script in ("bench.py", "__graft_entry__.py"):
        tree = ast.parse(open(os.path.join(root, script)).read())

        def bound_in(scope):
            out = set()
            for n in ast.walk(scope):
                if isinstance(n, ast.Name) and isinstance(n.ctx, ast.Store):
                    out.add(n.id)
                elif isinstance(n, ast.arg):
                    out.add(n.arg)
                elif isinstance(n, (ast.FunctionDef, ast.ClassDef)):
                    out.add(n.name)
                elif isinstance(n, (ast.Import, ast.ImportFrom)):
                    out.update((a.asname or a.name).split(".")[0] for a in n.names)
                elif isinstance(n, ast.ExceptHandler) and n.name:
                    out.add(n.name)
            return out

        module_names = set(dir(builtins))
        for n in tree.body:                      # module level only (not the bodies of other functions)
            if isinstance(n, (ast.FunctionDef, ast.ClassDef)):
                module_names.add(n.name)
            elif isinstance(n, (ast.Import, ast.ImportFrom)):
                module_names.update((a.asname or a.name).split(".")[0] for a in n.names)
            elif isinstance(n, (ast.Assign, ast.AugAssign, ast.AnnAssign, ast.If, ast.Try, ast.With, ast.For)):
                module_names |= bound_in(n)
        for fn in [n for n in tree.body if isinstance(n, ast.FunctionDef)]:
            names = module_names | bound_in(fn)
            missing = {n.id for n in ast.walk(fn) if isinstance(n, ast.Name) and isinstance(n.ctx, ast.Load)
                       and n.id not in names}
            assert not missing, (script, fn.name, sorted(missing))


def test_bench_dump_outputs_keeps_dtypes_and_the_size_cap(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 stays float32, indices become float64, and past the size cap the
    largest array is replaced by the same seeded sample of its elements on every run."""
    import numpy as np
    import bench
    sim, topi = torch.randn(3, 1000), torch.arange(15).view(3, 5)
    bench.dump_outputs(str(tmp_path / "full"), {"sim": sim, "topi": topi})
    a, b = np.load(tmp_path / "full" / "sim.npy"), np.load(tmp_path / "full" / "topi.npy")
    assert a.dtype == np.float32 and np.array_equal(a, sim.numpy())
    assert b.dtype == np.float64 and np.array_equal(b, topi.numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 3 * 4096 + 2000)
    for run in ("one", "two"):
        bench.dump_outputs(str(tmp_path / run), {"sim": sim, "topi": topi})
    files = [tmp_path / "one" / f for f in ("sim.npy", "topi.npy")]
    assert sum(f.stat().st_size for f in files) <= bench.DUMP_LIMIT_BYTES
    s1, s2 = np.load(tmp_path / "one" / "sim.npy"), np.load(tmp_path / "two" / "sim.npy")
    assert 0 < s1.size < sim.numel() and np.array_equal(s1, s2) and np.isin(s1, sim.numpy()).all()
    assert np.array_equal(np.load(tmp_path / "one" / "topi.npy"), topi.numpy())


def test_both_unets_offer_the_interface_the_sharded_sweep_drives():
    """nope_b200.dist.ShardedSweep calls set_metric() and sweep(query_feat=, want_emb=, want_sim=, k=, idx_base=,
    out=) on whichever UNet it is given; the LDM mirror once lagged behind (multi-GPU LDM sweeps raised)."""
    import inspect
    from nope_b200.ldm import UNetModelPose
    from nope_b200.unet import UNet
    need = {"query_feat", "want_emb", "want_sim", "k", "idx_base", "out"}
    for cls in (UNet, UNetModelPose):
        assert callable(getattr(cls, "set_metric", None)), cls.__name__
        params = set(inspect.signature(cls.sweep).parameters)
        assert need <= params, (cls.__name__, sorted(need - params))
