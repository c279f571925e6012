"""CPU: the drop-in boundary -- C-ABI symbols, module interface, registries, host-side data-parallel logic.
No kernel is launched here (there is no GPU in the build container)."""
import io
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from oracle import cnn_linear_oracle as O  # noqa: E402


def test_library_builds_loads_and_exports_every_declared_symbol():
    import __graft_entry__ as g
    g.build()
    from deepards_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "deepards_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(dards_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), "library does not export %s" % name
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared, "ctypes binding and header disagree"
    assert lib.dards_version() == _lib.ABI_VERSION == 8
    # the shared object is self-contained: it must not need libcuda / libcudart at load time
    out = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "libcuda.so" not in out and "libcudart" not in out


def test_argument_validation_returns_error_codes_not_crashes():
    from deepards_b200 import _lib
    lib = _lib.load()
    rc = lib.dards_conv1d_fwd(None, None, None, None, 1, 56, 56, 64, 64, 64, 64, 0, 3, 1, 1, 0, 0, None)
    assert rc == -1 and "null pointer" in _lib.last_error()
    rc = lib.dards_conv1d_fwd(16, 16, 16, None, 1, 56, 55, 64, 64, 64, 64, 0, 3, 1, 1, 0, 0, None)
    assert rc == -1 and "l_out" in _lib.last_error()
    rc = lib.dards_linear_fwd(16, 16, 16, 16, 1, 128, 99, None)
    assert rc == -1
    with pytest.raises(RuntimeError, match="deepards_b200"):
        _lib.call("dards_stem_fwd", 16, 16, 16, 16, 16, 16, 16, 1, 20, 40, 40, 1e-5, 0, None, 0, 0, None)  # C0 = 40 unsupported
    # a BatchNorm group beyond the one-kernel stem needs a workspace: asked for, and refused without one
    assert lib.dards_stem_workspace_bytes(2, 226, 64, 0) == 0 and lib.dards_stem_workspace_bytes(2, 300, 64, 0) == 2 * 5 * 3 * 64 * 4
    with pytest.raises(RuntimeError, match="needs .* bytes of workspace"):
        _lib.call("dards_stem_fwd", 16, 16, 16, 16, 16, 16, 16, 2, 300, 64, 64, 1e-5, 0, None, 0, 0, None)


@pytest.mark.parametrize("backbone", ["resnet18", "densenet18"])
def test_state_dict_keys_shapes_and_module_protocol(backbone):
    import deepards_b200 as D
    bb = getattr(D, backbone)()
    net = D.CNNLinearNetwork(bb, 20, 0)
    ref = O.cnn_linear_state(backbone, seed=0)
    sd = net.state_dict()
    assert list(sd.keys()) == list(ref.keys())  # same names, same order as the reference's modules
    for k in ref:
        assert tuple(sd[k].shape) == tuple(ref[k].shape), k
    net.load_state_dict(ref, strict=True)
    assert net.seq_size == 224 and net.breath_block is bb
    assert bb.network_name == backbone
    assert bb.n_out_filters == (512 if backbone == "resnet18" else 128)
    assert net.linear_final.in_features == 20 * bb.n_out_filters
    assert all(isinstance(p, torch.nn.Parameter) for p in net.parameters())
    if backbone == "densenet18":
        ks, st, pd = bb.conv_info()
        assert len(ks) == len(st) == len(pd) == 2 + 8 * 2 + 3 * 2
        assert bb.drop_rate == 0.2 and isinstance(bb.avgpool, torch.nn.AvgPool1d)
        assert hasattr(bb, "features") and hasattr(bb, "forward_no_pool")
        assert not any(k.endswith("running_mean") for k in sd)
    else:
        assert "breath_block.conv1_alt.weight" in sd and "breath_block.bn2.running_var" in sd
    # picklable as a whole module (train_ards_detector.py:364)
    buf = io.BytesIO()
    torch.save(net, buf)
    buf.seek(0)
    net2 = torch.load(buf, weights_only=False)
    assert list(net2.state_dict().keys()) == list(sd.keys())


def test_init_distribution_matches_reference_recipe():
    import deepards_b200 as D
    torch.manual_seed(0)
    bb = D.resnet18()
    w = bb.layer3[0].conv1.weight
    assert abs(float(w.std()) - (2.0 / (3 * 256)) ** 0.5) < 2e-3  # He-normal, fan = k * Cout (resnet.py:115-118)
    assert float(bb.bn1.weight.min()) == 1.0 and float(bb.bn1.bias.abs().max()) == 0.0


def test_cpu_use_fails_loudly_no_fallback():
    import deepards_b200 as D
    net = D.CNNLinearNetwork(D.resnet18(initial_planes=16), 20, 0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net(torch.zeros(2, 20, 1, 224), None)
    with pytest.raises(Exception, match="sequence length of 224"):
        net(torch.zeros(2, 20, 1, 100), None)
    with pytest.raises(NotImplementedError):
        D.densenet18(with_fft=True)


def test_product_code_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "deepards_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+\.*oracle", src, re.M), "%s imports the oracle" % f
                assert "oracle." not in src and "oracle/" not in src, "%s refers to the oracle" % f
                # the reference tree may be cited in comments, never touched at run time
                assert not re.search(r"(sys\.path|open\(|import_module|CDLL)[^\n]*/root/reference", src), f


def test_registries_and_install():
    import types
    import deepards_b200 as D
    assert set(["resnet18", "densenet18"]) <= set(D.base_networks)
    assert D.network_heads["cnn_linear"] is D.CNNLinearNetwork
    fake = types.ModuleType("train_ards_detector")
    fake.base_networks = {"resnet18": object(), "vgg11": "kept"}
    D.install(fake)
    assert fake.base_networks["resnet18"] is D.resnet18 and fake.base_networks["vgg11"] == "kept"
    assert fake.CNNLinearNetwork is D.CNNLinearNetwork


def test_trainer_calls_build_b200_networks_after_install():
    """What deepards/train_ards_detector.py does with a module patched by install(), replayed with the arguments it passes
    (SURVEY.md, INTEGRATION.md): get_base_network calls resnet18(initial_planes, first_pool_type, double_conv_first)
    (:389-394) or densenet18(with_fft, only_fft, fft_real_only) (:404-409); get_network builds
    CNNLinearNetwork(base, n_sub_batches, n_metadata_inputs) (:938-939) or CNNSingleBreathLinearNetwork(base) (:963-964);
    get_model registers a clamp hook on every parameter (:474-476); get_optimizer hands all parameters to SGD-Nesterov
    (:416-422)."""
    import types
    import deepards_b200 as D
    fake = types.ModuleType("train_ards_detector")
    fake.base_networks = {}
    D.install(fake)
    assert fake.CNNSingleBreathLinearNetwork is D.CNNSingleBreathLinearNetwork
    resnet = lambda: fake.base_networks["resnet18"](initial_planes=64, first_pool_type="max", double_conv_first=False)
    densenet = lambda: fake.base_networks["densenet18"](with_fft=False, only_fft=False, fft_real_only=False)
    for base, get_network, head_cls in ((resnet, lambda bb: fake.CNNLinearNetwork(bb, 20, 0), D.CNNLinearNetwork),
                                        (densenet, lambda bb: fake.CNNLinearNetwork(bb, 20, 0), D.CNNLinearNetwork),
                                        (resnet, fake.CNNSingleBreathLinearNetwork, D.CNNSingleBreathLinearNetwork)):
        bb = base()
        model = get_network(bb)
        assert type(model) is head_cls and model.breath_block is bb
        assert type(bb).__module__.startswith("deepards_b200.")
        for p in model.parameters():
            p.register_hook(lambda grad: torch.clamp(grad, -0.01, 0.01))   # raises for a tensor without requires_grad
        opt = torch.optim.SGD(model.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)
        assert sum(p.numel() for g in opt.param_groups for p in g["params"]) == sum(p.numel() for p in model.parameters())
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            model(torch.zeros(2, 20, 1, 224), None)


def test_shard_bounds_live_ranges_and_buckets():
    from deepards_b200 import data_parallel as dp
    import deepards_b200 as D
    for batch, world in [(256, 8), (10, 4), (3, 8), (16, 1)]:
        spans = [dp.shard_bounds(batch, world, r) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == batch
        assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
        assert max(e - b for b, e in spans) - min(e - b for b, e in spans) <= 1
    net = D.CNNLinearNetwork(D.resnet18(initial_planes=16), 20, 0)
    layout, total = dp.param_layout(net)
    assert all(off % 4 == 0 for _, _, off in layout) and total % 4 == 0
    dead = set(id(p) for n, p in net.named_parameters() if any(s in n for s in (".conv1_alt.", "block.conv2.", "block.bn2.")))
    live = set(id(p) for _, p in net.named_parameters()) - dead
    ranges = dp.live_ranges(layout, live)
    covered = sum(e - b for b, e in ranges)
    assert covered == sum((p.numel() + 3) // 4 * 4 for _, p in net.named_parameters() if id(p) in live)
    assert len(ranges) == 3  # conv1 | bn1 | everything after the unused stem parameters
    buckets = dp.make_buckets(1000, [900, 700, 650, 100], 200)
    assert buckets == [(700, 1000), (100, 700), (0, 100)]
    assert dp.make_buckets(50, [], 10) == [(0, 50)]


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from deepards_b200 import data_parallel as dp
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    flat = torch.arange(1000, dtype=torch.float32) * (rank + 1)
    red = dp.BucketedAllReduce()
    for b, e in dp.make_buckets(1000, [800, 300], 100):
        red.reduce(flat, b, e)
    red.wait()
    q.put((rank, float(flat.sum()), float(flat[999])))
    dist.destroy_process_group()


def test_bucketed_allreduce_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    expect_sum = float(torch.arange(1000, dtype=torch.float32).sum()) * 3
    for rank, s, last in res:
        assert abs(s - expect_sum) < 1e-3 and last == 999 * 3


def _gloo_map_worker(rank, world, port, q):
    import torch.distributed as dist
    from deepards_b200 import data_parallel as dp
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    res = {}
    for n in (5, 1, 4):                                  # ragged, fewer sequences than ranks, even
        x = torch.arange(n * 3, dtype=torch.float32).view(n, 3)
        maps, logits = dp.sharded_map(lambda s: ((s * 2).to(torch.uint8), s.sum(1, keepdim=True) + 100 * rank), x)
        res[n] = (maps.tolist(), logits.view(-1).tolist())
    q.put((rank, res))
    dist.destroy_process_group()


def test_sharded_replicas_world2_gloo():
    """configs[3]/[4] on several GPUs = independent replicas over contiguous shards of the sequences + an ordered
    gather of the per-sequence results; no collective on the data path."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_map_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res[0] == res[1]                              # every rank holds the full, ordered result
    for n in (5, 1, 4):
        x = torch.arange(n * 3, dtype=torch.float32).view(n, 3)
        maps, logits = res[0][n]
        assert maps == (x * 2).to(torch.uint8).tolist()
        owner = [0 if i < (n + 1) // 2 else 1 for i in range(n)]      # shard_bounds: remainder to the first ranks
        assert logits == [float(x[i].sum()) + 100 * owner[i] for i in range(n)]


def test_sibling_heads_gradcam_and_scaler_boundary_on_cpu():
    """The rows added after the core path keep the reference's names / state_dict keys and fail loudly off the GPU."""
    import types
    import numpy as np
    import deepards_b200 as D
    from deepards_b200 import gradcam as G
    z = np.load(os.path.join(ROOT, "tests", "golden", "sibling_heads.npz"))
    bb = D.resnet18(initial_planes=16)
    heads = {"to_mean": D.CNNLinearToMean(bb), "compr_to_rf": D.CNNLinearComprToRF(bb),
             "double_linear": D.CNNDoubleLinearNetwork(bb, 20, 0), "regressor": D.CNNRegressor(bb, 3),
             "lstm": D.CNNLSTMNetwork(bb, 0, False, 32)}
    for kind, net in heads.items():
        assert list(net.state_dict().keys()) == list(z[kind + "/keys"]), kind    # recorded from the reference's modules
        assert net.seq_size == 224 and net.breath_block is bb
    with pytest.raises(Exception, match="sequence length of 224"):
        heads["to_mean"](torch.zeros(2, 20, 1, 100), None)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        heads["double_linear"](torch.zeros(2, 20, 1, 224), None)
    with pytest.raises(NotImplementedError):
        D.CNNLSTMNetwork(bb, 3, False, 32)
    fake = types.ModuleType("train_ards_detector")
    fake.base_networks = {}
    D.install(fake)
    for name in ("CNNLinearToMean", "CNNLinearComprToRF", "CNNDoubleLinearNetwork", "CNNRegressor", "CNNLSTMNetwork"):
        assert getattr(fake, name) is getattr(D, name)
    assert D.network_heads["cnn_lstm"] is D.CNNLSTMNetwork
    # GradCAM: same class names and methods as deepards/gradcam.py; DenseNet only; never a CPU path
    for cls in ("GradCam", "MaxMinNormCam", "UnNormalizedCam", "FracTotalNormCam"):
        assert hasattr(getattr(G, cls), "generate_one_hot_grad_and_output")
    assert hasattr(G.MaxMinNormCam, "generate_cam") and hasattr(G.MaxMinNormCam, "generate_read_cam")
    with pytest.raises(TypeError, match="DenseNet"):
        G.MaxMinNormCam(D.CNNLinearNetwork(bb, 20, 0)).generate_cam(torch.zeros(20, 1, 224))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        G.MaxMinNormCam(D.CNNLinearNetwork(D.densenet18(), 20, 0)).generate_cam(torch.zeros(20, 1, 224))
    with pytest.raises(NotImplementedError):
        G.FracTotalNormCam(None).generate_cam(None, 0)
    # window scaling: the padded rule follows the dataset type string; host tensors need an explicit device
    assert D.WindowScaler.for_dataset_type(2.0, 28.0, "padded_breath_by_breath_with_full_bm_target").padded
    assert not D.WindowScaler.for_dataset_type(2.0, 28.0, "unpadded_centered_sequences").padded
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        D.WindowScaler(2.0, 28.0)(torch.zeros(2, 224, dtype=torch.float64))
    with pytest.raises(ValueError):
        D.WindowScaler(2.0, 0.0)
    with pytest.raises(TypeError):
        D.WindowScaler(2.0, 28.0)(torch.zeros(2, 224, dtype=torch.int16))


def test_data_parallel_marks_are_bucket_sized():
    """engine.Plan.mark: a mark (= a partial-sum reduction launch + a graph boundary in the multi-GPU step) only where
    at least one 1 MB bucket of gradients has become final; the trainer's buckets are cut at marks only.  The LAST bucket
    (all-reduce + optimizer update on the step's tail, nothing left to overlap them with) stays small."""
    from deepards_b200 import data_parallel as dp, engine
    assert engine.DP_MARK_ELEMS == 1 << 30      # default: one bucket after the backward (measured faster on NVSwitch)
    mark_elems = 1 << 18                         # the overlapped schedule (DEEPARDS_B200_DP_BUCKET_ELEMS=262144)
    # ResNet-18 slot offsets of the first parameter of each block, last block first (3.89 M elements in total)
    total = 3_893_378
    offs = [2_318_000, 1_006_000, 612_000, 283_000, 185_000, 103_000, 78_000, 53_000]
    marks, last = [], total
    for off in offs:                       # the rule of Plan.mark
        if last - off >= mark_elems:
            marks.append(off)
            last = off
    assert marks == [2_318_000, 1_006_000, 612_000, 283_000]
    assert dp.make_buckets(total, marks, 1 << 18) == [(2_318_000, total), (1_006_000, 2_318_000), (612_000, 1_006_000),
                                                      (283_000, 612_000), (0, 283_000)]
    assert dp.make_buckets(214_850, [], 1 << 18) == [(0, 214_850)]          # DenseNet-18: one bucket


def test_benchmark_workload_generator_equals_the_oracles():
    """bench.py's product arm takes its synthetic batches from deepards_b200.synthetic (so that it imports nothing from
    oracle/); the oracle's own generator, used by the parity tests, must produce the same tensors bit for bit."""
    import torch
    from deepards_b200 import synthetic as S
    from oracle import cnn_linear_oracle as O
    for seed in (1234, 77):
        assert torch.equal(S.synthetic_breaths(3, seed=seed), O.synthetic_breaths(3, seed=seed))
        assert torch.equal(S.synthetic_targets(5, seed=seed), O.synthetic_targets(5, seed=seed))
    src = open(os.path.join(ROOT, "bench.py")).read()
    b200_arm = src[src.index("def run_b200"):src.index("def kernel_roofline")]
    # the only oracle use inside the product arm is the cpu_baseline leg (cpu_reference_steps), never an import
    assert "from oracle" not in b200_arm and "import oracle" not in b200_arm
