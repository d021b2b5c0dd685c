"""Host-side checks of the training harness (no GPU): model shapes the hot path sees,
loss formula, schedules, and the N>1 data-parallel plumbing on gloo with world_size 2."""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp
import torch.nn.functional as F

from quantized_distillation_b200.cnn_models import conv_forward_model as cfm
from quantized_distillation_b200.cnn_models import help_fun as hf
from quantized_distillation_b200.cnn_models.wide_resnet import Wide_ResNet


def student():
    spec = dict(cfm.smallerModelSpec)
    spec["spec_dropout_rates"] = []
    return cfm.ConvolForwardNet(**spec, useBatchNorm=True, useAffineTransformInBatchNorm=True)


def test_student_parameter_list_matches_survey():
    m = student()
    sizes = [p.numel() for p in m.parameters()]
    assert len(sizes) == 22 and sum(sizes) == 1_000_235          # SURVEY.md section 8
    assert sizes[0] == 5000 and sizes[1] == 10                     # out_layer registered first
    assert sizes[2] == 5625 and sizes[10] == 800_000
    sel = cfm._selected_parameters(m, False)
    assert len(sel) == 20 and sel[0].numel() == 10
    teacher = cfm.ConvolForwardNet(**cfm.teacherModelSpec, useBatchNorm=True, useAffineTransformInBatchNorm=True)
    assert sum(p.numel() for p in teacher.parameters()) == 5_346_142


def test_wrn_16_22_parameter_list_matches_survey():
    m = Wide_ResNet(depth=16, widen_factor=22, dropout_rate=0.3, num_classes=10)
    sizes = [p.numel() for p in m.parameters()]
    assert len(sizes) == 60 and sum(sizes) == 82_746_890
    assert sizes[0] == 432 and sizes[-1] == 10 and max(sizes) == 17_842_176
    with pytest.raises(ValueError):
        Wide_ResNet(depth=17, widen_factor=2, dropout_rate=0.0, num_classes=10)


def test_forward_shapes_and_distillation_loss_formula():
    torch.manual_seed(0)
    m = student()
    x = torch.randn(4, 3, 32, 32)
    y = torch.randint(0, 10, (4,))
    assert m(x).shape == (4, 10)
    out, t_out = torch.randn(4, 10), torch.randn(4, 10)
    T = 2
    kl = F.kl_div(F.log_softmax(out / T, dim=1), F.softmax(t_out / T, dim=1), reduction="sum") / out.numel()
    expect = 0.7 * T * T * kl + 0.3 * F.cross_entropy(out, y)
    assert torch.allclose(hf.distillation_loss(out, y, t_out), expect)
    teacher = student().eval()
    loss, asked, total = hf.forward_and_backward(m, (x, y), 1, 0, use_distillation_loss=True, teacher_model=teacher,
                                                 return_more_info=True)
    assert isinstance(loss, float) and asked == 4 and total == 4
    assert all(p.grad is not None for p in m.parameters())
    with pytest.raises(ValueError):
        hf.forward_and_backward(m, (x, y), 1, 0, use_distillation_loss=True)
    for strat in (("incorrect_labels", None), ("cutoff_entropy", 1.0), ("random_entropy", None)):
        m.zero_grad()
        hf.forward_and_backward(m, (x, y), 1, 0, use_distillation_loss=True, teacher_model=teacher, ask_teacher_strategy=strat)


def test_learning_rate_schedules():
    s = hf.LearningRateScheduler(0.1, "cifar100")
    assert s.update_learning_rate(10, 0.5)[0] == 0.1
    assert abs(s.update_learning_rate(61, 0.5)[0] - 0.02) < 1e-12
    assert abs(s.update_learning_rate(161, 0.5)[0] - 0.1 * 0.2 ** 3) < 1e-12
    g = hf.LearningRateScheduler(1.0, "generic")
    lr = 1.0
    for epoch in range(12):
        lr, stop = g.update_learning_rate(epoch, 0.5)
    assert lr == 0.5 and stop is False
    with pytest.raises(ValueError):
        hf.LearningRateScheduler(0.1, "cosine")


def test_train_model_without_quantization_runs_on_cpu():
    torch.manual_seed(0)
    m = student()
    data = hf.synthetic_cifar_loader(3, 4, pin=False)
    model, info = cfm.train_model(m, data, data, epochs_to_train=1, print_every=1, verbose=False)
    assert info["numStepsTrained"] == 3 and info["errorFlag"] is False and len(info["predictionAccuracy"]) == 1
    with pytest.raises(ValueError):
        cfm.train_model(m, data, data, use_distillation_loss=True)


def test_weight_quantizer_nmt_loop_options_choreography(monkeypatch):
    """The options only the NMT loop passes (translation_models/model.py:162-164, 198-204, 247-279: stochastic rounding,
    max_element, subtract_mean) select WeightQuantizer's per-tensor path.  Its save / quantize-in-place / restore /
    truncated fix-up choreography is host logic: checked here with the fused op replaced by the oracle (the op itself
    with these options is GPU-tested in tests/test_gpu_parity.py)."""
    import numpy as np
    from oracle import quant_oracle as O
    seen = []

    def oracle_op(tensor, s, type_of_scaling="linear", stochastic_rounding=False, max_element=False, subtract_mean=False,
                  bucket_size=None, modify_in_place=False):
        seen.append((type_of_scaling, stochastic_rounding, max_element, subtract_mean, bucket_size, modify_in_place))
        q = O.uniform_fwd(tensor.numpy().reshape(-1), s, bucket_size, subtract_mean=subtract_mean, max_element=max_element)[0]
        tensor.copy_(torch.from_numpy(np.ascontiguousarray(q)).view(tensor.shape))
        return tensor, None

    monkeypatch.setattr(cfm.quantization, "uniformQuantization", oracle_op)
    torch.manual_seed(3)
    model = student()
    params = list(model.parameters())
    with torch.no_grad():
        params[2].view(-1)[:7] = 3.0                                 # 'truncated' clamps the weights to [-1, 1] first (:240-241)
    wq = cfm.WeightQuantizer(model, numBits=4, bucket_size=256, backprop_quantization_style="truncated",
                             quantize_first_and_last_layer=False, max_element=0.5, subtract_mean=True)
    assert wq.plan is None and len(wq.params) == len(params) - 2
    before = [p.detach().clone() for p in params]
    wq.quantize_weights_model()
    assert len(seen) == len(wq.params) and all(c == ("linear", False, 0.5, True, 256, True) for c in seen)
    for i, (p, o) in enumerate(zip(params, before)):
        if i in (0, len(params) - 1):
            assert torch.equal(p, o)                                  # first / last tensor left alone (:237-239)
        else:
            want = O.uniform_fwd(o.clamp(-1, 1).numpy().reshape(-1), 16, 256, subtract_mean=True, max_element=0.5)[0]
            assert np.array_equal(p.detach().numpy().reshape(-1).view(np.uint32), np.asarray(want).reshape(-1).view(np.uint32))
    wq.restore_weights_model()
    for i, (p, o) in enumerate(zip(params, before)):
        assert torch.equal(p, o if i in (0, len(params) - 1) else o.clamp(-1, 1))     # the clamp persists, like in the reference
    with torch.no_grad():
        params[3].view(-1)[:5] = -2.0
    for p in params:
        p.grad = torch.ones_like(p)
    wq.backward_quant_weights_model()                                 # p.grad[|p| > 1] = 0 (:263-264)
    assert float(params[3].grad.view(-1)[:5].abs().sum()) == 0.0 and float(params[3].grad.sum()) == params[3].numel() - 5
    assert all(bool((p.grad == 1).all()) for i, p in enumerate(params) if i != 3)
    # stochastic rounding is passed through; 'complicated' refuses the three options like the reference's backward does
    seen.clear()
    cfm.WeightQuantizer(model, 2, 256, stochastic_rounding=True).quantize_weights_model(save=False)
    assert seen and all(c[1] is True and c[2] is False and c[3] is False for c in seen)
    for opt in ({"stochastic_rounding": True}, {"max_element": 1.0}, {"subtract_mean": True}):
        with pytest.raises(NotImplementedError):
            cfm.WeightQuantizer(model, 4, 256, backprop_quantization_style="complicated", **opt)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _spawn_host_ranks(fn, args, world):
    """Starts the ranks with CUDA_VISIBLE_DEVICES empty, so that they are host processes on any machine (with one GPU,
    rank 1 would otherwise ask for cuda:1).  It is set before they start: importing the package already queries CUDA."""
    saved = os.environ.get("CUDA_VISIBLE_DEVICES")
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    try:
        mp.spawn(fn, args=args, nprocs=world, join=True)
    finally:
        if saved is None:
            del os.environ["CUDA_VISIBLE_DEVICES"]
        else:
            os.environ["CUDA_VISIBLE_DEVICES"] = saved


def _ddp_worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    from quantized_distillation_b200 import distributed as D
    w, r, device = D.init_distributed(backend="gloo")
    torch.manual_seed(1234)                                        # same init on every rank
    model = D.wrap_ddp(student(), device)
    global_batches = hf.synthetic_cifar_loader(2, 8, seed=7, pin=False)
    local = D.shard_batches(global_batches, r, w)
    assert local[0][0].size(0) == 4
    cfm.train_model(model, local, local, epochs_to_train=1, print_every=1, verbose=False, evaluate=False)
    flat = torch.cat([p.detach().view(-1) for p in model.parameters()])
    gathered = [torch.zeros_like(flat) for _ in range(w)]
    torch.distributed.all_reduce(flat.clone())                     # exercises the collective path
    torch.distributed.all_gather(gathered, flat)
    ret[rank] = bool(torch.equal(gathered[0], gathered[1]))
    assert D.max_over_ranks(float(r), device) == w - 1
    torch.distributed.destroy_process_group()


def test_ddp_replicas_stay_identical_gloo_world2():
    """N>1 path on CPU: two gloo ranks, sharded global batch, DDP gradient all-reduce;
    after training the replicas hold bit-identical parameters."""
    world = 2
    port = _free_port()
    with mp.Manager() as mgr:
        ret = mgr.dict()
        _spawn_host_ranks(_ddp_worker, (world, port, ret), world)
        assert ret[0] is True and ret[1] is True


def _student_no_bn():
    spec = dict(cfm.smallerModelSpec)
    spec["spec_dropout_rates"] = []
    return cfm.ConvolForwardNet(**spec, useBatchNorm=False)


def _flat_worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    from quantized_distillation_b200 import distributed as D
    w, r, device = D.init_distributed(backend="gloo")
    torch.manual_seed(1234 + r)                                    # DIFFERENT init per rank: the wrapper must broadcast rank 0's
    # 0.25 MB buckets: the 4 MB gradient buffer is cut into several, each reduced from a post-accumulate-grad hook
    model = D.wrap_data_parallel(_student_no_bn(), device, bucket_mb=0.25)
    assert isinstance(model, D.FlatDataParallel) and model.views_intact()
    assert len(model._buckets) > 3 and model._early
    assert model._buckets[0]["lo"] == 0 and model._buckets[-1]["hi"] == model.flat_grad.numel()
    assert all(a["hi"] == b["lo"] for a, b in zip(model._buckets, model._buckets[1:]))
    lo = model.flat_grad.data_ptr()
    assert all((p.grad.data_ptr() - lo) % 256 == 0 for p in model.parameters())   # 128-bit kernels need aligned rows
    global_batches = hf.synthetic_cifar_loader(3, 8, seed=7, pin=False)
    local = D.shard_batches(global_batches, r, w)
    cfm.train_model(model, local, local, epochs_to_train=1, print_every=1, verbose=False, evaluate=False)
    assert model.views_intact()                                    # the optimizer never replaced a gradient tensor
    flat = torch.cat([p.detach().view(-1) for p in model.parameters()])
    gathered = [torch.zeros_like(flat) for _ in range(w)]
    torch.distributed.all_gather(gathered, flat)
    ok = bool(torch.equal(gathered[0], gathered[1]))
    if r == 0:
        ret["params"] = flat.clone()
    # two hand-written steps that clear the gradients through the OPTIMIZER, never through the wrapper's
    # zero_grad(): reduce_gradients() itself re-arms the buckets, so the second step is reduced as well
    opt = torch.optim.SGD(model.parameters(), lr=0.0)
    for step in range(2):
        opt.zero_grad(set_to_none=False)
        x, y = local[step]
        F.cross_entropy(model(x), y).backward()
        model.reduce_gradients()
        assert all(b["sent"] is False and b["pending"] == len(b["members"]) for b in model._buckets)
        g = model.flat_grad.clone()
        both = [torch.zeros_like(g) for _ in range(w)]
        torch.distributed.all_gather(both, g)
        ok = ok and bool(torch.equal(both[0], both[1])) and bool(g.abs().sum() > 0)
    ret[rank] = ok
    torch.distributed.destroy_process_group()


def test_flat_data_parallel_gloo_world2_matches_single_process():
    """FlatDataParallel: one flat gradient buffer, one all-reduce per step.  Two gloo ranks on the
    two halves of each global batch end bit-identical to each other and equal (to float32
    summation order) to a single process that saw the whole batches with rank 0's start; the model
    has no batch-norm here, whose statistics are per replica by design."""
    world = 2
    port = _free_port()
    with mp.Manager() as mgr:
        ret = mgr.dict()
        _spawn_host_ranks(_flat_worker, (world, port, ret), world)
        assert ret[0] is True and ret[1] is True
        dp = ret["params"]
    torch.manual_seed(1234)
    single = _student_no_bn()
    batches = hf.synthetic_cifar_loader(3, 8, seed=7, pin=False)
    cfm.train_model(single, batches, batches, epochs_to_train=1, print_every=1, verbose=False, evaluate=False)
    ref = torch.cat([p.detach().view(-1) for p in single.parameters()])
    assert torch.allclose(dp, ref, atol=2e-6, rtol=1e-4), float((dp - ref).abs().max())


def test_state_dict_prefix_helpers():
    from quantized_distillation_b200 import distributed as D
    sd = student().state_dict()
    wrapped = D.convert_state_dict_to_data_parallel(sd)
    assert all(k.startswith("module.") for k in wrapped)
    assert list(D.convert_state_dict_from_data_parallel(wrapped)) == list(sd)
    with pytest.raises(ValueError):
        D.shard_batches([(torch.zeros(5, 3), torch.zeros(5))], 0, 2)


def test_models_match_reference_built_fixtures():
    """ConvolForwardNet / Wide_ResNet against the reference's own classes (tests/golden/make_golden_models.py builds them
    from /root/reference in small configurations): same parameter and state-dict order -- the hot path quantizes
    ``parameters()`` in that order and ``quantize_first_and_last_layer=False`` skips its first and last entry -- the
    reference's weights load with strict=True, and the logits agree in eval() and train() mode, running statistics included."""
    import numpy as np
    data = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_models.npz"))
    small = {"spec_conv_layers": [(6, 3, 3), (8, 5, 5), (8, 3, 3)], "spec_max_pooling": [(0, 2, 2), (2, 2, 2)],
             "spec_dropout_rates": [], "spec_linear": [24, 12], "width": 16, "height": 16}
    builds = {"conv_bn_affine": lambda: cfm.ConvolForwardNet(**small, useBatchNorm=True, useAffineTransformInBatchNorm=True),
              "conv_bn": lambda: cfm.ConvolForwardNet(**small, useBatchNorm=True, useAffineTransformInBatchNorm=False),
              "conv_plain": lambda: cfm.ConvolForwardNet(**small, useBatchNorm=False),
              "wrn_10_1": lambda: Wide_ResNet(depth=10, widen_factor=1, dropout_rate=0.0, num_classes=10)}
    for tag, build in builds.items():
        m = build()
        assert [n for n, _ in m.named_parameters()] == list(data[tag + "_param_names"]), tag
        assert list(m.state_dict().keys()) == list(data[tag + "_state_names"]), tag
        sd = {k: torch.from_numpy(data[f"{tag}_sd_{k}"].copy()) for k in data[tag + "_state_names"]}
        m.load_state_dict(sd, strict=True)
        x = torch.from_numpy(data[tag + "_x"])
        m.eval()
        with torch.no_grad():
            y = m(x).numpy()
        assert np.array_equal(y, data[tag + "_y_eval"]), (tag, float(np.abs(y - data[tag + "_y_eval"]).max()))
        m.train()
        with torch.no_grad():
            y = m(x).numpy()
        assert np.array_equal(y, data[tag + "_y_train"]), (tag, float(np.abs(y - data[tag + "_y_train"]).max()))
        for k, v in m.state_dict().items():
            if "running" in k or "num_batches" in k:
                assert np.array_equal(v.numpy(), data[f"{tag}_after_{k}"]), (tag, k)
    assert repr(cfm.teacherModelSpec) == str(data["teacherModelSpec"]) and repr(cfm.smallerModelSpec) == str(data["smallerModelSpec"])
