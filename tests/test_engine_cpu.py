"""passl_b200/engine/engine.py (the v2.5 `Engine` surface) on CPU: config -> model / optimizer / schedule wiring, the loop's ordering
of optimizer step and schedule step (the reference reads get_lr() and then calls lr_step(global_step), optimizer.py:117-123,216-222),
max_train_step, checkpoint files and resume.  Kernels are not run here: the model / optimizer are stubbed where a step is taken."""
import functools
import os
import pickle

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
CFG = os.path.join(os.path.dirname(HERE), "configs/mocov3/mocov3_vit_base_patch16_224_pt.yaml")


def _tiny_factory(**kw):
    from passl_b200.models.mocov3 import MoCoV3Pretrain, MoCoV3ViT
    enc = functools.partial(MoCoV3ViT, img_size=32, patch_size=8, embed_dim=64, depth=1, num_heads=2, qkv_bias=True, stop_grad_conv1=True)
    return MoCoV3Pretrain(enc, dim=32, mlp_dim=48, T=0.2, **kw)


@pytest.fixture()
def engine(monkeypatch, tmp_path):
    import passl_b200.models as M
    from passl_b200.engine.engine import Engine
    from passl_b200.utils.config import get_config
    monkeypatch.setattr(M, "tiny_mocov3_pretrain", _tiny_factory, raising=False)
    cfg = get_config(CFG, ["Model.name=tiny_mocov3_pretrain", "Global.epochs=3", "Global.max_train_step=null", "Global.save_interval=2",
                           "Global.output_dir=%s" % tmp_path, "DataLoader.Train.synthetic_steps=4", "DataLoader.Train.sampler.batch_size=8",
                           "LRScheduler.warmup_epoch=1", "Global.print_batch_step=100"])
    cfg["Global"]["max_train_step"] = None
    return Engine(cfg, device="cpu", dataloader=[[None, None]] * 4)


def test_config_wiring(engine):
    from passl_b200.optimizer import AdamW
    from passl_b200.optimizer.lr import TimmCosine
    e = engine
    assert type(e.model).__name__ == "MoCoV3Pretrain" and e.model.max_steps == 12 == e.max_steps
    assert isinstance(e.lr_scheduler, TimmCosine) and (e.lr_scheduler.T_max, e.lr_scheduler.warmup_steps) == (12, 4) and e.lr_decay_unit == "step"
    assert isinstance(e.optimizer, AdamW) and (e.optimizer.beta1, e.optimizer.beta2, e.optimizer.eps) == (0.9, 0.999, 1e-8)
    assert e.optimizer.lr == 0.0                                                       # warm-up start
    by_name = dict(zip(e.store.names, e.optimizer.seg_wd.tolist()))
    assert by_name["0.vit.pos_embed"] == 0 and by_name["0.vit.patch_embed.proj.weight"] == 0        # frozen: no step, no decay
    assert abs(by_name["0.vit.blocks.0.norm1.weight"] - 0.1) < 1e-7 and abs(by_name["1.fcs.0.weight"] - 0.1) < 1e-7   # everything else decays
    assert e.batch_size == 8


def test_loop_order_checkpoints_and_resume(engine, monkeypatch):
    e = engine

    class _Loss:
        def backward(self):
            pass

        def detach(self):
            return torch.tensor(1.25)

    used = []

    class _Opt:
        lr = 0.0

        def set_lr(self, v):
            self.lr = v

        def get_lr(self):
            return self.lr

        def step(self):
            used.append(self.lr)

        def clear_grad(self):
            pass

        def state_dict(self):
            return {"step": len(used), "lr": self.lr}

        def set_state_dict(self, st):
            self.restored = st
    real_model = e.model
    e.optimizer = _Opt()
    monkeypatch.setattr(type(real_model), "forward", lambda self, batch: _Loss())
    assert e.train() == 12
    G = np.load(os.path.join(HERE, "golden", "reference_lr.npz"))
    sched = e.lr_scheduler
    assert np.allclose(used, [sched.lr_at(k - 1) for k in range(1, 13)], rtol=0, atol=0)   # step k runs at lr_at(k - 1)
    assert used[0] == 0.0 and used[4] == pytest.approx(0.0024) and used[-1] < used[5]
    assert G["timm_step_prefix"].shape == (66,)                                            # protocol pinned in tests/test_lr_cpu.py
    base = os.path.join(e.output_dir, "tiny_mocov3_pretrain")
    assert sorted(os.listdir(base)) == sorted(["epoch_2.pdparams", "epoch_2_base_encoder.pdparams", "epoch_2.pdstates", "epoch_2.opt.pt",
                                               "epoch_3.pdparams", "epoch_3_base_encoder.pdparams", "epoch_3.pdstates", "epoch_3.opt.pt"])
    meta = pickle.load(open(os.path.join(base, "epoch_2.pdstates"), "rb"))
    assert (meta["epoch"], meta["global_step"]) == (2, 8)
    from passl_b200.utils import checkpoint as C
    trunk = C.load_pdparams(os.path.join(base, "epoch_3_base_encoder.pdparams"))
    assert "blocks.0.attn.qkv.weight" in trunk and not any(k.startswith("head") for k in trunk)
    with torch.no_grad():
        for p in real_model.parameters():
            p.add_(1.0)
    e.resume(os.path.join(base, "epoch_2"))
    assert (e.cur_epoch_id, e.global_step) == (2, 8) and e.lr_scheduler.last_epoch == 8 and e.optimizer.restored["step"] == 8
    full = C.load_pdparams(os.path.join(base, "epoch_2.pdparams"))
    assert np.array_equal(C.to_paddle_state(real_model)["predictor.0.weight"], full["predictor.0.weight"])
    used.clear()
    assert e.train() == 12 and len(used) == 4                                              # only the third epoch is left


def test_max_train_step_and_unbuilt_options(engine, monkeypatch):
    from passl_b200.engine.engine import Engine
    from passl_b200.utils.config import get_config
    e = engine
    e.max_train_step = 5
    e.optimizer = type("O", (), dict(lr=0.0, set_lr=lambda s, v: None, get_lr=lambda s: 0.0, step=lambda s: None, clear_grad=lambda s: None,
                                     state_dict=lambda s: {}))()
    monkeypatch.setattr(type(e.model), "forward", lambda self, batch: type("L", (), dict(backward=lambda s: None, detach=lambda s: torch.tensor(0.5)))())
    assert e.train() == 5
    assert Engine(get_config(CFG, ["Global.accum_steps=2"]), device="cpu").accum_steps == 2      # gradient merge is built
    with pytest.raises(NotImplementedError):
        Engine(get_config(CFG, ["Optimizer.layer_decay=0.75"]), device="cpu")
    Engine(get_config(CFG, ["Optimizer.tensor_fusion=False"]), device="cpu")                     # falsy = not requested
    with pytest.raises(NotImplementedError):
        Engine(get_config(CFG, []), mode="eval", device="cpu")


def test_mae_pretrain_entry_arguments_and_rates():
    """tools/mae_pretrain.py: the reference's argument names and its lr = blr * total batch / 256 rule (main_pretrain.py:239-243)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("mae_pretrain", os.path.join(os.path.dirname(HERE), "tools", "mae_pretrain.py"))
    M = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(M)
    a = M.get_args_parser().parse_args(["--batch_size", "512", "--blr", "1.5e-4", "--norm_pix_loss", "--mask_ratio", "0.75"])
    assert M.effective_lr(a, 8) == (1.5e-4 * 4096 / 256, 4096) and a.norm_pix_loss and a.model == "mae_vit_base_patch16"
    assert (a.weight_decay, a.warmup_epochs, a.min_lr, a.input_size) == (0.05, 40, 0.0, 224)
    assert M.effective_lr(M.get_args_parser().parse_args(["--lr", "0.001"]), 2) == (0.001, 128)


def test_profiler_options_and_step_window(tmp_path):
    """utils/profiler.py: the reference's option-string grammar (profiler.py:46-72) and the step window, on a recording backend."""
    from passl_b200.utils.profiler import ProfilerOptions, StepProfiler
    o = ProfilerOptions("batch_range=[3, 5]; tracer_option=OpDetail; profile_path=%s; exit_on_finished=false" % (tmp_path / "p.txt"))
    assert o["batch_range"] == [3, 5] and o["tracer_option"] == "OpDetail" and o["exit_on_finished"] is False and o["state"] == "All"
    assert ProfilerOptions("batch_range=[7,2]")["batch_range"] == [10, 20]                 # invalid range: default kept
    with pytest.raises(ValueError):
        o["no_such_key"]
    events = []

    class _Rec:
        class nvtx:
            range_push = staticmethod(lambda name: events.append(("push", name)))
            range_pop = staticmethod(lambda: events.append(("pop",)))

        class profiler:
            start = staticmethod(lambda: events.append(("start",)))
            stop = staticmethod(lambda: events.append(("stop",)))
        synchronize = staticmethod(lambda: None)
    p = StepProfiler("batch_range=[3, 5]; profile_path=%s; exit_on_finished=false" % (tmp_path / "p.txt"), backend=_Rec)
    for _ in range(8):
        p.step()
    assert events == [("start",), ("push", "step_3"), ("pop",), ("push", "step_4"), ("pop",), ("stop",)]
    assert "profiled steps [3, 5)" in open(tmp_path / "p.txt").read()
    q = StepProfiler("batch_range=[0, 1]; profile_path=%s" % (tmp_path / "q.txt"), backend=_Rec)
    q.step()
    with pytest.raises(SystemExit):
        q.step()
    StepProfiler(None).step()                                                             # disabled: no-op


def test_bench_prints_exactly_one_json_line_on_stdout():
    """bench.py's contract: ONE JSON line on stdout (library banners and progress go to stderr).  The reference arm of a config
    without a CPU port is the cheapest path through main()."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--config", "c4"], capture_output=True,
                       text=True, cwd=root, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and "unavailable" in d


def test_bench_dump_outputs_is_seeded_and_bounded(tmp_path):
    """--dump-outputs writes loss / params / grads as float32; a buffer longer than DUMP_SAMPLE is sampled at the same positions
    in every run (the master and gradient buffers at identical indices)."""
    import types
    import bench
    n = bench.DUMP_SAMPLE + 12345
    master = torch.arange(n, dtype=torch.float32)
    store = types.SimpleNamespace(numel=n, master=master, grad=-master)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), torch.tensor([2.5]), store)
    got = {f: np.load(tmp_path / "a" / (f + ".npy")) for f in ("loss", "params", "grads")}
    assert all(v.dtype == np.float32 for v in got.values())
    assert got["loss"].shape == () and float(got["loss"]) == 2.5
    p = got["params"]
    assert p.shape == (bench.DUMP_SAMPLE,) and np.all(np.diff(p) > 0) and p[-1] < n
    assert np.array_equal(got["grads"], -p)
    assert all(np.array_equal(v, np.load(tmp_path / "b" / (f + ".npy"))) for f, v in got.items())
    small = types.SimpleNamespace(numel=5, master=master[:5], grad=master[:5])
    bench.dump_outputs(str(tmp_path / "c"), torch.tensor(1.0), small)
    assert np.array_equal(np.load(tmp_path / "c" / "params.npy"), master[:5].numpy())
