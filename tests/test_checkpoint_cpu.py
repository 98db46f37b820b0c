"""Paddle-checkpoint name / layout mapping (passl_b200/utils/checkpoint.py) checked against the reference classes themselves: the
reference's ResNet-50 (resnetimagenet.py) and NonLinearNeckV1 (base_neck.py) were constructed over the paddle shim — no weights
needed, only their parameter / buffer names and shapes, stored in tests/golden/reference_checkpoint_names.npz by
tests/golden/make_golden_checkpoint.py — and must equal what `moco_to_paddle` emits."""
import os

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))


def _model():
    from passl_b200.modeling import build_model
    from passl_b200.utils.config import get_config
    cfg = get_config(os.path.join(os.path.dirname(HERE), "configs/moco/moco_v2_r50.yaml"), ["model.K=512"])
    return build_model(dict(cfg.model))


def test_roundtrip_and_file_container(tmp_path):
    from passl_b200.utils import checkpoint as C
    torch.manual_seed(0)
    a, b = _model(), _model()
    for p in a.parameters():
        torch.nn.init.normal_(p, std=0.1)
    for n, buf in a.named_buffers():
        if buf.dtype.is_floating_point:
            buf.normal_()
    a.queue_ptr.fill_(128)
    state = C.moco_to_paddle(a)
    assert state["queue"].shape == (128, 512) and state["encoder_q.0.conv1.weight"].shape == (64, 3, 7, 7)
    assert state["encoder_q.1.mlp.0.weight"].shape == (2048, 2048) and state["encoder_q.1.mlp.2.weight"].shape == (2048, 128)
    path = str(tmp_path / "epoch_1.pdparams")
    C.save_pdparams(state, path)
    C.moco_from_paddle(b, C.load_pdparams(path))
    sa, sb = a.state_dict(), b.state_dict()
    for k in sa:
        if k.endswith("stem.weight"):
            assert torch.equal(sa[k][:, :147], sb[k][:, :147]) and sb[k][:, 147:].abs().sum() == 0
        else:
            assert torch.equal(sa[k], sb[k]), k


def _ref_names(group):
    """{name: shape} of one model's state_dict as the reference classes build it (tests/golden/make_golden_checkpoint.py)."""
    G = np.load(os.path.join(HERE, "golden", "reference_checkpoint_names.npz"))
    return {k[len(group) + 1:]: tuple(int(d) for d in G[k]) for k in G.files if k.startswith(group + ":")}, G


def test_names_and_shapes_equal_the_reference_classes():
    want, _ = _ref_names("moco")
    from passl_b200.utils import checkpoint as C
    got = {k: tuple(v.shape) for k, v in C.moco_to_paddle(_model()).items() if k.startswith("encoder_q.")}
    assert set(got) == set(want), (sorted(set(want) - set(got))[:5], sorted(set(got) - set(want))[:5])
    for k in want:
        assert got[k] == want[k], (k, got[k], want[k])


# ------------------------------------------------------------------ ViT families: MAE, CLIP, MoCo v3 ------------------------------
GOLD = os.path.join(HERE, "golden")


def _ref_weights(npz):
    G = np.load(os.path.join(GOLD, npz))
    return G, {k[2:]: G[k] for k in G.files if k.startswith("w_")}


def _roundtrip(from_fn, to_fn, model, state):
    from_fn(model, state)
    back = to_fn(model)
    assert set(back) == set(state), (sorted(set(state) - set(back))[:5], sorted(set(back) - set(state))[:5])
    for k, v in state.items():
        assert back[k].shape == v.shape, (k, back[k].shape, v.shape)
        assert np.array_equal(back[k], v.astype(np.float32)), k


def test_mae_names_and_layouts_equal_the_reference_model():
    """Names / shapes are those of the reference MaskedAutoencoderViT.named_parameters() (recorded by make_golden_models.gen_mae_model);
    after mae_from_paddle the module's tensors, fed to the oracle, reproduce the reference model's own loss — so the layouts
    (Linear transpose, patch-embedding flattening order) are the ones the forward path uses."""
    from passl_b200.models.mae import MaskedAutoencoderViT
    from passl_b200.utils import checkpoint as C
    import oracle.vit as OV
    G, state = _ref_weights("reference_mae_model.npz")
    m = MaskedAutoencoderViT(img_size=32, patch_size=8, in_chans=3, embed_dim=32, depth=2, num_heads=2, decoder_embed_dim=16,
                             decoder_depth=1, decoder_num_heads=2)
    _roundtrip(C.mae_from_paddle, C.mae_to_paddle, m, state)
    p = {k: v.double() for k, v in m.state_dict().items()}
    cfg = dict(patch=8, heads=2, dec_heads=2, depth=2, dec_depth=1, norm_pix=False, round_pixels=False)
    loss = OV.mae_forward(torch.from_numpy(G["imgs"]), torch.from_numpy(G["noise"]), p, cfg, mask_ratio=0.75)[0]
    assert abs(float(loss) - float(G["loss0"])) < 1e-5 * abs(float(G["loss0"]))          # weights went through fp32


def test_clip_names_and_layouts_equal_the_reference_model():
    from passl_b200.models.clip import CLIP
    from passl_b200.utils import checkpoint as C
    G, state = _ref_weights("reference_clip_model.npz")
    cfg = {k[4:]: int(G[k]) for k in G.files if k.startswith("cfg_")}
    m = CLIP(**{k: (bool(v) if k in ("pre_norm", "proj", "patch_bias", "qkv_bias") else v) for k, v in cfg.items()})
    _roundtrip(C.clip_from_paddle, C.clip_to_paddle, m, state)


def test_mocov3_position_table_is_the_reference_one():
    from passl_b200.models.mocov3 import mocov3_sincos_pos_embed
    G = np.load(os.path.join(GOLD, "reference_mocov3_pos.npz"))
    for t in "abc":
        h, w, d = (int(v) for v in G["cfg_" + t])
        got = mocov3_sincos_pos_embed(d, h, w).numpy()
        assert got.shape == G["pos_" + t].shape and np.abs(got - G["pos_" + t]).max() < 1e-6


def _small_mocov3(literal=False):
    import functools
    from passl_b200.models.mocov3 import MoCoV3Pretrain, MoCoV3ViT
    return MoCoV3Pretrain(functools.partial(MoCoV3ViT, img_size=32, patch_size=8, embed_dim=64, depth=1, num_heads=2, qkv_bias=True),
                          dim=32, mlp_dim=48, reference_ema_quirk=literal)


@pytest.mark.parametrize("literal", [False, True])
def test_mocov3_roundtrip(tmp_path, literal):
    """literal: the averaged predictor copy of the reference's CosineEMA(Sequential(encoder, predictor)) is a tensor set of its own
    (momentum_encoder.model.1.*); otherwise the live predictor is written under those names."""
    from passl_b200.utils import checkpoint as C
    torch.manual_seed(1)
    a, b = _small_mocov3(literal), _small_mocov3(literal)
    for t in list(a.parameters()) + [bf for bf in a.buffers() if bf.dtype.is_floating_point]:
        t.data.normal_()
    a.steps = 7
    path = str(tmp_path / "mocov3.pdparams")
    C.save_pdparams(C.mocov3_to_paddle(a), path)
    C.mocov3_from_paddle(b, C.load_pdparams(path))
    sa, sb = a.state_dict(), b.state_dict()
    assert b.steps == 7 and all(torch.equal(sa[k], sb[k]) for k in sa)
    st = C.load_pdparams(path)
    same = np.array_equal(st["momentum_encoder.model.1.0.weight"], st["predictor.0.weight"])
    assert same != literal and ("momentum_predictor.fcs.0.weight" in sa) == literal


def test_mocov3_names_and_shapes_equal_the_reference_class():
    """passl/models/mocov3.py MoCoV3Pretrain (no weights needed): its state_dict keys and shapes, including the CosineEMA
    wrapper's `momentum_encoder.model.{0,1}.*` / `steps`, must equal what mocov3_to_paddle emits."""
    want, G = _ref_names("mocov3")
    from passl_b200.utils import checkpoint as C
    ours = _small_mocov3()
    got = {k: tuple(v.shape) for k, v in C.mocov3_to_paddle(ours).items()}
    assert set(got) == set(want), (sorted(set(want) - set(got))[:5], sorted(set(got) - set(want))[:5])
    for k in want:
        assert got[k] == want[k], (k, got[k], want[k])
    assert np.abs(ours.base_encoder.vit.pos_embed.numpy() - G["mocov3_pos"]).max() < 1e-6      # the fixed table the reference builds


def test_dispatch_covers_every_model_family():
    """to_paddle_state / load_paddle_state pick the mapping from the model class; SimCLR writes both `encoder.0.*` and the aliased
    `backbone.*` (simclr.py:43-46) and reads either."""
    from passl_b200.modeling import build_model
    from passl_b200.utils import checkpoint as C
    from passl_b200.utils.config import get_config
    cfg = get_config(os.path.join(os.path.dirname(HERE), "configs/simclr/simclr_r50_IM.yaml"), [])
    torch.manual_seed(3)
    a, b = build_model(dict(cfg.model)), build_model(dict(cfg.model))
    st = C.to_paddle_state(a)
    assert st["encoder.0.conv1.weight"].shape == (64, 3, 7, 7) and np.array_equal(st["backbone.conv1.weight"], st["encoder.0.conv1.weight"])
    assert st["encoder.1.mlp.6.weight"].shape == (2048, 128)
    C.load_paddle_state(b, {k: v for k, v in st.items() if not k.startswith("encoder.0.")})      # backbone.* alone is enough
    assert all(torch.equal(v[:, :147] if k.endswith("stem.weight") else v, (b.state_dict()[k][:, :147] if k.endswith("stem.weight") else b.state_dict()[k]))
               for k, v in a.state_dict().items())
    m = _small_mocov3()
    assert set(C.to_paddle_state(m)) == set(C.mocov3_to_paddle(m))
    with pytest.raises(NotImplementedError):
        C.to_paddle_state(torch.nn.Linear(2, 2))


def test_v110_training_checkpoint_container(tmp_path):
    """`epoch_N.pd` of the v110 trainer: a plain pickle {'epoch', 'state_dict', 'lr_scheduler', ...} (hooks/checkpoint_hook.py:22-49);
    written without optimizer state, read back with or without the wrapper, and told apart from this package's torch archives."""
    import pickle
    from passl_b200.optimizer import build_lr_scheduler
    from passl_b200.utils import checkpoint as C
    torch.manual_seed(2)
    a, b = _small_mocov3(), _small_mocov3()
    for t in a.parameters():
        t.data.normal_()
    sched = build_lr_scheduler(dict(name="CosineAnnealingDecay", learning_rate=0.03, T_max=5), 13)
    for _ in range(26):
        sched.step()
    path = str(tmp_path / "epoch_3.pd")
    C.save_v110_checkpoint(path, a, 3, sched)
    raw = pickle.load(open(path, "rb"))
    assert set(raw) == {"epoch", "state_dict", "lr_scheduler"} and raw["epoch"] == 3 and raw["lr_scheduler"]["last_epoch"] == 26
    assert isinstance(raw["state_dict"]["base_encoder.blocks.0.attn.qkv.weight"], np.ndarray)
    assert C.is_paddle_pickle(path)
    ck = C.load_v110_checkpoint(path)
    C.load_paddle_state(b, ck["state_dict"])
    assert ck["epoch"] == 3 and ck["lr_scheduler"]["last_epoch"] == 26
    assert all(torch.equal(v, b.state_dict()[k]) for k, v in a.state_dict().items())
    fresh = build_lr_scheduler(dict(name="CosineAnnealingDecay", learning_rate=0.03, T_max=5), 13)
    fresh.set_state_dict(ck["lr_scheduler"])
    assert fresh() == sched()
    # a bare weights file comes back under 'state_dict' too; torch archives are not mistaken for pickles
    bare = str(tmp_path / "w.pdparams")
    C.save_pdparams(C.to_paddle_state(a), bare)
    assert set(C.load_v110_checkpoint(bare)) == {"state_dict"}
    tpath = str(tmp_path / "iter_2.pd")
    torch.save({"iter": 2}, tpath)
    assert not C.is_paddle_pickle(tpath)
