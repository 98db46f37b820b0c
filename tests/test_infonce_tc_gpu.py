"""tcgen05 fused InfoNCE forward vs the CPU oracle (fp64) and vs the fp32 SIMT variant.

Tolerances (BASELINE.json north_star): loss / logits within 1e-2 relative for the bf16 path; labels and rank
counters are integer-exact given identical logits.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _inputs(N, D, K, seed):
    rng = np.random.RandomState(seed)
    q = rng.randn(N, D).astype(np.float32)
    k = rng.randn(N, D).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    k /= np.linalg.norm(k, axis=1, keepdims=True)
    k = 0.6 * q + 0.4 * k
    k /= np.linalg.norm(k, axis=1, keepdims=True)
    queue = rng.randn(K, D).astype(np.float32)
    queue /= np.linalg.norm(queue, axis=1, keepdims=True)
    return q, k.astype(np.float32), queue


@pytest.mark.parametrize("N,D,K,T", [(256, 128, 65536, 0.2), (16, 128, 65536, 0.2), (128, 128, 4096, 0.07),
                                     (200, 128, 1000, 0.2), (96, 256, 2048, 0.2), (64, 64, 640, 0.1)])
def test_moco_form_matches_oracle(N, D, K, T):
    from oracle import contrastive as O
    from passl_b200 import kernels as K_
    q, k, queue = _inputs(N, D, K, 1234)
    qb = torch.from_numpy(q).cuda().bfloat16()
    kb = torch.from_numpy(queue).cuda().bfloat16()
    kd = torch.from_numpy(k).cuda()
    # oracle on the bf16-rounded operands (isolates kernel error from the quantisation error) ...
    q64 = qb.float().cpu().numpy().astype(np.float64)
    queue64 = kb.float().cpu().numpy().astype(np.float64)
    l_pos, l_neg = O.moco_logits(q64, k.astype(np.float64), queue64.T)
    ref = O.contrastive_head(l_pos, l_neg, T)
    # ... and on the original fp32 operands (the end-to-end bf16 tolerance of BASELINE.json)
    l_pos0, l_neg0 = O.moco_logits(q.astype(np.float64), k.astype(np.float64), queue.astype(np.float64).T)
    ref0 = O.contrastive_head(l_pos0, l_neg0, T)

    out, lse, tgt, rows = K_.infonce_tc_fwd(qb, kb, pos=kd, scale=1.0 / T, want_rows=True)
    torch.cuda.synchronize()
    out = out.cpu().numpy()
    lse_ref = O.logsumexp(ref["logits"], -1)
    np.testing.assert_allclose(lse.cpu().numpy(), lse_ref, rtol=2e-5, atol=2e-5)
    np.testing.assert_allclose(tgt.cpu().numpy(), ref["logits"][:, 0], rtol=1e-5, atol=1e-5)
    assert abs(out[0] - ref["loss"]) <= 1e-4 * abs(ref["loss"]), (out[0], ref["loss"])
    assert abs(out[0] - ref0["loss"]) <= 1e-2 * abs(ref0["loss"]), (out[0], ref0["loss"])
    assert out[1] == pytest.approx(ref["acc1"], abs=100.0 / N + 1e-3)
    assert out[2] == pytest.approx(ref["acc5"], abs=100.0 / N + 1e-3)


def test_label_mode_and_exclusion_match_simt_variant():
    from passl_b200 import kernels as K_
    torch.manual_seed(5)
    N, D, K = 300, 128, 1536
    q = torch.nn.functional.normalize(torch.randn(N, D, device="cuda"), dim=1)
    keys = torch.nn.functional.normalize(torch.randn(K, D, device="cuda"), dim=1)
    lab = (torch.arange(N, device="cuda") + 600).to(torch.int64)
    excl = (torch.arange(N, device="cuda") + 100).to(torch.int32)
    qb, kb = q.bfloat16(), keys.bfloat16()
    o_tc, lse_tc, tgt_tc, _ = K_.infonce_tc_fwd(qb, kb, label=lab, excl=excl, scale=10.0, loss_scale=0.4)
    o_f, lse_f, tgt_f, _ = K_.simce_fwd(qb.float(), kb, label=lab, excl=excl, scale=10.0, loss_scale=0.4)
    torch.cuda.synchronize()
    assert torch.allclose(lse_tc, lse_f, rtol=1e-4, atol=1e-4), (lse_tc - lse_f).abs().max()
    assert torch.allclose(tgt_tc, tgt_f, rtol=1e-4, atol=1e-4)
    assert torch.allclose(o_tc, o_f, rtol=1e-4, atol=1e-2), (o_tc, o_f)


def test_known_answers():
    """SURVEY.md §8c golden identities: zero embeddings -> ln(K+1); q==k, queue orthogonal -> ln(1+K e^{-1/T})."""
    from passl_b200 import kernels as K_
    N, D, K, T = 128, 128, 65536, 0.2
    z = torch.zeros(N, D, device="cuda")
    out, _, _, _ = K_.infonce_tc_fwd(z.bfloat16(), torch.zeros(K, D, device="cuda").bfloat16(), pos=z, scale=1 / T)
    assert abs(out[0].item() - np.log(K + 1)) < 1e-4          # 11.09035
    q = torch.zeros(N, D, device="cuda")
    q[:, 0] = 1.0
    queue = torch.zeros(K, D, device="cuda")
    queue[:, 1] = 1.0
    out, _, _, _ = K_.infonce_tc_fwd(q.bfloat16(), queue.bfloat16(), pos=q, scale=1 / T)
    assert abs(out[0].item() - np.log(1 + K * np.exp(-1 / T))) < 1e-3
    assert out[1].item() == 100.0 and out[2].item() == 100.0


def test_state_is_left_clean_between_calls_and_shapes():
    """The forward merges its key slices through a persistent state buffer (epoch flags, atomics, last-CTA ticket): repeated
    and interleaved calls must give the results of a fresh call."""
    from passl_b200 import kernels as K_
    torch.manual_seed(11)
    outs = {}
    for rep in range(3):
        for (N, K) in [(256, 8192), (64, 4096), (256, 8192), (300, 1536)]:
            g = torch.Generator(device="cuda").manual_seed(N * 7 + K)
            q = torch.nn.functional.normalize(torch.randn(N, 128, device="cuda", generator=g), dim=1).bfloat16()
            keys = torch.nn.functional.normalize(torch.randn(K, 128, device="cuda", generator=g), dim=1).bfloat16()
            pos = torch.nn.functional.normalize(torch.randn(N, 128, device="cuda", generator=g), dim=1)
            o, lse, tgt, _ = K_.infonce_tc_fwd(q, keys, pos=pos, scale=5.0)
            torch.cuda.synchronize()
            key = (N, K)
            if key in outs:
                assert torch.allclose(o, outs[key][0], rtol=1e-6, atol=1e-6), (rep, key, o, outs[key][0])
                assert torch.allclose(lse, outs[key][1], rtol=1e-6, atol=1e-6)
            else:
                o_f, lse_f, _, _ = K_.simce_fwd(q.float(), keys, pos=pos, scale=5.0)
                assert torch.allclose(lse, lse_f, rtol=1e-4, atol=1e-4), (lse - lse_f).abs().max()
                assert torch.allclose(o, o_f, rtol=1e-4, atol=1e-2), (o, o_f)
                outs[key] = (o.clone(), lse.clone())


def test_exponent_mix_matches_fp64_logsumexp():
    """1 in 4 of the exponentials on the FMA-pipe polynomial, the rest on MUFU: lse within 2e-5 of the fp64 logsumexp."""
    from passl_b200 import kernels as K
    torch.manual_seed(3)
    q = torch.nn.functional.normalize(torch.randn(256, 128, device="cuda"), dim=1).bfloat16()
    k = torch.nn.functional.normalize(torch.randn(65536, 128, device="cuda"), dim=1).bfloat16()
    p = torch.nn.functional.normalize(torch.randn(256, 128, device="cuda"), dim=1)
    for T in (0.2, 0.07):
        o, lse, tgt, _ = K.infonce_tc_fwd(q, k, pos=p, scale=1 / T)
        S = torch.cat([(q.float() * p).sum(1, keepdim=True), q.float() @ k.float().T], 1).double() / T
        ref = torch.logsumexp(S, 1)
        err = (lse.double() - ref).abs().max().item()
        assert err < 2e-5 * ref.abs().max().item() + 2e-5, (T, err)


def _ref_dq(qb, kb, pos, label, excl, scale, loss_scale, dloss):
    """fp64 gradient of loss_scale * mean CE w.r.t. q on the given (bf16-rounded) operands."""
    q = qb.double()
    S = q @ kb.double().T * scale
    if excl is not None:
        S[torch.arange(q.shape[0]), excl.long()] = -float("inf")
    if pos is not None:
        lp = (q * pos.double()).sum(1, keepdim=True) * scale
        Pm = torch.softmax(torch.cat([lp, S], 1), 1)
        dq = Pm[:, 1:] @ kb.double() + (Pm[:, :1] - 1.0) * pos.double()
    else:
        Pm = torch.softmax(S, 1)
        dq = Pm @ kb.double() - kb.double()[label]
    return dq * scale * loss_scale * dloss / q.shape[0]


@pytest.mark.parametrize("N,D,K,T", [(256, 128, 65536, 0.2), (16, 128, 65536, 0.2), (128, 128, 4096, 0.07),
                                     (200, 128, 1000, 0.2), (96, 256, 2048, 0.2), (64, 64, 640, 0.1)])
def test_tcgen05_backward_moco_form_vs_fp64(N, D, K, T):
    from passl_b200 import kernels as K_
    q, k, queue = _inputs(N, D, K, 4321)
    qb = torch.from_numpy(q).cuda().bfloat16()
    kb = torch.from_numpy(queue).cuda().bfloat16()
    kd = torch.from_numpy(k).cuda()
    out, lse, tgt, _ = K_.infonce_tc_fwd(qb, kb, pos=kd, scale=1.0 / T)
    dl = torch.tensor([0.7], device="cuda")
    dq = K_.infonce_tc_bwd(qb, kb, lse, tgt, pos=kd, scale=1.0 / T, dloss=dl)
    torch.cuda.synchronize()
    ref = _ref_dq(qb, kb, kd, None, None, 1.0 / T, 1.0, 0.7)
    err = (dq.double() - ref).norm() / ref.norm()
    assert err < 4e-3, err                                # P tiles are rounded to bf16 (2^-9 per element, averaged over the keys)
    worst = ((dq.double() - ref).norm(dim=1) / ref.norm(dim=1)).max()
    assert worst < 1e-2, worst
    # and against the fp32 SIMT backward of round 1
    if D % 128 == 0:                                      # the SIMT kernel works on 128-wide feature chunks
        dq_f = K_.simce_bwd(qb.float(), kb, lse, tgt, pos=kd, scale=1.0 / T, dloss=dl)
        assert (dq - dq_f).norm() / dq_f.norm() < 4e-3


def test_tcgen05_backward_label_mode_and_exclusion():
    from passl_b200 import kernels as K_
    torch.manual_seed(5)
    N, D, K = 300, 128, 1536
    q = torch.nn.functional.normalize(torch.randn(N, D, device="cuda"), dim=1)
    keys = torch.nn.functional.normalize(torch.randn(K, D, device="cuda"), dim=1)
    lab = (torch.arange(N, device="cuda") + 600).to(torch.int64)
    excl = (torch.arange(N, device="cuda") + 100).to(torch.int32)
    qb, kb = q.bfloat16(), keys.bfloat16()
    o, lse, tgt, _ = K_.infonce_tc_fwd(qb, kb, label=lab, excl=excl, scale=10.0, loss_scale=0.4)
    dq = K_.infonce_tc_bwd(qb, kb, lse, tgt, label=lab, excl=excl, scale=10.0, loss_scale=0.4)
    torch.cuda.synchronize()
    ref = _ref_dq(qb, kb, None, lab, excl, 10.0, 0.4, 1.0)
    err = (dq.double() - ref).norm() / ref.norm()
    assert err < 4e-3, err


def test_autograd_node_uses_the_tcgen05_backward():
    from passl_b200.loss import contrastive as C
    torch.manual_seed(2)
    N, D, K = 256, 128, 4096
    q = torch.nn.functional.normalize(torch.randn(N, D, device="cuda"), dim=1).requires_grad_(True)
    k = torch.nn.functional.normalize(torch.randn(N, D, device="cuda"), dim=1)
    queue = torch.nn.functional.normalize(torch.randn(K, D, device="cuda"), dim=1).bfloat16()
    loss, a1, a5 = C.moco_infonce(q, k, queue, 0.2)
    loss.backward()
    ref = _ref_dq(q.detach().bfloat16(), queue, k, None, None, 5.0, 1.0, 1.0)
    assert (q.grad.double() - ref).norm() / ref.norm() < 4e-3
