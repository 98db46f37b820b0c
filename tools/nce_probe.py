"""Fused InfoNCE forward / backward timing (CUDA graph of 8 calls over 8 different queues, L2 flushed between replays, the same
method as bench.py's roofline_infonce) + per-CTA timeline.  Developer tool:  python tools/nce_probe.py [timeline]"""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from passl_b200 import _lib, kernels as K  # noqa: E402


def graph_time(fn_of_queue, queues, flush, reps=20):
    gph = torch.cuda.CUDAGraph()
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        fn_of_queue(queues[0])
        with torch.cuda.graph(gph, stream=st):
            for qq in queues:
                fn_of_queue(qq)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        gph.replay()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e) / len(queues))
    ts.sort()
    return ts[len(ts) // 2] * 1e3        # us per call


def main():
    lib = _lib.load()
    dev = torch.device("cuda")
    res = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for (N, D, Kq, T) in [(256, 128, 65536, 0.2), (16, 128, 65536, 0.2), (1024, 256, 8192, 0.2)]:
        q = torch.nn.functional.normalize(torch.randn(N, D, device=dev), dim=1)
        kpos = torch.nn.functional.normalize(torch.randn(N, D, device=dev), dim=1)
        nq = max(2, (140 << 20) // (Kq * D * 2) + 1)
        nq = min(nq, 16)
        queues = [torch.nn.functional.normalize(torch.randn(Kq, D, device=dev), dim=1).bfloat16() for _ in range(nq)]
        qb = q.bfloat16()
        out, lse, tgt, _ = K.infonce_tc_fwd(qb, queues[0], pos=kpos, scale=1 / T)
        us_f = graph_time(lambda qq: K.infonce_tc_fwd(qb, qq, pos=kpos, scale=1 / T), queues, flush)
        us_b = graph_time(lambda qq: K.infonce_tc_bwd(qb, qq, lse, tgt, pos=kpos, scale=1 / T), queues, flush)
        by = (2 * N * D + D * Kq) * 2 + 4 * N
        res["N%d_D%d_K%d" % (N, D, Kq)] = dict(fwd_us=us_f, bwd_us=us_b, fwd_gbs=by / us_f / 1e3, bwd_gbs=by / us_b / 1e3,
                                                fwd_frac_of_6569=by / us_f / 1e3 / 6569.3)
        if N == 256:
            qf = qb.float()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            K.simce_bwd(qf, queues[0], lse, tgt, pos=kpos, scale=1 / T)
            s.record()
            for i in range(4):
                K.simce_bwd(qf, queues[i % nq], lse, tgt, pos=kpos, scale=1 / T)
            e.record()
            torch.cuda.synchronize()
            res["simt_bwd_us"] = s.elapsed_time(e) / 4 * 1e3
    print(json.dumps(res), flush=True)
    if len(sys.argv) > 1 and sys.argv[1] == "timeline":
        N, D, Kq, T = 256, 128, 65536, 0.2
        q = torch.nn.functional.normalize(torch.randn(N, D, device=dev), dim=1).bfloat16()
        k = torch.nn.functional.normalize(torch.randn(N, D, device=dev), dim=1)
        queues = [torch.nn.functional.normalize(torch.randn(Kq, D, device=dev), dim=1).bfloat16() for _ in range(8)]
        for qq in queues:
            K.infonce_tc_fwd(q, qq, pos=k, scale=1 / T)
        names = ["start", "after setup (alloc, PDL wait, sync)", "Q staged in TMEM", "target fetched"]
        for it in range(5):
            names += ["t%d: begin wait s_full" % it, "t%d: S ready" % it, "t%d: S in registers" % it, "t%d: tile done" % it]
        names = names[:22] + ["loop done, atomics issued", "after __threadfence"]
        names += ["mma: q_ready"] + ["mma: issue t%d" % i for i in range(4)] + ["last CTA: finalize done", "producer: owner targets published",
                                                                               "ticket taken"]
        for mode in ("warm (8th of 8 back-to-back calls over different queues)", "cold (L2 flushed, single call)"):
            dbg = torch.zeros(148 * 32, dtype=torch.int64, device=dev)
            torch.cuda.synchronize()
            if mode.startswith("cold"):
                flush.zero_()
                torch.cuda.synchronize()
            lib.passl_b200_infonce_tc_set_debug(dbg.data_ptr())
            for qq in (queues if mode.startswith("warm") else queues[:1]):
                K.infonce_tc_fwd(q, qq, pos=k, scale=1 / T)
            torch.cuda.synchronize()
            lib.passl_b200_infonce_tc_set_debug(None)
            t = dbg.cpu().reshape(148, 32).double()
            g0 = t[:, 0][t[:, 0] > 0]
            print("---- timeline,", mode, "| CTA start spread (globaltimer) %.2f us; rows below: SM cycles since the CTA's own start" %
                  ((g0.max() - g0.min()) / 1e3))
            for i, n in enumerate(names):
                if i == 0:
                    continue
                col = t[:, i]
                col = col[col > 0]
                if len(col):
                    print("%-36s min %7.0f  median %7.0f  max %7.0f cycles" % (n, col.min(), col.median(), col.max()))


if __name__ == "__main__":
    main()
