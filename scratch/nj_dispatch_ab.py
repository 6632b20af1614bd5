#!/usr/bin/env python
"""A/B of two libnnj.so builds on the NJ pair-score dispatch: same results, same kernels.

    NNJ_LIB_PATH=old/libnnj.so python scratch/nj_dispatch_ab.py run  OUT/old.pt
                               python scratch/nj_dispatch_ab.py run  OUT/new.pt
                               python scratch/nj_dispatch_ab.py diff OUT/old.pt OUT/new.pt

`run` (one library per process, the one NNJ_LIB_PATH or the tree's build names) goes through shapes that between them reach
every row of the pair-score selection table (DESIGN 4):
  * fused rollouts, bf16x3: 50 x 1024 (B = 4; step 0 on k_score_tc, then k_score_inc, the register-fragment kernels, and the last
    step's k_score<false>), 12 x 128, 17 x 192, 100 x 1024 (B = 2; 101 slots: the large-slot path), 40 x 250 (C % 8 != 0: fp32 kernels);
  * fused rollouts at 50 x 256 in fp32 and in bf16;
  * the step-wise API (pair_scores_full / list / incr, aggregate, merge) in bf16x3 at 20 x 256 (fused kernels) and 70 x 256 (large-slot).
It stores the merge lists, selected log-probabilities and logits traces (and the step-wise outputs), then repeats everything once
under torch.profiler and stores the sequence of CUDA kernel / memset names.  `diff` requires both to be identical, bit for bit."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

ROLLOUTS = [("bf16x3", 50, 1024, 4), ("bf16x3", 12, 128, 2), ("bf16x3", 17, 192, 2), ("bf16x3", 100, 1024, 2), ("bf16x3", 40, 250, 2),
            ("fp32", 50, 256, 2), ("bf16", 50, 256, 2)]
STEPWISE = [("bf16x3", 20, 256, 2), ("bf16x3", 70, 256, 2)]


def models():
    from neuralnj_b200 import PhyloATTN, inference_config
    out = {}
    for prec in ("bf16x3", "fp32", "bf16"):
        torch.manual_seed(0)
        out[prec] = PhyloATTN(inference_config(), precision=prec).to("cuda:0").eval()
    return out


def stepwise(model, R, L, B):
    """full scores -> aggregate -> merge -> incremental scores (closed form and the pair-list form) at R - 1 nodes."""
    import nnj_oracle as O
    from neuralnj_b200 import _lib
    data = O.evolved_msa(B, R, L, seed=R).cuda()
    mask = torch.zeros(B, L, dtype=torch.bool, device="cuda")
    mask[:, 5::37] = True
    state = model.encode_zxr(data, mask)
    full = model.decode_zxr(state, mask, (None, None, None))["logits"]
    ij = torch.tensor([[1, 4], [0, R - 1]][:B], dtype=torch.int32, device="cuda")
    agg = model.aggregate(None, None, (ij[:, 0], ij[:, 1]), batchwise_ij_indices=True)
    merged = model.merge_state(state, ij)
    incr = model.decode_zxr(merged, mask, (ij, None, full))["logits"]
    n = R - 1
    pi = ij[:, :1].expand(B, n).contiguous()
    r = torch.arange(n, dtype=torch.int32, device="cuda").unsqueeze(0).expand(B, n)
    a, b = torch.minimum(pi, r).contiguous(), torch.maximum(pi, r).contiguous()
    new = torch.empty(B, n, dtype=torch.float32, device="cuda")
    ws = model._workspace(1, B, n, L)
    m8 = mask.to(torch.uint8).contiguous()
    _lib.check(_lib.lib().nnj_pair_scores_list(model.handle(), merged.data_ptr(), m8.data_ptr(), B, n, L, a.data_ptr(), b.data_ptr(), n,
                                               new.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream),
               "nnj_pair_scores_list")
    return {"full": full, "aggregate": agg, "merge": merged, "incr": incr, "list": new}


def workload(ms):
    import nnj_oracle as O
    res = {}
    for prec, R, L, B in ROLLOUTS:
        data = O.evolved_msa(B, R, L, seed=R + L).cuda()
        mask = torch.zeros(B, L, dtype=torch.bool, device="cuda")
        mask[:, 3::29] = True
        merges, slp, trace = ms[prec].rollout_fused(data, mask, want_logits=True)
        res[f"rollout/{prec}/{R}x{L}"] = {"merges": merges, "selected_logp": slp, "trace": trace}
    for prec, R, L, B in STEPWISE:
        res[f"stepwise/{prec}/{R}x{L}"] = stepwise(ms[prec], R, L, B)
    torch.cuda.synchronize()
    return {k: {n: t.detach().cpu() for n, t in v.items()} for k, v in res.items()}


def run(out):
    from torch.profiler import ProfilerActivity, profile
    from neuralnj_b200 import _lib
    assert torch.cuda.is_available(), "the A/B needs a GPU"
    print("library:", os.environ.get("NNJ_LIB_PATH") or _lib.LIB_PATH, flush=True)
    ms = models()
    results = workload(ms)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        workload(ms)
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    ev.sort(key=lambda e: e.time_range.start)
    names = [e.name for e in ev]
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    torch.save({"results": results, "kernels": names, "card": torch.cuda.get_device_name(0)}, out)
    print(f"{out}: {len(results)} cases, {len(names)} device activities", flush=True)


def diff(a_path, b_path):
    a, b = torch.load(a_path), torch.load(b_path)
    bad = 0
    for case in sorted(set(a["results"]) | set(b["results"])):
        ra, rb = a["results"].get(case), b["results"].get(case)
        if ra is None or rb is None:
            print(f"{case}: missing on one side"); bad += 1; continue
        for k in sorted(ra):
            same = ra[k].shape == rb[k].shape and ra[k].dtype == rb[k].dtype and torch.equal(ra[k].view(torch.uint8), rb[k].view(torch.uint8))
            if not same:
                bad += 1
            print(f"{case:28s} {k:15s} {'bit-identical' if same else 'DIFFERENT'}")
    ka, kb = a["kernels"], b["kernels"]
    first = next((i for i, (x, y) in enumerate(zip(ka, kb)) if x != y), None)
    ok_k = ka == kb
    print(f"kernel sequence: {len(ka)} vs {len(kb)} activities, {'identical' if ok_k else 'DIFFERENT'}"
          + ("" if ok_k else f" (first difference at {first}: {ka[first] if first is not None else '-'} / {kb[first] if first is not None else '-'})"))
    names = sorted(set(ka))
    print(f"{len(names)} distinct names:")
    for n in names:
        print(f"  {ka.count(n):6d}  {n[:150]}")
    bad += 0 if ok_k else 1
    print("A/B:", "PASS" if bad == 0 else f"FAIL ({bad})")
    return 1 if bad else 0


if __name__ == "__main__":
    if sys.argv[1] == "run":
        run(sys.argv[2])
    elif sys.argv[1] == "diff":
        sys.exit(diff(sys.argv[2], sys.argv[3]))
    else:
        sys.exit(__doc__)
