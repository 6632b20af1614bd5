#!/usr/bin/env python
"""A/B of two checkouts on the tree likelihood, branch support and the host-buffer rollout: same results, same kernels.

    cd OLD && python scratch/llh_ab.py run  OUT/old.pt
    cd NEW && python scratch/llh_ab.py run  OUT/new.pt
              python scratch/llh_ab.py diff OUT/old.pt OUT/new.pt

`run` uses the Python package and libnnj.so of the checkout it is started from (NNJ_LIB_PATH, if set, names another library):
  * nnj_llh_eval / optimize_brlen / optimize_all / branch_support through ctypes: llh, brlen, model, branch_node, L0/L1/L2, NNI lengths,
    SH / LBP counts and site_llh_dev, at R = 3 and 4; 50 x 1024 (B = 16) under JC, GTR+G and GTR+I+G; 200 x 1000 (B = 2); 4096 x 200
    (scaled vectors); n_rell 0, 1, 300 from replicate 0 and 300 from replicate 700;
  * score_topologies (with and without the model search), optimize_brlen, compute_llh, likelihood_support and bootstrap_support
    (256 replicates: two chunks) on tests/golden/msa/ex50x1024_71 and _73, and the files of Argmax_inference(alrt=100, bootstrap=50);
  * nnj_rollout_host at 50 x 1024 with B = 200 (two chunks) under a mask, Argmax and Gumbel, with selected_logp; nnj_rank_loss on the
    trace of a teacher-forced rollout.
It stores every output, then repeats the ctypes part once under torch.profiler and stores the sequence of CUDA kernel / memset
names.  `diff` requires all of it to be identical, bit for bit."""
import ctypes as C
import os
import shutil
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
GOLD = os.path.join(ROOT, "tests", "golden", "msa")
NAMES = ["ex50x1024_71", "ex50x1024_73"]
GEN = dict(rates6=(1.2, 3.1, 0.8, 1.1, 4.2, 1.0), freqs=(0.3, 0.2, 0.2, 0.3), alpha=0.7, pinv=0.15)
# (R, L, B, model)
SHAPES = [(3, 50, 2, "GTR+I+G"), (4, 60, 2, "GTR+I+G"), (50, 1024, 16, "JC"), (50, 1024, 16, "GTR+G"), (50, 1024, 16, "GTR+I+G"),
          (200, 1000, 2, "GTR+I+G"), (4096, 200, 1, "GTR+I+G")]
RELL = [(0, 0), (1, 0), (300, 0), (300, 700)]
vp = C.c_void_p


def _case(R, L, B, spec):
    import llh_oracle as O
    from neuralnj_b200 import likelihood as LH
    rng = np.random.default_rng(1000 * R + L)
    chs, bls = zip(*[O.random_tree(R, rng) for _ in range(B)])
    tips = O.simulate(chs[0], bls[0], R, L, O.Model(**GEN), rng, gap_frac=0.05)
    sm = LH.SubstModel(spec, np.asarray(GEN["freqs"]), B)
    if sm.gtr:
        sm.rates[:] = GEN["rates6"]
    sm.alpha[:] = GEN["alpha"]
    sm.pinv[:] = GEN["pinv"] if sm.inv else 0.0
    w = rng.integers(1, 4, size=L).astype(np.float64)
    return np.ascontiguousarray(np.stack(chs), dtype=np.int32), np.ascontiguousarray(np.stack(bls)), tips, w, sm


def direct():
    """The four nnj_llh_* entry points through ctypes."""
    from neuralnj_b200 import _lib
    lib = _lib.lib()
    res = {}
    P = lambda a: a.ctypes.data_as(vp)
    for R, L, B, spec in SHAPES:
        ch, bl, tips, w, sm = _case(R, L, B, spec)
        key = f"llh/{R}x{L}x{B}/{spec}"
        t = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(tips, (B, R, L)))).cuda()
        wd = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(w, (B, L)))).cuda()
        n_ws = max(int(lib.nnj_llh_support_workspace_bytes(B, R, L, n)) for n, _ in RELL)
        ws = torch.empty(n_ws, dtype=torch.uint8, device="cuda")
        st = vp(torch.cuda.current_stream().cuda_stream)
        dev = (vp(t.data_ptr()), vp(wd.data_ptr()), P(ch))
        tail = (vp(ws.data_ptr()), ws.numel(), st)
        packed = sm.pack()
        out = {}
        ll = np.zeros(B)
        _lib.check(lib.nnj_llh_eval(*dev, P(bl), P(packed), B, R, L, P(ll), *tail), "eval")
        out["eval"] = ll.copy()
        b1, ll0, ll1 = bl.copy(), np.zeros(B), np.zeros(B)
        _lib.check(lib.nnj_llh_optimize_brlen(*dev, P(b1), P(packed), B, R, L, 32, C.c_double(1e-3), P(ll0), P(ll1), *tail), "brlen")
        out.update(brlen_brlen=b1, brlen_before=ll0.copy(), brlen_after=ll1.copy())
        b2, m2 = bl.copy(), packed.copy()
        _lib.check(lib.nnj_llh_optimize_all(*dev, P(b2), P(m2), B, R, L, 32, C.c_double(1e-3), C.c_double(1.0), 10, P(ll0), P(ll1), *tail), "all")
        out.update(all_brlen=b2, all_model=m2, all_before=ll0.copy(), all_after=ll1.copy())
        nb = max(R - 3, 0)
        for n_rell, rep0 in RELL:
            bn, l3, nl = np.zeros((B, nb), np.int32), np.zeros((B, nb, 3)), np.zeros((B, nb, 2, 5))
            sh, lbp = np.zeros((B, nb), np.int32), np.zeros((B, nb), np.int32)
            site = torch.full((B, nb, 3, L), -1.0, dtype=torch.float64, device="cuda")
            _lib.check(lib.nnj_llh_branch_support(*dev, P(b2), P(m2), B, R, L, C.c_uint64(11), C.c_int64(rep0), n_rell, P(bn), P(l3), P(nl), P(sh),
                                                  P(lbp), vp(site.data_ptr() if nb else 0), *tail), "branch_support")
            out.update({f"sup{n_rell}@{rep0}/{k}": v for k, v in dict(branch_node=bn, llh=l3, nni_brlen=nl, sh=sh, lbp=lbp,
                                                                         site=site.cpu().numpy()).items()})
        torch.cuda.synchronize()
        res[key] = {k: torch.from_numpy(np.asarray(v)) for k, v in out.items()}
    return res


def models():
    from neuralnj_b200 import PhyloATTN, inference_config
    torch.manual_seed(0)
    return PhyloATTN(inference_config(), precision="bf16x3").to("cuda:0").eval()


def high_level(model, tmp):
    import llh_oracle as O
    from neuralnj_b200 import Argmax_inference, bootstrap_support, inference_config, likelihood_support
    from neuralnj_b200 import likelihood as LH
    from neuralnj_b200.phydata import load_pi_instance
    src = os.path.join(tmp, "msas")
    os.makedirs(src)
    for n in NAMES:
        shutil.copyfile(os.path.join(GOLD, n + ".phy"), os.path.join(src, n + ".phy"))
    kw = dict(cfgs=inference_config(), device=torch.device("cuda:0"), files_per_call=1, policy_network=model)
    Argmax_inference(src, os.path.join(tmp, "out"), None, alrt=100, alrt_seed=2, bootstrap=50, bootstrap_seed=5, **kw)
    res = {}
    for f in sorted(os.listdir(os.path.join(tmp, "out"))):
        with open(os.path.join(tmp, "out", f), "rb") as fh:
            res[f"file/{f}"] = {"bytes": torch.frombuffer(bytearray(fh.read()), dtype=torch.uint8)}
    for n in NAMES:
        path = os.path.join(src, n + ".phy")
        tre = open(os.path.join(tmp, "out", n + ".tre")).read()
        batch = load_pi_instance(path)
        keys, seqs = [str(k) for k in batch["seq_keys"][0]], [str(s) for s in batch["seqs"][0]]
        msa = {"labels": keys, "sequences": seqs}
        masks = LH.sequences_to_masks(seqs)
        rng = np.random.default_rng(3)
        ch = np.stack([O.random_tree(len(keys), rng)[0] for _ in range(4)]).astype(np.int32)
        out = {}
        for opt in (True, False):
            ll, t = LH.score_topologies(masks, ch, keys, opt_model=opt)
            out[f"score_topologies/{opt}/llh"], out[f"score_topologies/{opt}/brlen"] = ll, t
        nw, b, a = LH.optimize_brlen(tre, msa, model="GTR+I+G")
        out["optimize_brlen/newick"] = np.frombuffer(nw.encode(), dtype=np.uint8)
        out["optimize_brlen/llh"] = np.array([b, a])
        out["compute_llh"] = np.array([LH.compute_llh(tre, msa, model="GTR+I+G"), LH.compute_llh(tre, msa, model="JC", opt_model=False)])
        ls = likelihood_support(path, model, n_rell=300, seed=4)
        for k in ("alrt", "sh_alrt", "abayes", "lbp", "llh_nni"):
            out[f"likelihood_support/{k}"] = ls[k]
        out["likelihood_support/text"] = np.frombuffer((ls["tree"] + ls["newick_alrt"] + ls["newick_abayes"]).encode(), dtype=np.uint8)
        bs = bootstrap_support(path, model, 256, seed=9)
        out["bootstrap/fbp"], out["bootstrap/tbe"] = bs["fbp"], bs["tbe"]
        out["bootstrap/text"] = np.frombuffer((bs["newick_fbp"] + bs["newick_tbe"]).encode(), dtype=np.uint8)
        res[f"api/{n}"] = {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in out.items()}
    return res


def host_rollout(model):
    import random

    import nnj_oracle as O
    from neuralnj_b200 import PhyInferEnv, _lib, balanced_elu_loss, inference_config, supervise_rollout
    from neuralnj_b200.supervise import LabelTree
    lib = _lib.lib()
    R, L, B = 50, 1024, 200
    data = O.evolved_msa(B, R, L, seed=17).to(torch.int8).contiguous()
    mask = torch.zeros(B, L, dtype=torch.uint8)
    mask[:, 7::31] = 1
    P0 = R * (R - 1) // 2
    g = torch.Generator().manual_seed(5)
    gum = -torch.log(-torch.log(torch.rand(B, R - 1, P0, generator=g).clamp_min(1e-20)))
    res = {}
    for mode, noise in ((0, None), (1, gum)):
        merges = torch.zeros(B, R - 1, 2, dtype=torch.int32)
        slp = torch.zeros(B, R - 1, dtype=torch.float32)
        _lib.check(lib.nnj_rollout_host(model.handle(), vp(data.data_ptr()), vp(mask.data_ptr()), B, R, L, mode,
                                        vp(noise.data_ptr() if noise is not None else 0), vp(merges.data_ptr()), vp(slp.data_ptr())), "rollout_host")
        res[f"rollout_host/{mode}"] = {"merges": merges, "selected_logp": slp}
    label = LabelTree("(((taxon1,taxon7),(taxon3,(taxon12,taxon5))),((taxon2,taxon9),((taxon4,taxon11),(taxon6,(taxon8,taxon10)))));")
    acts, sets = label.sample_trajectory(random.Random(0))
    Rs, Ls = 12, 128
    d = O.evolved_msa(1, Rs, Ls, seed=3)
    batch = {"data": d, "seq_weights": torch.ones(1, Ls), "seqs": [["A" * Ls] * Rs], "seq_keys": [[f"taxon{i + 1}" for i in range(Rs)]],
             "actions": torch.tensor([[acts]], dtype=torch.int32), "actions_set": [[sets]]}
    sup = supervise_rollout(batch, model, PhyInferEnv(inference_config(), torch.device("cuda:0")), eval=True)
    loss = balanced_elu_loss(sup, epoch=0, ratio_factor=0.5)
    res["rank_loss"] = {"loss": torch.tensor([loss["loss"], loss["precision"]], dtype=torch.float64), "steps": torch.as_tensor(loss["step_losses"])}
    return res


def run(out):
    from torch.profiler import ProfilerActivity, profile
    from neuralnj_b200 import _lib
    assert torch.cuda.is_available(), "the A/B needs a GPU"
    print("library:", os.environ.get("NNJ_LIB_PATH") or _lib.LIB_PATH, flush=True)
    results = direct()
    model = models()
    with tempfile.TemporaryDirectory() as tmp:
        results.update(high_level(model, tmp))
    results.update(host_rollout(model))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        direct()
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
        for k in sorted(set(ra) | set(rb)):
            x, y = ra.get(k), rb.get(k)
            same = x is not None and y is not None and x.shape == y.shape and x.dtype == y.dtype and \
                x.contiguous().numpy().tobytes() == y.contiguous().numpy().tobytes()
            bad += not same
            if not same or k.count("/") < 2:
                print(f"{case:40s} {k:32s} {'bit-identical' if same else 'DIFFERENT'}")
    ka, kb = a["kernels"], b["kernels"]
    ok_k = ka == kb
    print(f"kernel sequence: {len(ka)} vs {len(kb)} activities, {'identical' if ok_k else 'DIFFERENT'}")
    for n in sorted(set(ka)):
        print(f"  {ka.count(n):6d}  {n[:150]}")
    bad += 0 if ok_k else 1
    print("A/B:", "PASS" if bad == 0 else f"FAIL ({bad})")
    return 1 if bad else 0


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "run":
        run(sys.argv[2])
    elif len(sys.argv) > 3 and sys.argv[1] == "diff":
        sys.exit(diff(sys.argv[2], sys.argv[3]))
    else:
        sys.exit(__doc__)
