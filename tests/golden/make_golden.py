"""Generate the golden fixtures in this directory from the UPSTREAM reference itself.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

It imports the reference modules (CPU, fp32, torch as installed in the image), runs
them on seeded synthetic inputs and writes ``*.npz`` files next to this script.  The
fixtures are what pins ``oracle/grafp_oracle.py`` to the reference
(tests/test_oracle_golden.py) and what the GPU parity tests replay on the B200 box,
where /root/reference does not exist.

``fingerprints.npz`` is the exception: it comes from the oracle at full size on the GPU (see make_fingerprints).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import _reference_import  # noqa: E402
from grafp_b200 import synth  # noqa: E402

torch.set_num_threads(4)
torch.backends.cudnn.enabled = False


def save(name, **arrays):
    path = os.path.join(HERE, name + ".npz")
    out = {}
    for k, v in arrays.items():
        if isinstance(v, torch.Tensor):
            v = v.detach().cpu().numpy()
        out[k] = np.asarray(v)
    np.savez_compressed(path, **out)
    print(f"wrote {path}  ({os.path.getsize(path) / 1024:.1f} KiB)")


KNN_CASES = [
    # name,            B, C,   N,   k, d, M (0: y=None), relpos, input kind
    ("plain_k3",       2, 16,  96,  3, 1, 0,  False, "randn"),
    ("dil2_k4",        2, 16,  96,  4, 2, 0,  False, "randn"),
    ("dil3_k3",        2, 32,  128, 3, 3, 0,  False, "relu"),
    ("stage2_like",    1, 64,  256, 3, 1, 0,  False, "relu"),
    ("stress_like",    1, 64,  256, 16, 4, 0, False, "randn"),
    ("ragged_n",       2, 12,  70,  5, 1, 0,  False, "randn"),
    ("xy_pooled",      2, 16,  64,  4, 1, 16, False, "randn"),
    ("xy_relpos",      2, 16,  64,  4, 2, 16, True,  "randn"),
    ("relpos_self",    1, 16,  64,  4, 1, 0,  True,  "randn"),
    ("k_equals_n",     1, 8,   16,  16, 1, 0, False, "randn"),
]


def knn_input(kind, B, C, N, seed):
    x = synth.synth_point_cloud(B, C, N, seed, relu=(kind == "relu"))
    return x


def make_knn(ref):
    arrays = {}
    names = []
    for i, (name, B, C, N, k, d, M, relpos, kind) in enumerate(KNN_CASES):
        x = knn_input(kind, B, C, N, 100 + i)
        y = knn_input(kind, B, C, M, 200 + i) if M else None
        rp = None
        if relpos:
            rp = 0.05 * torch.randn(1, N, M or N, generator=torch.Generator().manual_seed(300 + i))
        graph = ref.torch_edge.DenseDilatedKnnGraph(k=k, dilation=d, stochastic=False, epsilon=0.0)
        edge = graph(x, y, rp)
        assert edge.shape == (2, B, N, k) and edge.dtype == torch.int64
        names.append(name)
        arrays[f"{name}.x"] = x
        if y is not None:
            arrays[f"{name}.y"] = y
        if rp is not None:
            arrays[f"{name}.relative_pos"] = rp
        arrays[f"{name}.edge_index"] = edge.contiguous()
        arrays[f"{name}.kd"] = np.array([k, d])
    arrays["names"] = np.array(names)
    save("knn", **arrays)


COS_CASES = [
    # name,          cls,   B, C,  N,   k, d, M (0: y=None), relpos
    ("plg_self",     "plg", 2, 16, 96,  3, 1, 0,  False),
    ("plg_self_d2",  "plg", 2, 32, 128, 4, 2, 0,  False),
    ("plg_relpos",   "plg", 1, 16, 64,  4, 1, 0,  True),
    ("plg_xy",       "plg", 2, 16, 64,  4, 2, 16, True),
    ("new_xy",       "new", 2, 16, 64,  4, 1, 16, False),
    ("plg_stage2",   "plg", 1, 64, 256, 3, 1, 0,  False),
]


def make_knn_cos(ref):
    """The cosine graph builders DenseDilatedKnnGraph_plg / _new (torch_edge.py:286-361)."""
    arrays = {"names": np.array([c[0] for c in COS_CASES])}
    for i, (name, cls, B, C, N, k, d, M, relpos) in enumerate(COS_CASES):
        x = knn_input("randn", B, C, N, 300 + i)
        y = knn_input("randn", B, C, M, 400 + i) if M else None
        rp = None
        if relpos:
            rp = 0.1 * torch.randn(1, N, M if M else N, generator=torch.Generator().manual_seed(500 + i))
        mod = (ref.torch_edge.DenseDilatedKnnGraph_plg if cls == "plg" else ref.torch_edge.DenseDilatedKnnGraph_new)(k=k, dilation=d)
        with torch.no_grad():
            edge = mod(x, y, rp)
        arrays[f"{name}.x"] = x
        if y is not None:
            arrays[f"{name}.y"] = y
        if rp is not None:
            arrays[f"{name}.relative_pos"] = rp
        arrays[f"{name}.kd"] = np.array([k, d])
        arrays[f"{name}.cls"] = np.array(cls)
        arrays[f"{name}.edge_index"] = edge.contiguous()
    save("knn_cos", **arrays)


def make_aggregate(ref):
    arrays = {}
    g = torch.Generator().manual_seed(7)
    B, C, N, k = 2, 16, 64, 4
    x = synth.synth_point_cloud(B, C, N, 11, relu=True)
    x[:, :, 5] = x[:, :, 9]           # duplicate nodes -> argmax ties
    x[:, :, 20] = 0                   # an all-zero node
    edge = ref.torch_edge.DenseDilatedKnnGraph(k=k, dilation=1)(x)
    arrays["self.x"], arrays["self.edge_index"] = x, edge
    arrays["self.gather"] = ref.torch_nn.batched_index_select(x, edge[0])

    # arbitrary user-supplied graph incl. a non-arange centre row and a separate key set y
    M = 24
    y = synth.synth_point_cloud(B, C, M, 12)
    e0 = torch.randint(0, M, (B, N, k), generator=g)
    e1 = torch.randint(0, N, (B, N, k), generator=g)
    edge_xy = torch.stack((e0, e1), 0)
    arrays["xy.x"], arrays["xy.y"], arrays["xy.edge_index"] = x, y, edge_xy
    arrays["xy.gather"] = ref.torch_nn.batched_index_select(y, e0)

    def mr_features(xx, ee, yy):
        # the part of MRConv2d.forward before self.nn (torch_vertex.py:21-32)
        conv = ref.torch_vertex.MRConv2d(C, 2 * C, "relu", None, True)
        captured = {}
        conv.nn = torch.nn.Identity()
        conv.nn.register_forward_hook(lambda m, i, o: captured.setdefault("v", i[0]))
        conv(xx, ee, yy)
        return captured["v"]

    def edge_feats(xx, ee, yy):
        conv = ref.torch_vertex.EdgeConv2d(C, 2 * C, "relu", None, True)
        captured = {}
        conv.nn = torch.nn.Identity()
        conv.nn.register_forward_hook(lambda m, i, o: captured.setdefault("v", i[0]))
        conv(xx, ee, yy)
        return captured["v"]

    for tag, (xx, ee, yy) in {"self": (x, edge, None), "xy": (x, edge_xy, y)}.items():
        xx = xx.clone().requires_grad_(True)
        yy2 = None if yy is None else yy.clone().requires_grad_(True)
        feat = mr_features(xx, ee, yy2)
        up = torch.randn(feat.shape, generator=g)
        feat.backward(up)
        arrays[f"{tag}.mr_features"] = feat
        arrays[f"{tag}.mr_upstream"] = up
        arrays[f"{tag}.mr_grad_x"] = xx.grad
        if yy2 is not None:
            arrays[f"{tag}.mr_grad_y"] = yy2.grad

        xx = xx.detach().clone().requires_grad_(True)
        yy2 = None if yy is None else yy.clone().requires_grad_(True)
        ef = edge_feats(xx, ee, yy2)
        up = torch.randn(ef.shape, generator=g)
        ef.backward(up)
        arrays[f"{tag}.edge_features"] = ef
        arrays[f"{tag}.edge_upstream"] = up
        arrays[f"{tag}.edge_grad_x"] = xx.grad
        if yy2 is not None:
            arrays[f"{tag}.edge_grad_y"] = yy2.grad
    save("aggregate", **arrays)


def load_synth(module, seed):
    sd = module.state_dict()
    keep = {k: v for k, v in sd.items() if k.endswith("relative_pos")}
    module.load_state_dict(synth.synth_state_dict({k: v.shape for k, v in sd.items()}, seed, keep))


def make_gconv(ref):
    arrays = {}
    B, C, N, k = 2, 16, 64, 4
    g = torch.Generator().manual_seed(21)
    x0 = synth.synth_point_cloud(B, C, N, 31)
    for conv in ("mr", "edge", "sage", "gin"):
        for d in (1, 2):
            tag = f"{conv}_d{d}"
            mod = ref.torch_vertex.DyGraphConv2d(C, 2 * C, kernel_size=k, dilation=d, conv=conv, act="relu",
                                                 norm="batch", bias=True, stochastic=False, epsilon=0.0, r=1)
            load_synth(mod, 40 + d)
            mod.train()
            x = x0.clone().requires_grad_(True)
            out = mod(x)
            up = torch.randn(out.shape, generator=g)
            out.backward(up)
            arrays[f"{tag}.out"] = out
            arrays[f"{tag}.upstream"] = up
            arrays[f"{tag}.grad_x"] = x.grad
            for name, p in mod.named_parameters():
                arrays[f"{tag}.grad.{name}"] = p.grad
            for name, b in mod.named_buffers():
                arrays[f"{tag}.buf.{name}"] = b
    arrays["x"] = x0
    arrays["cfg"] = np.array([B, C, N, k])
    save("gconv", **arrays)


def make_gconv_r2(ref):
    """DyGraphConv2d with r = 2 on an H x W feature map: the keys are the 2 x 2 average-pooled map
    (torch_vertex.py:130-132), N = H * W queries against M = N / 4 keys."""
    arrays = {}
    B, C, H, W, k = 2, 16, 8, 8, 4
    g = torch.Generator().manual_seed(23)
    x0 = torch.randn(B, C, H, W, generator=torch.Generator().manual_seed(33))
    for conv in ("mr", "edge", "sage", "gin"):
        for d in (1, 2):
            tag = f"{conv}_d{d}"
            mod = ref.torch_vertex.DyGraphConv2d(C, 2 * C, kernel_size=k, dilation=d, conv=conv, act="relu",
                                                 norm="batch", bias=True, stochastic=False, epsilon=0.0, r=2)
            load_synth(mod, 50 + d)
            mod.train()
            x = x0.clone().requires_grad_(True)
            out = mod(x)
            up = torch.randn(out.shape, generator=g)
            out.backward(up)
            arrays[f"{tag}.out"] = out
            arrays[f"{tag}.upstream"] = up
            arrays[f"{tag}.grad_x"] = x.grad
            for name, p in mod.named_parameters():
                arrays[f"{tag}.grad.{name}"] = p.grad
            for name, b in mod.named_buffers():
                arrays[f"{tag}.buf.{name}"] = b
    arrays["x"] = x0
    arrays["cfg"] = np.array([B, C, H, W, k])
    save("gconv_r2", **arrays)


def make_grapher(ref):
    arrays = {}
    B, C, N, k, d = 2, 32, 64, 4, 2
    g = torch.Generator().manual_seed(51)
    mod = ref.torch_vertex.Grapher(C, k, d, "mr", "relu", "batch", True, False, 0.2, 1, n=N, drop_path=0.0,
                                   relative_pos=True)
    load_synth(mod, 61)
    mod.train()
    x = synth.synth_point_cloud(B, C, N, 71).requires_grad_(True)
    out = mod(x)
    up = torch.randn(out.shape, generator=g)
    out.backward(up)
    arrays.update(x=x, out=out, upstream=up, grad_x=x.grad, cfg=np.array([B, C, N, k, d]))
    arrays["relative_pos"] = mod.relative_pos
    for name, p in mod.named_parameters():
        if p.grad is not None:
            arrays[f"grad.{name}"] = p.grad
    mod.eval()
    arrays["out_eval"] = mod(x.detach())
    save("grapher", **arrays)


def make_encoder(ref):
    cfg = dict(synth.DEFAULT_CFG)
    B = 4
    enc = ref.graph_encoder.GraphEncoder(cfg=cfg, in_channels=cfg["n_filters"], k=3)
    sd = enc.state_dict()
    arrays = {"keys": np.array(list(sd.keys())),
              "shapes": np.array([",".join(map(str, v.shape)) for v in sd.values()]),
              "requires_grad": np.array([k for k, p in enc.named_parameters() if p.requires_grad])}
    load_synth(enc, 81)
    # relative_pos tables: store a fingerprint only (2.25 M floats)
    for k, v in enc.state_dict().items():
        if k.endswith("relative_pos"):
            arrays[f"relpos_sum.{k}"] = v.double().sum()
            arrays[f"relpos_head.{k}"] = v.flatten()[:64]
    g = torch.Generator().manual_seed(91)
    x = torch.rand(B, cfg["n_filters"], 1024, generator=g)
    enc.train()
    xin = x.clone().requires_grad_(True)
    out = enc(xin)
    up = torch.randn(out.shape, generator=g)
    (out * up).sum().backward()
    arrays.update(x=x, out_train=out, upstream=up, grad_x=xin.grad)
    arrays["grad_norm"] = np.array([float(p.grad.double().norm()) if p.grad is not None else -1.0
                                    for _, p in enc.named_parameters()])
    arrays["grad_names"] = np.array([n for n, _ in enc.named_parameters()])
    arrays["grad.stem.0.weight"] = enc.stem[0].weight.grad
    arrays["grad.proj.weight.head"] = enc.proj.weight.grad.flatten()[:4096]
    arrays["grad.backbone.0.0.graph_conv.gconv.nn.0.weight"] = enc.backbone[0][0].graph_conv.gconv.nn[0].weight.grad
    arrays["grad.backbone.8.0.fc1.0.weight.head"] = enc.backbone[8][0].fc1[0].weight.grad.flatten()[:4096]
    arrays["bn_running_mean.stem.1"] = enc.stem[1].running_mean
    arrays["bn_running_var.backbone.14.1.fc2.1"] = enc.backbone[14][1].fc2[1].running_var
    enc.eval()
    with torch.no_grad():
        arrays["out_eval"] = enc(x)
    save("encoder", **arrays)


def make_simclr(ref):
    cfg = dict(synth.DEFAULT_CFG)
    cfg["bsz_train"] = 4
    B = 4
    model = ref.simclr.SimCLR(cfg, encoder=ref.graph_encoder.GraphEncoder(cfg=cfg, in_channels=cfg["n_filters"], k=3))
    arrays = {"keys": np.array(list(model.state_dict().keys())),
              "shapes": np.array([",".join(map(str, v.shape)) for v in model.state_dict().values()])}
    load_synth(model, 101)
    s_i, s_j = synth.synth_spec(B, 111)
    model.train()
    h_i, h_j, z_i, z_j = model(s_i, s_j)
    loss = ref.ntxent.ntxent_loss(z_i, z_j, cfg)
    loss.backward()
    arrays.update(spec_i=s_i, spec_j=s_j, h_i=h_i, h_j=h_j, z_i=z_i, z_j=z_j, loss=loss)
    arrays["grad_norm"] = np.array([float(p.grad.double().norm()) if p.grad is not None else -1.0
                                    for _, p in model.named_parameters()])
    arrays["grad_names"] = np.array([n for n, _ in model.named_parameters()])
    arrays["peaks_i"] = model.peak_extractor(s_i)
    # fingerprints + retrieval on a small synthetic DB (config 5 in miniature).  Like generate.py
    # (:34-47,67-72), which never calls model.eval(), BatchNorm runs on batch statistics here.
    with torch.no_grad():
        db_specs, q_specs = synth.synth_spec(32, 121)
        _, _, db, _ = model(db_specs, db_specs)
        _, _, q, _ = model(q_specs[:16], q_specs[:16])
    arrays.update(db=db, queries=q)
    d = (q * q).sum(1, keepdim=True) - 2 * q @ db.T + (db * db).sum(1)[None]
    arrays["top1"] = torch.argmin(d, dim=1)
    best2 = torch.topk(-d, 2, dim=1).values
    print("retrieval top1", arrays["top1"].tolist(), "min margin", float((best2[:, 0] - best2[:, 1]).min()))
    save("simclr", **arrays)


def make_retrieval(ref):
    """Top-1 retrieval on a synthetic fingerprint DB whose margins are far above the embedding noise (the check of
    the north star: "identical top-1 retrieval hits on a synthetic fingerprint DB").  Eval-mode model (running
    statistics), 64 DB segments, 32 queries = DB segments + 0.02 dB of white noise (a random-weight encoder is chaotic in its graphs: 0.1 dB already flips hits); the generator asserts that every
    query's best candidate leads the runner-up by > 0.05 in inner product, so no k-NN tie can flip a hit."""
    cfg = dict(synth.DEFAULT_CFG)
    cfg["bsz_train"] = 32
    model = ref.simclr.SimCLR(cfg, encoder=ref.graph_encoder.GraphEncoder(cfg=cfg, in_channels=cfg["n_filters"], k=3))
    load_synth(model, 101)
    db_specs, _ = synth.synth_spec(64, 131)
    # calibrate the BatchNorm running statistics on the DB itself (one train-mode pass with momentum 1), as a trained
    # checkpoint's would be; the calibrated buffers are stored so the device model evaluates the same function
    bns = [m for m in model.modules() if isinstance(m, torch.nn.BatchNorm2d)]
    for m in bns:
        m.momentum = 1.0
    model.train()
    with torch.no_grad():
        model(db_specs, db_specs)
    model.eval()
    buffers = {f"buf.{k}": v for k, v in model.state_dict().items() if k.endswith("running_mean") or k.endswith("running_var")}
    pick = torch.randperm(64, generator=torch.Generator().manual_seed(132))[:32]
    q_specs = db_specs[pick] + 0.02 * torch.randn(32, 64, 32, generator=torch.Generator().manual_seed(133))
    with torch.no_grad():
        db = torch.cat([model(db_specs[i:i + 32], db_specs[i:i + 32])[2] for i in (0, 32)])
        q = model(q_specs, q_specs)[2]
    sims = q @ db.T
    best2 = torch.topk(sims, 2, dim=1).values
    margin = best2[:, 0] - best2[:, 1]
    top1 = sims.argmax(1)
    print("retrieval: hits", int((top1 == pick).sum()), "/ 32, min margin", float(margin.min()))
    assert float(margin.min()) > 0.05
    save("retrieval", q_specs=q_specs, pick=pick, db=db, queries=q, top1=top1, margin=margin, **buffers)


def make_fingerprints():
    """configs[4] at its stated size (10 000 DB segments, 1 000 queries, top-1 by inner product) through the reference
    algorithm as oracle/grafp_oracle.py restates it (pinned to the upstream modules by the fixtures above), run eager in
    fp32 on a B200 with TF32 off, as test_fingerprint_generation_at_size_matches_the_reference_on_the_same_gpu runs
    everything else.  Needs the built library and a CUDA device, no upstream checkout:

        python tests/golden/make_golden.py fingerprints

    BatchNorm running statistics as a trained checkpoint would carry them: one train-mode pass (momentum 1) of the
    device model over 512 DB segments; the test loads the stored statistics, so both sides evaluate the same function.
    Stored: those statistics, the query hits and their margins over the runner-up, and a seeded sample of 768 DB
    fingerprints (the whole DB is 5 MB)."""
    from oracle import grafp_oracle as O
    from grafp_b200.encoder.graph_encoder import GraphEncoder
    from grafp_b200.simclr.simclr import SimCLR
    dev = torch.device("cuda")
    torch.backends.cudnn.enabled = True
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    cfg = dict(synth.DEFAULT_CFG)
    n_db, n_q, chunk = 10_000, 1_000, 128
    torch.manual_seed(0)
    model = SimCLR(cfg, GraphEncoder(cfg=cfg, in_channels=cfg["n_filters"], k=3))
    load_synth(model, 303)
    db_specs, _ = synth.synth_spec(n_db, 7)
    model.to(dev).train()
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.momentum = 1.0
    with torch.no_grad():
        model(db_specs[:512].to(dev), db_specs[:512].to(dev))
    p = {k: v.detach().clone() for k, v in model.state_dict().items()}
    buffers = {f"buf.{k}": v for k, v in p.items() if k.endswith("running_mean") or k.endswith("running_var")}
    pick = torch.randperm(n_db, generator=torch.Generator().manual_seed(8))[:n_q]
    q_specs = db_specs[pick] + 0.02 * torch.randn(n_q, 64, 32, generator=torch.Generator().manual_seed(9))

    def fingerprints(specs):
        with torch.no_grad():
            return torch.cat([O.simclr_forward(p, specs[lo:lo + chunk].to(dev), specs[:1].to(dev), False, k=3)[2]
                              for lo in range(0, specs.shape[0], chunk)])

    db, q = fingerprints(db_specs), fingerprints(q_specs)
    sims = q @ db.T
    best2 = sims.topk(2, dim=1).values
    top1 = sims.argmax(1).cpu()
    sample = torch.randperm(n_db, generator=torch.Generator().manual_seed(10))[:768].sort().values
    print(torch.cuda.get_device_name(), "fingerprints at size: hits", int((top1 == pick).sum()), f"/ {n_q}")
    save("fingerprints", top1=top1.int(), margin=best2[:, 0] - best2[:, 1], sample=sample.int(),
         db_sample=db[sample.to(dev)], **buffers)


def main():
    only = set(sys.argv[1:])
    if "fingerprints" in only:
        make_fingerprints()
        only.discard("fingerprints")
        if not only:
            return
    ref = _reference_import.load()
    torch.manual_seed(0)
    for name, fn in (("knn", make_knn), ("knn_cos", make_knn_cos), ("aggregate", make_aggregate), ("gconv", make_gconv), ("gconv_r2", make_gconv_r2),
                     ("grapher", make_grapher), ("encoder", make_encoder), ("simclr", make_simclr), ("retrieval", make_retrieval)):
        if not only or name in only:
            fn(ref)


if __name__ == "__main__":
    main()
