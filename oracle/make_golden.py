"""Generate tests/golden/*.pt from the reference's own model code.

TEST INFRASTRUCTURE ONLY.  Run in the build container (needs /root/reference):

    python -m oracle.make_golden

The reference ships no golden vectors (SURVEY.md section 4), so these fixtures
are outputs of the reference itself -- embedder_eDOS/DOSTransformer.py and
embedder_phDOS/DOSTransformer_phonon.py imported unchanged behind
oracle/shims.py -- on seeded synthetic batches
(dostransformer_b200/synthetic.py).  Loss lines follow main_eDOS.py:111-123 and
main_phDOS.py:109-114.

Fixtures
  edos_small.pt / phonon_small.pt   hidden=32: outputs, loss and every live gradient in (arbiter) fp64,
                                    outputs and loss in the model dtype, and per gradient the model
                                    dtype's distance from fp64 (see compact()).
  edos_h256.pt / phonon_h256.pt     hidden=256, torch.manual_seed(0) init (weights NOT stored: the
                                    product model must reproduce them from the seed), outputs, loss,
                                    per-parameter gradient summaries, fp32 and fp64.
"""
from __future__ import annotations

import hashlib
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dostransformer_b200.synthetic import make_edos_batch, make_phonon_batch  # noqa: E402
from oracle import reference_loader  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _edos_loss(dg, ds, g, beta=1.0):
    zero = torch.tensor(0, dtype=g.y_ft.dtype)
    y_ft = torch.where(g.y_ft < 0, zero, g.y_ft)
    y = y_ft.reshape(len(g.mp_id), -1)
    return torch.sqrt(((y - dg) ** 2).mean(dim=1)).mean() + beta * torch.sqrt(((y - ds) ** 2).mean(dim=1)).mean()


def _phonon_loss(dg, ds, g, beta=1.0):
    crit = torch.nn.MSELoss()
    return torch.sqrt(crit(dg, g.phdos)).mean() + beta * torch.sqrt(crit(ds, g.phdos)).mean()


def _cast_batch(g, dtype):
    h = g.clone()
    for k in h.keys():
        v = getattr(h, k)
        if torch.is_tensor(v) and v.is_floating_point():
            setattr(h, k, v.to(dtype))
    return h


def _run(model, g, loss_fn):
    model.train()
    model.zero_grad(set_to_none=True)
    dg, x, ds = model(g)
    loss = loss_fn(dg, ds, g)
    loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}
    dead = sorted(k for k, p in model.named_parameters() if p.grad is None)
    return dict(dos_global=dg.detach().clone(), x=x.detach().clone(), dos_system=ds.detach().clone(),
                loss=loss.detach().clone(), grads=grads, dead=dead)


def _relerr(a, b):
    """max |a - b| / max |b|, as tests/conftest.py:relerr."""
    a, b = a.detach().double(), b.detach().double()
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _rel_l2(a, b):
    a, b = a.detach().double(), b.detach().double()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def digest(d: dict) -> str:
    """SHA-256 over the names, dtypes, shapes and bytes of a dict's tensors (other values by repr)."""
    h = hashlib.sha256()
    for k, v in d.items():
        h.update(k.encode())
        if torch.is_tensor(v):
            h.update(f"{v.dtype}{tuple(v.shape)}".encode())
            h.update(v.detach().contiguous().cpu().numpy().tobytes())
        else:
            h.update(repr(v).encode())
    return h.hexdigest()


def compact(fx, kind, batch_args):
    """The stored form of a small fixture.  The initial weights and the batch are kept as what draws them - the init seed
    with the model's own constructor, the synthetic generator's arguments - plus a digest of their bytes: expand() redraws
    them and checks the digest, so a fixture still holds the reference's weights bit for bit.  Of the model-dtype gradients
    only what the tests read is kept: per tensor, their max-norm and L2 distance from the fp64 arbiter.  An fp64 model is
    its own arbiter: its *64 outputs are the same tensors."""
    sd, batch, grads = fx.pop("state_dict"), fx.pop("batch"), fx.pop("grads")
    fx.pop("state_keys")
    fx.update(model=kind, state_dict_sha256=digest(sd), batch_args=batch_args, batch_keys=list(batch),
              batch_sha256=digest(batch),
              grads_noise={k: (_relerr(v, fx["grads64"][k]), _rel_l2(v, fx["grads64"][k])) for k, v in grads.items()})
    for k in ("loss", "dos_global", "dos_system", "x"):
        if fx[k].dtype == fx[k + "64"].dtype and torch.equal(fx[k], fx[k + "64"]):
            fx[k + "64"] = fx[k]
    flat = torch.cat([v.reshape(-1) for v in fx["grads64"].values()])     # one storage in the file, not one per tensor
    ends = torch.tensor([v.numel() for v in fx["grads64"].values()]).cumsum(0).tolist()
    fx["grads64"] = {k: flat[e - v.numel():e].view(v.shape) for (k, v), e in zip(fx["grads64"].items(), ends)}
    return fx


def expand(fx):
    """Inverse of compact() (fixtures without a weight digest are returned as they are)."""
    if "state_dict_sha256" not in fx:
        return fx
    from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer
    from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon
    cls = {"edos": DOSTransformer, "phonon": DOSTransformer_phonon}[fx["model"]]
    prev = torch.get_default_dtype()
    with torch.random.fork_rng(devices=[]):
        torch.set_default_dtype(getattr(torch, fx["dtype"].split(".")[-1]))
        try:
            torch.manual_seed(fx["init_seed"])
            sd = {k: v.detach().clone() for k, v in cls(*fx["ctor_args"]).state_dict().items()}
        finally:
            torch.set_default_dtype(prev)
    g = {"edos": make_edos_batch, "phonon": make_phonon_batch}[fx["model"]](**fx["batch_args"])
    batch = {k: getattr(g, k) for k in fx["batch_keys"]}
    if digest(sd) != fx["state_dict_sha256"]:
        raise AssertionError(f"{fx['model']} fixture: the initial weights drawn from seed {fx['init_seed']} are not the "
                             "reference's (the model's parameter order or initialisation changed)")
    if digest(batch) != fx["batch_sha256"]:
        raise AssertionError(f"{fx['model']} fixture: synthetic batch {fx['batch_args']} is not the stored one (the "
                             "generator changed)")
    fx.update(state_dict=sd, batch=batch)
    return fx


def _summ(gr):
    return {k: dict(norm=v.double().norm().item(), sum=v.double().sum().item(),
                    head=v.flatten()[:8].clone(), shape=tuple(v.shape)) for k, v in gr.items()}


def _fixture(cls, ctor_args, g, loss_fn, dtype, store_weights, seed=0):
    torch.set_default_dtype(dtype)
    torch.manual_seed(seed)
    model = cls(*ctor_args)
    res = _run(model, g, loss_fn)
    # fp64 arbiter from the same weights
    torch.set_default_dtype(torch.float64)
    m64 = cls(*ctor_args)
    m64.load_state_dict({k: (v.double() if v.is_floating_point() else v) for k, v in model.state_dict().items()})
    res64 = _run(m64, _cast_batch(g, torch.float64), loss_fn)
    torch.set_default_dtype(torch.float32)
    fx = dict(ctor_args=ctor_args[:-2] + ("cpu", ctor_args[-1]), init_seed=seed, dtype=str(dtype),
              state_keys=[(k, tuple(v.shape), str(v.dtype)) for k, v in model.state_dict().items()],
              dead=res["dead"], loss=res["loss"], loss64=res64["loss"],
              dos_global=res["dos_global"], dos_system=res["dos_system"],
              dos_global64=res64["dos_global"], dos_system64=res64["dos_system"])
    if store_weights:
        fx.update(state_dict={k: v.clone() for k, v in model.state_dict().items()},
                  batch={k: getattr(g, k) for k in g.keys()}, x=res["x"], x64=res64["x"],
                  grads=res["grads"], grads64=res64["grads"])
    else:
        fx.update(x_sum=res["x"].double().sum().item(), x_norm=res["x"].double().norm().item(),
                  x64_norm=res64["x"].norm().item(), x_head=res["x"][:4, :8].clone(),
                  grads=_summ(res["grads"]), grads64=_summ(res64["grads"]),
                  weights=_summ({k: v for k, v in model.state_dict().items() if v.is_floating_point()}))
    return fx


def main():
    os.makedirs(OUT, exist_ok=True)
    EDOS, PHONON, _ = reference_loader.load()
    cpu = torch.device("cpu")

    args = dict(B=4, seed=2001, mean_atoms=6.0, max_atoms=14)
    fx = _fixture(EDOS, (3, 2, 200, 41, 2, 32, cpu, 0.0), make_edos_batch(**args), _edos_loss, torch.float32, True)
    torch.save(compact(fx, "edos", args), os.path.join(OUT, "edos_small.pt"))

    g = make_edos_batch(8, seed=2002)
    fx = _fixture(EDOS, (3, 2, 200, 41, 2, 256, cpu, 0.0), g, _edos_loss, torch.float32, False)
    fx["batch_seed"] = 2002
    fx["batch_B"] = 8
    torch.save(fx, os.path.join(OUT, "edos_h256.pt"))

    args = dict(B=3, seed=1001, K=8, max_atoms=6)
    fx = _fixture(PHONON, (3, 2, 118, 4, 32, cpu, 0.0), make_phonon_batch(**args), _phonon_loss, torch.float64, True)
    torch.save(compact(fx, "phonon", args), os.path.join(OUT, "phonon_small.pt"))

    g = make_phonon_batch(1, seed=1002)
    fx = _fixture(PHONON, (3, 2, 118, 4, 256, cpu, 0.0), g, _phonon_loss, torch.float64, False)
    fx["batch_seed"] = 1002
    fx["batch_B"] = 1
    torch.save(fx, os.path.join(OUT, "phonon_h256.pt"))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
