"""The batch body of reference utils/train.py:51-85 (encoder -> decoder -> Chamfer / MSE / EMD / Hungarian MSE (+L1/L2) -> backward ->
two Adams) as a fixed sequence of fused kernels over flat buffers.

* all parameters of encoder and decoder live in ONE flat fp32 buffer (the nn.Linear parameters are
  re-homed as views, so ``state_dict`` / checkpoints are unaffected); gradients, Adam moments likewise;
* forward + loss + backward is a fixed list of C-ABI launches with preallocated activations -- captured
  once into a CUDA graph and replayed (the reference pays ~10^3 ATen launches and a ``.item()`` sync per
  batch, utils/train.py:77);
* data parallel: jets are independent, each rank runs its shard and the only collective is ONE
  all-reduce(sum) of the flat gradient buffer (the loss is a sum over jets, chamfer_loss.py:35,40, so sum
  reproduces the single-process gradient); the two reference Adams (utils/initialize.py:152-153) have equal
  hyper-parameters and are elementwise, so one fused flat Adam is identical to both.
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Optional

import numpy as np
import torch

from . import _lib, ops
from .losses import EMDLoss, _norm_id
from .models.const import GLOBAL_MIX, LOCAL_MIX

POLAR_EPS = 1e-16      # utils/const.py:5 (clamp of (E, pT) in polar coordinates, utils/train.py:58-65)


# --------------------------------------------------------------------------------------------------
# host-side helpers (no CUDA needed: covered by the CPU / gloo tests)
# --------------------------------------------------------------------------------------------------
def synthetic_jets(batch: int, num_particles: int, seed: int = 1234, dtype=np.float32) -> np.ndarray:
    """JetNet-shaped jets (B,N,3) = [pt_rel, eta_rel, phi_rel] (feature order of the reference's
    utils/data/preprocess.py:75-76): eta,phi ~ N(0, 0.1^2) clipped to +-0.5; pt_rel ~ Dirichlet(0.5) sorted
    descending (JetNet is pT ordered); n ~ UniformInt[N/3, N] real particles, the rest zero padded."""
    rng = np.random.default_rng(seed)
    eta = np.clip(rng.normal(0.0, 0.1, (batch, num_particles)), -0.5, 0.5)
    phi = np.clip(rng.normal(0.0, 0.1, (batch, num_particles)), -0.5, 0.5)
    pt = rng.dirichlet(np.full(num_particles, 0.5), size=batch)
    pt = -np.sort(-pt, axis=1)
    n = rng.integers(max(1, num_particles // 3), num_particles + 1, size=batch)
    mask = np.arange(num_particles)[None, :] < n[:, None]
    x = np.stack([pt, eta, phi], axis=-1) * mask[..., None]
    return x.astype(dtype)


def shard_range(global_batch: int, rank: int, world_size: int):
    """Jets [lo, hi) of rank ``rank``: contiguous shards, the remainder spread over the first ranks."""
    base, rem = divmod(global_batch, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def flat_layout(encoder, decoder) -> "OrderedDict[str, tuple]":
    """name -> (offset, shape) of every parameter in the flat buffer.  Order: encoder GraphNet steps in kernel
    packing order, encoder mix layer, decoder input linear, decoder GraphNet steps."""
    out, off = OrderedDict(), 0

    def add(name, p):
        nonlocal off
        out[name] = (off, tuple(p.shape))
        off += p.numel()

    def add_graphnet(prefix, g):
        for t in range(g.num_mps):
            for kind, net in (("edge_net", g.edge_net[t]), ("node_net", g.node_net[t])):
                for k, layer in enumerate(net):
                    add(f"{prefix}{kind}.{t}.{k}.weight", layer.weight)
                    add(f"{prefix}{kind}.{t}.{k}.bias", layer.bias)

    add_graphnet("encoder.encoder.", encoder.encoder)
    if hasattr(encoder, "mix_layer"):
        add("encoder.mix_layer.weight", encoder.mix_layer.weight)
        if encoder.mix_layer.bias is not None:
            add("encoder.mix_layer.bias", encoder.mix_layer.bias)
    add("decoder.linear.weight", decoder.linear.weight)
    add("decoder.linear.bias", decoder.linear.bias)
    add_graphnet("decoder.decoder.", decoder.decoder)
    return out


def layout_size(layout) -> int:
    return sum(int(np.prod(s)) for _, s in layout.values())


def allreduce_flat_(grad: torch.Tensor, group=None) -> torch.Tensor:
    """The path's only collective: sum the flat gradient buffer over the data-parallel ranks."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(grad, op=dist.ReduceOp.SUM, group=group)
    return grad


# --------------------------------------------------------------------------------------------------
# the fused step
# --------------------------------------------------------------------------------------------------
def _with_batch(desc, batch: int):
    """A copy of a message-passing step descriptor for ``batch`` jets."""
    d = _lib.MPDesc.from_buffer_copy(desc)
    d.batch = int(batch)
    return d


def _on_trainer_device(fn):
    """Runs a trainer method with the trainer's GPU as the current device (launchers and streams follow the current device)."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *args, **kw):
        with torch.cuda.device(self.dev):
            return fn(self, *args, **kw)
    return wrapper


class GNNAETrainer:
    """One optimisation step per call, on the caller's CUDA device.

    >>> tr = GNNAETrainer(encoder, decoder, batch_size=4096)
    >>> loss = tr.step(x_host_pinned)          # float; H2D copy, graph replay, all-reduce, Adam, D2H of the loss

    Covers every latent map of the reference ('mean', 'max', 'min', the GLOBAL_MIX and LOCAL_MIX spellings), the decoder's
    ``normalize_output`` (tanh), the polar-coordinate clamp of utils/train.py:55-65 (``polar_coord``) and the Chamfer, MSE,
    EMD and Hungarian MSE branches of ``get_loss`` (utils/train.py:330-385, ``loss_choice``).  Dropout and batch-norm are not part of the fused step
    (the reference's batch-norm path crashes; dropout > 0 raises in the modules).

    ``loss_choice="emd"`` trains with the exact energy mover's distance (one gj_emd_loss solve of the whole batch per step, inside
    the CUDA graph).  Its options come from ``emd_loss`` (default ``EMDLoss(polar_coord=polar_coord)``): R, beta, norm,
    periodic_phi, polar_coord (must equal the trainer's) and reduction ("sum" over the jets, or "mean" over the global batch;
    "none" raises).  Cartesian 3- / 4-vectors are converted as EMDLoss converts them; at most 150 particles per jet.  A jet whose
    solver stops at its augmentation cap makes ``loss_from_stats`` (``step``, ``run_epoch``) raise.

    ``loss_choice="hungarian"`` trains with the Hungarian-matched MSE of ``HungarianMSELoss`` (one gj_hungarian_mse_loss launch of the
    whole batch per step, inside the CUDA graph): the step computes ``HungarianMSELoss()(recon, x, abs_coord=hungarian_abs_coord,
    polar_coord=hungarian_polar_coord)`` on the reconstruction after tanh and the polar clamp, the mean over the B N D' elements of
    the global batch (D' = the input width in absolute Cartesian coordinates, else 3).  No gradient flows through the matching.  At
    most 220 particles per jet.

    ``partial_batches`` (default off: every batch has exactly ``batch_size`` jets, and any other size raises) also accepts
    batches of 1 <= B' < batch_size jets in ``step``, ``step_async``, ``load_batch`` / ``compute_gradients``, ``forward_only`` and
    ``run_epoch`` (its last batch), such as the tail a ``DataLoader`` without ``drop_last`` yields.  The first batch of a size
    builds that size's plan: the step descriptors and loss scales of B' (MSE over world B' N D elements, EMD "mean" 1/(world B'),
    Hungarian 1/(world B' N D')), with every activation, gradient and loss buffer a prefix view of the full-size one; with
    ``use_cuda_graph`` it also captures that size's graph.  A B'-jet step then returns exactly what a trainer built with
    ``batch_size=B'`` returns, and allocates no device memory: the workspace, saved and partials buffers are sized at
    construction for every batch of up to ``batch_size`` jets.  Not with data parallelism: for ``world > 1`` a short batch raises
    ``NotImplementedError`` -- the mean reductions would need the global jet count, which ranks with different tails only learn
    through an extra collective.

    ``batched_launches`` (default on, used where every step runs the fused tensor-core kernels): the six message-passing steps
    run as a chain -- ONE launch packs all steps' bf16 edge-parameter images, ONE launch reduces all steps' parameter-gradient
    partials (gj_mp_steps_pack / gj_mp_steps_reduce) -- instead of one of each per step; identical results.
    """

    def __init__(self, encoder, decoder, batch_size: int, *, lr: float = 1e-5, betas=(0.9, 0.999), eps: float = 1e-8,
                 l1_lambda: float = 1e-8, l2_lambda: float = 0.0, loss_norm_choice: str = "cartesian",
                 jet_features_weight: float = 1.0, chamfer_mode: str = "intended", encoder_metric: str = "euclidean",
                 decoder_metric: str = "euclidean", process_group=None, use_cuda_graph: bool = True,
                 loss_choice: str = "chamfer", polar_coord: bool = False, optimizer: str = "adam",
                 batched_launches: bool = True, emd_loss: Optional[EMDLoss] = None, hungarian_abs_coord: bool = True,
                 hungarian_polar_coord: bool = False, partial_batches: bool = False):
        self.enc, self.dec = encoder, decoder
        g_e, g_d = encoder.encoder, decoder.decoder
        dev = next(encoder.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("GNNAETrainer needs the models on a CUDA device (there is no CPU fallback)")
        if g_e.batch_norm or g_d.batch_norm or g_e.dropout_p > 0 or g_d.dropout_p > 0:
            raise NotImplementedError("batch_norm / dropout are not part of the fused step")
        canon = encoder.latent_map.lower().replace(" ", "_")
        if canon in GLOBAL_MIX:
            self.map = "global"
        elif canon in LOCAL_MIX:
            self.map = "local"
        elif canon in ("max", "min"):
            self.map = canon
        else:
            self.map = "mean"
        self.optimizer = str(optimizer).lower()      # utils/initialize.py:148-172
        if self.optimizer != "adam" and self.optimizer not in ops.OPTIMIZERS:
            raise NotImplementedError("Other choices of optimizer are not implemented. Available choices are 'Adam' and 'RMSprop', "
                                      f"'Adagrad', 'SGD'. Found: {optimizer}.")
        lc = str(loss_choice).lower()
        if lc in ("chamfer", "chamferloss", "chamfer_loss"):
            self.loss_choice = "chamfer"
        elif lc in ("mse", "mseloss", "mse_loss"):
            self.loss_choice = "mse"
        elif lc in ("emd", "emdloss", "emd_loss"):
            self.loss_choice = "emd"
        elif lc in ("hungarian", "hungarian_mse", "hungarianmse", "hungarian_mse_loss", "hungarianmseloss"):
            self.loss_choice = "hungarian"
        else:
            raise NotImplementedError(f"loss_choice {loss_choice!r}: the fused step covers the Chamfer, MSE, EMD and Hungarian MSE "
                                      "branches of get_loss (utils/train.py:330-385); 'hybrid' is not covered")
        if self.loss_choice == "emd":
            if emd_loss is None:
                emd_loss = EMDLoss(polar_coord=polar_coord)
            if emd_loss.reduction == "none":
                raise ValueError("loss_choice='emd' needs a scalar loss: EMDLoss reduction 'sum' or 'mean', not 'none'")
            if emd_loss.polar_coord != bool(polar_coord):
                raise ValueError(f"EMDLoss(polar_coord={emd_loss.polar_coord}) does not match the trainer's polar_coord={polar_coord}")
            if polar_coord and encoder.input_node_size != 3:
                raise ValueError(f"polar_coord=True expects [pt, eta, phi] jets (3 features), got {encoder.input_node_size}")
            if encoder.num_nodes > 150:
                raise ValueError(f"the EMD loss supports at most 150 particles per jet, got {encoder.num_nodes}")
            self.emd = emd_loss
        if self.loss_choice == "hungarian":
            if encoder.num_nodes > 220:
                raise ValueError(f"the Hungarian MSE loss supports at most 220 particles per jet, got {encoder.num_nodes}")
            self.hmse_coords = ((_lib.GJ_HMSE_ABS_POLAR if hungarian_polar_coord else _lib.GJ_HMSE_ABS_CARTESIAN) if hungarian_abs_coord
                                else (_lib.GJ_HMSE_REL_POLAR if hungarian_polar_coord else _lib.GJ_HMSE_REL_CARTESIAN))
        if self.loss_choice == "chamfer" and chamfer_mode == "reference" and jet_features_weight == 0:
            raise UnboundLocalError("jet_loss referenced before assignment (reference chamfer_loss.py:42)")
        # the Chamfer target is the input batch: both sides must be 3- or 4-vectors of one width (distance_sq.py:31-42)
        if decoder.output_node_size != encoder.input_node_size or encoder.input_node_size not in (3, 4):
            raise ValueError(f"Dimension of q ({encoder.input_node_size}) does not match with dimension of p "
                             f"({decoder.output_node_size}), or is not 3 or 4.")
        self.dev, self.B, self.N = dev, int(batch_size), encoder.num_nodes
        self.batch_size, self.partial_batches = self.B, bool(partial_batches)
        self.lr, self.betas, self.eps = lr, betas, eps
        self.l1, self.l2 = float(l1_lambda), float(l2_lambda)
        self.wc, self.wj = (0.0, 1.0) if chamfer_mode == "reference" else (1.0, float(jet_features_weight))
        self.norm_choice = loss_norm_choice
        self.group = process_group
        self.step_count = 0
        self.lib = _lib.load()

        # ---- flat parameter / gradient / moment buffers; modules re-homed as views ----
        self.layout = flat_layout(encoder, decoder)
        n = layout_size(self.layout)
        self.flat = torch.empty(n, device=dev, dtype=torch.float32)
        self.grad = torch.zeros(n, device=dev, dtype=torch.float32)
        self.exp_avg = torch.zeros(n, device=dev, dtype=torch.float32)
        self.exp_avg_sq = torch.zeros(n, device=dev, dtype=torch.float32)
        named = OrderedDict([("encoder." + k, p) for k, p in encoder.named_parameters()] +
                            [("decoder." + k, p) for k, p in decoder.named_parameters()])
        assert set(named) == set(self.layout), "flat layout does not cover the models' parameters"
        n_e = g_e.num_flat_params
        g_e.flatten_parameters(self.flat[:n_e])
        with torch.no_grad():
            for name, (off, shape) in self.layout.items():
                p = named[name]
                seg = self.flat[off:off + p.numel()].view(shape)
                if p.data_ptr() != seg.data_ptr():
                    seg.copy_(p.detach().to(torch.float32))
                    p.data = seg
                p.grad = self.grad[off:off + p.numel()].view(shape)
        off_d = self.layout["decoder.decoder.edge_net.0.0.weight"][0]
        g_d._flat = self.flat[off_d:off_d + g_d.num_flat_params]
        g_d._step_offsets, o = [], 0
        for t in range(g_d.num_mps):
            c = sum(p.numel() for p in g_d.step_parameters(t))
            g_d._step_offsets.append((o, c))
            o += c
        assert g_e._flat_ok() and g_d._flat_ok()
        g_e._flat_owner = g_d._flat_owner = self      # forward raises (instead of silently re-packing) if the views break

        # ---- activations ----
        B, N = self.B, self.N
        f32 = dict(device=dev, dtype=torch.float32)
        self.F = encoder.input_node_size
        self.x = torch.zeros((B, N, self.F), **f32)
        self.enc_steps = self._plan_graphnet(g_e, 0, self.F, encoder_metric)
        self.dec_steps = self._plan_graphnet(g_d, off_d, decoder.node_sizes[0][0], decoder_metric)
        self.enc_out_w = g_e.output_node_size
        self.latent_w = encoder.latent_node_size
        self.h0 = decoder.node_sizes[0][0]
        zshape = (B, N * self.latent_w) if self.map == "local" else (B, self.latent_w)
        self.latent = torch.empty(zshape, **f32)
        self.dlatent = torch.empty(zshape, **f32)
        self.dec_in = torch.empty((B, N, self.h0), **f32)
        self.d_dec_in = torch.empty((B, N, self.h0), **f32)
        self.d_enc_out = torch.empty((B, N, self.enc_out_w), **f32)
        self.dx = torch.zeros((B, N, self.F), **f32)
        # decoder output -> [tanh] -> [clamp of (E, pT) / pT at EPS] -> loss (decoder.py:123-124, train.py:55-65)
        D = decoder.output_node_size
        self.use_tanh = bool(decoder.normalize_output)
        self.clamp_mask = (3 if D == 4 else 1) if polar_coord else 0
        self.recon_raw = self.dec_steps[-1]["out"]
        self.transform = self.use_tanh or self.clamp_mask != 0
        self.recon = torch.empty_like(self.recon_raw) if self.transform else self.recon_raw
        self.dp = torch.empty_like(self.recon)
        self.dp_raw = torch.empty_like(self.recon) if self.transform else self.dp
        self.world = 1
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            self.world = torch.distributed.get_world_size(process_group)
        if self.loss_choice == "emd":
            self.emd_flags = (_lib.GJ_EMD_NORM if self.emd.norm else 0) | (_lib.GJ_EMD_PERIODIC_PHI if self.emd.periodic_phi else 0)
        if self.loss_choice == "hungarian":
            self.hmse_d = D if self.hmse_coords == _lib.GJ_HMSE_ABS_CARTESIAN else 3
        self.emd_scale, self.hmse_scale = self._loss_scales(B)
        self.jet_terms = torch.empty((B, 2), **f32)
        # [chamfer | EMD | Hungarian squared error, jet, loss term, sum|p|, sum p^2, EMD jets whose solver hit its cap]
        self.stats = torch.zeros(8, **f32)
        self.stats_host = torch.zeros(8, dtype=torch.float32).pin_memory()
        all_steps = self.enc_steps + self.dec_steps
        ws, saved_bytes, pbytes = self._buffer_bytes(B, [s_["desc"] for s_ in all_steps])
        if self.partial_batches:
            # every smaller batch runs in these same buffers (_make_plan).  The per-CTA partials follow grids that are not monotonic
            # in the batch size (a grid capped at a few CTAs per SM evens out its tiles), so a smaller batch can need more than B
            for b in range(1, B):
                w, sv, pb = self._buffer_bytes(b, [_with_batch(s_["desc"], b) for s_ in all_steps])
                ws, saved_bytes, pbytes = max(ws, w), list(map(max, saved_bytes, sv)), list(map(max, pbytes, pb))
        self.ws_bytes = ws
        self.ws = torch.empty((self.ws_bytes + 3) // 4, **f32)
        # per-step buffers in which the forward call leaves P|Q, the packed edge parameters and the pair distances for the
        # backward call of the same step (0 bytes: that step recomputes them)
        for st_, nbytes in zip(all_steps, saved_bytes):
            st_["saved"] = torch.empty((nbytes + 3) // 4, **f32) if nbytes else None
        # per-chain helper launches (gj_mp_steps_pack / gj_mp_steps_reduce): the packed edge-parameter images of all steps in ONE
        # launch at the start of the forward pass, the parameter-gradient partials of all steps reduced in ONE launch at the end of
        # the backward pass (each step keeps its partials in its own buffer until then) -- where every step supports it
        self.batched = bool(batched_launches) and all(b > 0 for b in pbytes) and all(s_["saved"] is not None for s_ in all_steps)
        for s_, nb in zip(all_steps, pbytes):
            s_["partials"] = torch.empty((nb + 3) // 4, **f32) if self.batched else None
        self.graph = None
        self.use_graph = use_cuda_graph
        self.launches_per_step = None
        # per batch size: the plan (step descriptors, loss scales, buffers) and its CUDA graph; _use_plan swaps one in
        self._plans = {B: {k: getattr(self, k) for k in self._PLAN_ATTRS}}

    # what differs between batch sizes: swapped in as attributes, so that the launch sequence reads the resident batch's
    _PLAN_ATTRS = ("B", "x", "latent", "dlatent", "dec_in", "d_dec_in", "d_enc_out", "dx", "enc_steps", "dec_steps", "recon_raw",
                   "recon", "dp", "dp_raw", "jet_terms", "emd_scale", "hmse_scale", "graph", "launches_per_step")
    # batch-major, contiguous: the first B' rows of the full-size buffer are the buffer of a B'-jet batch
    _PREFIX_ATTRS = ("x", "latent", "dlatent", "dec_in", "d_dec_in", "d_enc_out", "dx", "recon", "dp", "dp_raw", "jet_terms")

    def _loss_scales(self, B):
        """(EMD, Hungarian MSE) gradient scales of a B-jet batch (None where that loss is not the trainer's)."""
        emd = hmse = None
        if self.loss_choice == "emd":
            # EMDLoss's reduction over the GLOBAL batch: with "mean" the all-reduced gradient equals the single-device one
            emd = 1.0 if self.emd.reduction == "sum" else 1.0 / (self.world * B)
        if self.loss_choice == "hungarian":
            # nn.functional.mse_loss's mean over the B N D' elements of the GLOBAL batch, as the MSE branch
            hmse = 1.0 / (self.world * B * self.N * self.hmse_d)
        return emd, hmse

    def _buffer_bytes(self, B, descs):
        """(workspace, [saved per step], [partials per step]) bytes that a B-jet batch of the steps ``descs`` needs."""
        lib, N = self.lib, self.N
        ws = max([lib.gj_mp_step_bwd_workspace(d) for d in descs] + [lib.gj_mp_step_fwd_workspace(d) for d in descs] +
                 [lib.gj_linear_bwd_workspace(B * N, max(self.latent_w, self.enc_out_w), max(self.h0, self.latent_w)),
                  lib.gj_linear_bwd_workspace(B, max(self.latent_w, N * self.enc_out_w), max(N * self.h0, self.latent_w)),
                  lib.gj_param_norms_workspace(self.flat.numel()), lib.gj_mse_workspace(), 16] +
                 ([lib.gj_emd_loss_workspace(B, N)] if self.loss_choice == "emd" else []) +
                 ([lib.gj_hungarian_mse_loss_workspace(B, N)] if self.loss_choice == "hungarian" else []))
        return (int(ws), [int(lib.gj_mp_step_saved_bytes(d)) for d in descs], [int(lib.gj_mp_step_partials_bytes(d)) for d in descs])

    def _make_plan(self, B):
        """The plan of a batch of B < batch_size jets: the step descriptors and loss scales of B over the full-size memory -- every
        activation, gradient and loss buffer a prefix view, the workspace, saved and partials buffers shared as they are."""
        full = self._plans[self.batch_size]
        plan = {k: full[k][:B] for k in self._PREFIX_ATTRS}
        steps = lambda ss: [dict(s, desc=_with_batch(s["desc"], B), out=s["out"][:B], e=s["e"][:B],
                                 din=None if s["din"] is None else s["din"][:B]) for s in ss]
        plan.update(B=B, enc_steps=steps(full["enc_steps"]), dec_steps=steps(full["dec_steps"]), graph=None, launches_per_step=None)
        plan["recon_raw"] = plan["dec_steps"][-1]["out"]
        plan["emd_scale"], plan["hmse_scale"] = self._loss_scales(B)
        all_steps = plan["enc_steps"] + plan["dec_steps"]
        ws, saved_bytes, pbytes = self._buffer_bytes(B, [s["desc"] for s in all_steps])
        have = lambda t: 0 if t is None else 4 * t.numel()
        if (ws > self.ws_bytes or any(n > have(s["saved"]) for n, s in zip(saved_bytes, all_steps)) or
                (self.batched and any(n > have(s["partials"]) for n, s in zip(pbytes, all_steps)))):
            raise RuntimeError(f"internal error: a batch of {B} jets needs larger workspace / saved / partials buffers than the trainer "
                               f"allocated for batches of up to {self.batch_size} jets")
        return plan

    def _use_plan(self, B):
        """Makes the plan of a B-jet batch the resident one (built the first time B appears)."""
        if B != self.B:
            plan = self._plans.get(B)
            if plan is None:
                plan = self._plans[B] = self._make_plan(B)
            self.__dict__.update(plan)

    def _jets_in(self, x) -> int:
        """The number of jets of batch ``x``.  Without ``partial_batches`` it is always ``batch_size``: a batch of another size
        then fails where it is copied in, as it always has."""
        if not self.partial_batches or x.numel() == self.batch_size * self.N * self.F:
            return self.batch_size
        if x.dim() != 3 or tuple(x.shape[1:]) != (self.N, self.F) or not 1 <= x.shape[0] <= self.batch_size:
            raise ValueError(f"batch of {tuple(x.shape)}: expected (B', {self.N}, {self.F}) with 1 <= B' <= batch_size = {self.batch_size}")
        if self.world > 1:
            raise NotImplementedError("a batch of fewer than batch_size jets with more than one data-parallel rank: the mean reductions "
                                      "would need the global jet count, which the ranks only learn through an extra collective")
        return int(x.shape[0])

    def _plan_graphnet(self, g, flat_off, in_width, metric):
        steps, off, width_in = [], flat_off, in_width
        B, N = self.B, self.N
        for t in range(g.num_mps):
            cfg = g.step_config(t, metric)
            _, H, ew, nw, alpha, mid, prec = cfg
            desc = _lib.make_desc(B, N, H, ew, nw, alpha, mid, prec, h_ld=width_in, h_cols=min(width_in, H))
            count = self.lib.gj_mp_param_count(desc)
            assert count == sum(p.numel() for p in g.step_parameters(t))
            steps.append(dict(desc=desc, off=off, count=count,
                              out=torch.empty((B, N, nw[-1]), device=self.dev, dtype=torch.float32),
                              e=torch.empty((B, N, ew[-1]), device=self.dev, dtype=torch.float32),
                              din=None))
            off += count
            width_in = nw[-1]
        # gradient w.r.t. each step's input (the first step's input gradient is produced by the kernel but unused)
        for t in range(1, g.num_mps):
            steps[t]["din"] = torch.empty_like(steps[t - 1]["out"])
        return steps

    # ---- the launch sequence ------------------------------------------------------------------------
    def _step_fwd(self, s, h, st):
        P = self.flat.data_ptr()
        if self.batched:
            ops.raw_mp_fwd_packed(s["desc"], h.data_ptr(), P + 4 * s["off"], s["out"].data_ptr(), s["e"].data_ptr(),
                                  self.ws.data_ptr(), self.ws_bytes, st, s["saved"].data_ptr())
        else:
            ops.raw_mp_fwd(s["desc"], h.data_ptr(), P + 4 * s["off"], s["out"].data_ptr(), s["e"].data_ptr(),
                           self.ws.data_ptr(), self.ws_bytes, st, s["saved"].data_ptr() if s["saved"] is not None else None)

    def _step_bwd(self, s, hin, g, din, st):
        P, G = self.flat.data_ptr(), self.grad.data_ptr()
        if self.batched:
            ops.raw_mp_bwd_deferred(s["desc"], hin.data_ptr(), s["e"].data_ptr(), P + 4 * s["off"], g.data_ptr(), din.data_ptr(),
                                    self.ws.data_ptr(), self.ws_bytes, st, s["saved"].data_ptr(), s["partials"].data_ptr())
        else:
            ops.raw_mp_bwd(s["desc"], hin.data_ptr(), s["e"].data_ptr(), P + 4 * s["off"], g.data_ptr(), din.data_ptr(),
                           G + 4 * s["off"], self.ws.data_ptr(), self.ws_bytes, st,
                           s["saved"].data_ptr() if s["saved"] is not None else None)

    def _fwd(self, st):
        lib, P = self.lib, self.flat.data_ptr()
        B, N = self.B, self.N
        h = self.x
        if self.batched:
            steps = self.enc_steps + self.dec_steps
            ops.raw_mp_pack_steps([s["desc"] for s in steps], [P + 4 * s["off"] for s in steps], [s["saved"].data_ptr() for s in steps], st)
        for s in self.enc_steps:
            self._step_fwd(s, h, st)
            h = s["out"]
        L = self.layout
        if self.map == "mean":
            _lib.check(lib.gj_latent_mean_fwd(B, N, self.enc_out_w, h.data_ptr(), self.latent.data_ptr(), st), "latent_mean_fwd")
        elif self.map in ("max", "min"):
            _lib.check(lib.gj_latent_extreme_fwd(B, N, self.enc_out_w, int(self.map == "min"), h.data_ptr(), self.latent.data_ptr(), st),
                       "latent_extreme_fwd")
        elif self.map == "global":
            _lib.check(lib.gj_linear_fwd(B, N * self.enc_out_w, self.latent_w, h.data_ptr(),
                                         P + 4 * L["encoder.mix_layer.weight"][0], None, self.latent.data_ptr(), st), "mix fwd")
        else:
            _lib.check(lib.gj_linear_fwd(B * N, self.enc_out_w, self.latent_w, h.data_ptr(),
                                         P + 4 * L["encoder.mix_layer.weight"][0], P + 4 * L["encoder.mix_layer.bias"][0],
                                         self.latent.data_ptr(), st), "mix fwd")
        ops.LAUNCHES["count"] += 1
        wl, bl = P + 4 * L["decoder.linear.weight"][0], P + 4 * L["decoder.linear.bias"][0]
        if self.map == "local":
            _lib.check(lib.gj_linear_fwd(B * N, self.latent_w, self.h0, self.latent.data_ptr(), wl, bl, self.dec_in.data_ptr(), st), "dec linear fwd")
        else:
            _lib.check(lib.gj_linear_fwd(B, self.latent_w, N * self.h0, self.latent.data_ptr(), wl, bl, self.dec_in.data_ptr(), st), "dec linear fwd")
        ops.LAUNCHES["count"] += 1
        h = self.dec_in
        for s in self.dec_steps:
            self._step_fwd(s, h, st)
            h = s["out"]
        if self.transform:
            _lib.check(lib.gj_output_transform_fwd(B * N, self.recon.shape[-1], int(self.use_tanh), self.clamp_mask, POLAR_EPS,
                                                   self.recon_raw.data_ptr(), self.recon.data_ptr(), st), "output transform fwd")
            ops.LAUNCHES["count"] += 1

    def _loss(self, st):
        """Loss terms (+ d loss / d recon) and parameter norms of the resident batch -> self.stats."""
        lib, B, N, D = self.lib, self.B, self.N, self.recon.shape[-1]
        if self.loss_choice == "mse":      # nn.MSELoss: mean over the elements of the GLOBAL batch
            _lib.check(lib.gj_mse_fwd_bwd(B * N * D, float(self.world * B * N * D), self.recon.data_ptr(), self.x.data_ptr(),
                                          self.stats.data_ptr(), self.dp.data_ptr(), self.ws.data_ptr(), self.ws_bytes, st), "mse")
        elif self.loss_choice == "emd":    # the recon after tanh / clamp against the input, as EMDLoss sees them in the train loop
            coords = _lib.GJ_EMD_COORDS_POLAR if self.emd.polar_coord else _lib.GJ_EMD_COORDS_CARTESIAN
            _lib.check(lib.gj_emd_loss(B, N, D, coords, self.recon.data_ptr(), self.x.data_ptr(), self.emd.R, self.emd.beta,
                                       self.emd_flags, self.emd_scale, self.stats.data_ptr(), self.stats.data_ptr() + 20,
                                       self.dp.data_ptr(), self.ws.data_ptr(), self.ws_bytes, st), "emd loss")
        elif self.loss_choice == "hungarian":    # likewise, as HungarianMSELoss sees them
            _lib.check(lib.gj_hungarian_mse_loss(B, N, D, self.hmse_coords, self.recon.data_ptr(), self.x.data_ptr(), self.hmse_scale,
                                                 self.stats.data_ptr(), self.dp.data_ptr(), None, self.ws.data_ptr(), self.ws_bytes, st),
                       "hungarian mse loss")
        else:
            _lib.check(lib.gj_chamfer_fwd_bwd(B, N, N, D, _norm_id(self.recon, self.norm_choice), self.wc, self.wj,
                                              self.recon.data_ptr(), self.x.data_ptr(), self.jet_terms.data_ptr(),
                                              self.stats.data_ptr(), self.dp.data_ptr(), st), "chamfer")
        _lib.check(lib.gj_param_norms(self.flat.data_ptr(), self.flat.numel(), self.stats.data_ptr() + 12, self.ws.data_ptr(),
                                      self.ws_bytes, st), "norms")
        ops.LAUNCHES["count"] += 4

    def _loss_and_bwd(self, st):
        lib, P, G = self.lib, self.flat.data_ptr(), self.grad.data_ptr()
        B, N, L = self.B, self.N, self.layout
        self._loss(st)
        if self.transform:
            _lib.check(lib.gj_output_transform_bwd(B * N, self.recon.shape[-1], int(self.use_tanh), self.clamp_mask, POLAR_EPS,
                                                   self.recon_raw.data_ptr(), self.dp.data_ptr(), self.dp_raw.data_ptr(), st),
                       "output transform bwd")
            ops.LAUNCHES["count"] += 1
        # decoder GraphNet, last step first
        g = self.dp_raw
        for t in reversed(range(len(self.dec_steps))):
            s = self.dec_steps[t]
            hin = self.dec_in if t == 0 else self.dec_steps[t - 1]["out"]
            din = self.d_dec_in if t == 0 else s["din"]
            self._step_bwd(s, hin, g, din, st)
            g = din
        wl = L["decoder.linear.weight"][0]
        bl = L["decoder.linear.bias"][0]
        if self.map == "local":
            _lib.check(lib.gj_linear_bwd(B * N, self.latent_w, self.h0, self.latent.data_ptr(), P + 4 * wl, g.data_ptr(),
                                         self.dlatent.data_ptr(), G + 4 * wl, G + 4 * bl, self.ws.data_ptr(), self.ws_bytes, st), "dec linear bwd")
        else:
            _lib.check(lib.gj_linear_bwd(B, self.latent_w, N * self.h0, self.latent.data_ptr(), P + 4 * wl, g.data_ptr(),
                                         self.dlatent.data_ptr(), G + 4 * wl, G + 4 * bl, self.ws.data_ptr(), self.ws_bytes, st), "dec linear bwd")
        ops.LAUNCHES["count"] += 3
        y = self.enc_steps[-1]["out"]
        if self.map == "mean":
            _lib.check(lib.gj_latent_mean_bwd(B, N, self.enc_out_w, self.dlatent.data_ptr(), self.d_enc_out.data_ptr(), st), "latent_mean_bwd")
            ops.LAUNCHES["count"] += 1
        elif self.map in ("max", "min"):
            _lib.check(lib.gj_latent_extreme_bwd(B, N, self.enc_out_w, y.data_ptr(), self.latent.data_ptr(), self.dlatent.data_ptr(),
                                                 self.d_enc_out.data_ptr(), st), "latent_extreme_bwd")
            ops.LAUNCHES["count"] += 1
        elif self.map == "global":
            wm = L["encoder.mix_layer.weight"][0]
            _lib.check(lib.gj_linear_bwd(B, N * self.enc_out_w, self.latent_w, y.data_ptr(), P + 4 * wm, self.dlatent.data_ptr(),
                                         self.d_enc_out.data_ptr(), G + 4 * wm, None, self.ws.data_ptr(), self.ws_bytes, st), "mix bwd")
            ops.LAUNCHES["count"] += 3
        else:
            wm, bm = L["encoder.mix_layer.weight"][0], L["encoder.mix_layer.bias"][0]
            _lib.check(lib.gj_linear_bwd(B * N, self.enc_out_w, self.latent_w, y.data_ptr(), P + 4 * wm, self.dlatent.data_ptr(),
                                         self.d_enc_out.data_ptr(), G + 4 * wm, G + 4 * bm, self.ws.data_ptr(), self.ws_bytes, st), "mix bwd")
            ops.LAUNCHES["count"] += 3
        g = self.d_enc_out
        for t in reversed(range(len(self.enc_steps))):
            s = self.enc_steps[t]
            hin = self.x if t == 0 else self.enc_steps[t - 1]["out"]
            din = self.dx if t == 0 else s["din"]
            self._step_bwd(s, hin, g, din, st)
            g = din
        if self.batched:
            steps = self.enc_steps + self.dec_steps
            ops.raw_mp_reduce_steps([s["desc"] for s in steps], [s["partials"].data_ptr() for s in steps],
                                    [G + 4 * s["off"] for s in steps], st)

    def _fwd_bwd(self):
        st = torch.cuda.current_stream().cuda_stream
        self._fwd(st)
        self._loss_and_bwd(st)

    # ---- public API ---------------------------------------------------------------------------------
    @_on_trainer_device
    def forward_only(self, x: torch.Tensor):
        """encoder + decoder forward on a (B,N,F) batch (host or device); returns (latent, recon) device views."""
        self.load_batch(x)
        self._fwd(torch.cuda.current_stream().cuda_stream)
        return self.latent, self.recon

    @_on_trainer_device
    def load_batch(self, x: torch.Tensor) -> None:
        """Host (ideally pinned) or device batch -> the step's resident input buffer (with ``partial_batches``, a batch of
        B' < batch_size jets makes the plan of B' the resident one)."""
        self._use_plan(self._jets_in(x))
        self.x.copy_(x.reshape(self.x.shape), non_blocking=True)

    @_on_trainer_device
    def compute_gradients(self) -> None:
        """forward + loss + backward on the resident batch; the flat gradient buffer holds d(sum loss)/dp."""
        if not self.use_graph:
            self._fwd_bwd()
            return
        if self.graph is None:
            before = ops.LAUNCHES["count"]
            self._fwd_bwd()                      # eager warm-up: loads the kernels outside the capture
            self.launches_per_step = ops.LAUNCHES["count"] - before + 1   # + Adam
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            # thread-local capture mode: other threads of the process (NCCL's watchdog, a pinned-memory loader) may call into the CUDA
            # runtime while the step is being captured; in the default global mode such a call invalidates a long capture
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self._fwd_bwd()
            ops.LAUNCHES["count"] -= self.launches_per_step - 1    # the capture pass launched nothing
            self.graph = g
            self._plans[self.B].update(graph=g, launches_per_step=self.launches_per_step)
        self.graph.replay()
        ops.LAUNCHES["count"] += self.launches_per_step - 1

    @_on_trainer_device
    def apply_gradients(self) -> None:
        allreduce_flat_(self.grad, self.group)
        self.step_count += 1
        if self.optimizer == "adam":
            ops.adam_step_flat_(self.flat, self.grad, self.exp_avg, self.exp_avg_sq, self.step_count, self.lr, self.betas,
                                self.eps, 1.0, self.l1, self.l2)
        else:      # exp_avg doubles as the momentum buffer, exp_avg_sq as the squared-gradient statistic
            ops.optimizer_step_flat_(self.optimizer, self.flat, self.grad, self.exp_avg, self.exp_avg_sq, self.lr, 1.0, self.l1, self.l2)

    @_on_trainer_device
    def step_async(self, x: torch.Tensor) -> None:
        self.load_batch(x)
        self.compute_gradients()
        self.stats_host.copy_(self.stats, non_blocking=True)
        self.apply_gradients()

    def loss_from_stats(self, stats) -> float:
        """train.py:376-384: batch loss = loss value + l1_lambda * sum|p| + l2_lambda * sum p^2 (this rank's shard).

        Raises ``RuntimeError`` if the EMD solver stopped at its augmentation cap for a jet of the batch (``stats[5] > 0``): that
        jet's EMD and gradient are not optimal.  The row is read after the step, so the parameter update of that step has already
        been applied.  The cap leaves a margin of about 8x over the augmentation counts seen in practice (DESIGN.md section 8)."""
        if float(stats[5]) > 0:
            raise RuntimeError(f"EMD loss: the transport solver did not converge for {int(float(stats[5]))} jet(s) of the batch "
                               "(the update of this step has already been applied)")
        v = float(stats[2])
        if self.l1 > 0:
            v += self.l1 * float(stats[3])
        if self.l2 > 0:
            v += self.l2 * float(stats[4])
        return v

    @_on_trainer_device
    def step(self, x: torch.Tensor) -> float:
        """One optimisation step; returns this rank's batch loss (a device->host read, like train.py:77)."""
        self.step_async(x)
        torch.cuda.current_stream().synchronize()
        return self.loss_from_stats(self.stats_host)

    @_on_trainer_device
    def run_epoch(self, loader, is_train: bool = True, collect: bool = True):
        """The batch loop of reference utils/train.py:51-120 (``train`` / ``validate``) without its per-batch host
        synchronisations: the reference reads ``batch_loss.cpu().item()`` (:77) and copies target / latent / reconstruction to
        the host (:99-101) after every batch; here the per-batch loss terms stay in a device log, the outputs leave through
        asynchronous copies into pinned host memory, and the stream is synchronised ONCE at the end of the epoch.

        ``loader`` yields (B, N, F) batches (host, ideally pinned, or device) of exactly ``batch_size`` jets (use
        ``drop_last=True``; the kernels run on fixed shapes) -- or, for a trainer built with ``partial_batches=True``, a last
        batch of fewer jets, as a ``DataLoader`` without ``drop_last`` yields it (a short batch anywhere else raises
        ``ValueError``).  ``is_train=False`` is the validation pass: forward and loss only, parameters untouched.  Returns
        ``(epoch_avg_loss, recons_data, target_data, latent_data)`` like the reference: the mean of the batch losses over the
        batches (train.py:108) and, with ``collect``, the concatenated host tensors of every jet the loader yielded (else
        ``None``).  The host tensors are views of pinned epoch buffers the trainer keeps, one set for training passes and
        one for validation passes (the reference's train_loop calls train() then validate() and uses both results afterwards,
        utils/train.py:196-236): they stay valid until the next ``run_epoch`` call of the SAME kind (clone them to keep several
        epochs)."""
        st = torch.cuda.current_stream()
        try:
            nb = len(loader)
        except TypeError:
            loader = list(loader)
            nb = len(loader)
        if nb == 0:
            raise ValueError("run_epoch: the loader yielded no batch")
        # epoch-sized pinned host buffers (allocated once and kept: pinning memory synchronises the device) and device log
        caches = self.__dict__.setdefault("_epoch_buffers", {})      # one set per pass kind: train()'s outputs survive validate()
        cache = caches.get(bool(is_train))
        full = self._plans[self.batch_size]
        if cache is None or cache["nb"] < nb or (collect and cache["recon"] is None):
            pin = lambda shape: torch.empty((nb,) + tuple(shape), dtype=torch.float32).pin_memory()
            cache = {"nb": nb, "log": torch.zeros((nb, self.stats.numel()), device=self.dev, dtype=torch.float32),
                     "recon": pin(full["recon"].shape) if collect else None, "latent": pin(full["latent"].shape) if collect else None,
                     "target": pin(full["x"].shape) if collect else None}
            caches[bool(is_train)] = cache
        i = jets = 0
        for x in loader:
            if i >= nb:
                raise ValueError("run_epoch: the loader yielded more batches than len(loader)")
            if x.numel() != full["x"].numel() and not (self.partial_batches and i == nb - 1):
                raise ValueError(f"run_epoch: batch of {tuple(x.shape)} does not match the trainer's fixed "
                                 f"{tuple(full['x'].shape)} (" + ("only the last batch may be short)" if self.partial_batches else
                                                                  "drop the last, ragged batch)"))
            self.load_batch(x)
            if is_train:
                self.compute_gradients()
            else:
                self._fwd(st.cuda_stream)
                self._loss(st.cuda_stream)
            cache["log"][i].copy_(self.stats, non_blocking=True)      # device -> device, stream ordered
            if collect:      # a short last batch fills the first B rows of its slot
                cache["recon"][i, :self.B].copy_(self.recon, non_blocking=True)
                cache["latent"][i, :self.B].copy_(self.latent, non_blocking=True)
                cache["target"][i, :self.B].copy_(self.x, non_blocking=True)
            if is_train:
                self.apply_gradients()
            i += 1
            jets += self.B
        log = cache["log"][:i].cpu()                                  # the epoch's one synchronising read
        st.synchronize()
        avg = sum(self.loss_from_stats(row) for row in log) / i
        if not collect:
            return avg, None, None, None
        flat = lambda t: t[:i].reshape((-1,) + tuple(t.shape[2:]))[:jets]     # views of the epoch buffers (see the docstring)
        return avg, flat(cache["recon"]), flat(cache["target"]), flat(cache["latent"])

    def flat_gradient(self) -> torch.Tensor:
        return self.grad

    def named_gradients(self):
        return OrderedDict((name, self.grad[off:off + int(np.prod(shape))].view(shape))
                           for name, (off, shape) in self.layout.items())
