"""One training step of the reconstruction loop, in the reference's order of operations
(Trainer.train_one_epoch2, reconstruction/nerf/utils.py:1116-1175 and train_step :532-679):

    encoder.reset_cahce(); encoder.get_planes()                # OUTSIDE autocast => fp32 IDWT, graph kept (:1138-1140)
    every `update_extra_interval` steps: model.update_extra_state() under autocast                      (:1144-1146)
    with autocast(fp16): render -> MSE(pred, gt).mean(-1).mean() + wavelet L1 regulariser               (:1158-1160)
    encoder.reset_cahce(); scaler.scale(loss).backward()                                                (:1161-1166)
    scaler.step(optimizer); scaler.update()                                                             (:1170-1173)

The Trainer class of the reference (datasets, checkpoints, logging, LR schedule) stays the host's business; this
module is the thin per-step driver the benchmark and the tests use, plus the ray-sharded multi-GPU variant.
"""
import os
from types import SimpleNamespace

import torch

from . import _lib, parallel


def default_opt(**over):
    opt = dict(fp16=True, max_steps=1024, dt_gamma=0.0, background_color=0.0, wavelet_regularization=0.2,
               update_extra_interval=16, lr=1e-2, fused_regulariser=True)
    opt.update(over)
    return SimpleNamespace(**opt)


def wavelet_regulariser(encoder, lam, fused=True):
    """nerf/utils.py:640-655 (unweighted branch): lam * sum_l mean|yh_l| * numel_l/numel_all / n_levels.
    fused=True takes the value from the |yh| sums of this step's plane reconstruction and applies the gradient inside
    the IDWT backward kernels; fused=False is the reference's literal torch expression (three extra passes per level)."""
    feats = encoder.get_wavelet_features()
    if lam <= 0 or len(feats) == 0:
        return None
    if fused:
        return encoder.wavelet_l1(lam)
    total = sum(v.numel() for v in feats)
    reg = sum(v.abs().mean() * (v.numel() / total) for v in feats) / len(feats)
    return lam * reg


class TrainStep:
    def __init__(self, model, opt=None, optimizer=None, world_size=1, sparse_allreduce=True, check_sparse=False,
                 transport=torch.bfloat16, exchange="auto"):
        if world_size > 1:   # before any distributed call
            _lib.alert_nondeterministic("a multi-GPU TrainStep (world_size > 1)")
        self.model = model
        self.opt = opt or default_opt()
        self.optimizer = optimizer
        self.scaler = torch.amp.GradScaler("cuda", enabled=self.opt.fp16)
        self.global_step = 0
        self.world_size = world_size
        self.criterion = torch.nn.MSELoss(reduction='none')
        # N > 1: the plane gradient is exchanged between the render backward and the IDWT backward, dirty tiles only
        self.reducer = parallel.PlaneGradReducer(model, world_size, check=check_sparse, transport=transport) if (world_size > 1 and sparse_allreduce) else None
        # exchange: "peer" = this package's own all-reduce kernels over NVLink peer / NVSwitch multicast memory, in place and in fp32
        # (parallel.PeerGradExchange); "nccl" = pack -> NCCL all-reduce of the bf16 dirty tiles -> unpack; "auto" = peer where the
        # symmetric-memory rendezvous and its known-answer self-test succeed on every rank, else nccl (with a note on rank 0)
        self.exch = None
        self.exchange_note = "nccl (pack / NCCL all-reduce of bf16 dirty tiles / unpack)" if self.reducer is not None else None
        if self.reducer is not None and exchange in ("auto", "peer") and not check_sparse and next(model.parameters()).is_cuda:
            try:
                self.reducer.refresh()
                self._reducer_gen = getattr(model, "bitfield_generation", 0)
                self.exch = parallel.PeerGradExchange(model, world_size, self.reducer)
                model.encoder.external_grad_buffer = self.exch.g_planes
                model.encoder.scatter_plane_hook = self._exchange_plane_async
                # high priority: when SM slots free up the (small, persistent) exchange kernels are placed before the next wave of
                # the scatter's CTAs, so the exchange of plane p really runs under the scatter of plane p + 1
                self._comm = torch.cuda.Stream(priority=-1)
                self.exchange_note = f"peer memory, {self.exch.mode} (own kernels: in place, fp32, one CUDA graph per step)"
            except Exception as ex:  # noqa: BLE001
                if exchange == "peer":
                    raise
                self.exchange_note += f" [peer exchange unavailable: {type(ex).__name__}: {str(ex)[:120]}]"
        # eager-mode option: per-plane exchange on a side stream overlapped with the per-plane IDWT backward.  Measured on
        # 8 x B200 it does not beat the sequential exchange (NCCL and the IDWT kernels contend for SMs / HBM), so it is off.
        self.pipelined_tail = False
        # steady-state steps reconstruct the planes on a second stream, concurrently with the ray marching + cell sort
        self.prefetch_planes = True
        self._side = None
        # steady-state steps reconstruct / differentiate the planes only where the occupancy grid puts samples
        # (idwt_plan.py); steps that refresh the density grid query the field everywhere and stay dense
        self.sparse_idwt = True
        self._plan = None
        self._plan_gen = None     # model.bitfield_generation the plan / the dirty-tile list were built from
        self._reducer_gen = getattr(self, "_reducer_gen", None)
        self.plan_on_any_device = False   # test hook: the CPU suite runs the work-list step over the host build of the kernels
        self._graphs = None

    # ---- the three segments of a step ---------------------------------------------------------------------------------
    def _render_loss(self, rays_o, rays_d, images):
        model, opt = self.model, self.opt
        with torch.autocast("cuda", dtype=torch.float16, enabled=opt.fp16):
            bg = torch.zeros_like(images) + opt.background_color
            out = model.render(rays_o.unsqueeze(0), rays_d.unsqueeze(0), staged=False, bg_color=bg, perturb=True,
                               force_all_rays=False, dt_gamma=opt.dt_gamma, max_steps=opt.max_steps)
            pred = out['image'].view(-1, 3)
            return self.criterion(pred, images).mean(-1).mean()

    def forward_backward(self, rays_o, rays_d, images, update_grid=None):
        """rays_o/rays_d/images: [N,3] device tensors (this rank's shard). Returns the detached loss tensor.
        Rays that require grad (e.g. drawn from poses.CameraPoses through RayFeeder.select_batch(poses=...)) pass their
        gradient on: the backward of this step also fills the .grad of whatever the rays were computed from."""
        if self.world_size > 1 and (rays_o.requires_grad or rays_d.requires_grad):
            raise RuntimeError("TrainStep: rays that require grad (camera pose refinement) are supported on one GPU only: "
                               "the multi-GPU step does not reduce the pose gradient across ranks")
        model, opt = self.model, self.opt
        enc = model.encoder
        model.train()
        enc.reset_cahce()
        self._planes_exchanged = 0
        do_update = (self.global_step % opt.update_extra_interval == 0) if update_grid is None else update_grid
        enc.idwt_plan = None
        use_plan = (self.sparse_idwt and not do_update and (rays_o.is_cuda or self.plan_on_any_device) and model.cuda_ray
                    and self._plan_supported())
        # anything derived from the density bitfield must follow it (update_extra_state here or in the caller's own loop,
        # load_state_dict of a checkpoint, ...): rebuild when the model's bitfield generation moved on
        gen = getattr(model, "bitfield_generation", 0)
        if self.reducer is not None and self.reducer.tile_ids is not None and self._reducer_gen != gen:
            self.reducer.refresh()
            self._reducer_gen = gen
        if use_plan:
            if self._plan is None or self._plan_gen != gen:
                self.refresh_plan()
            enc.idwt_plan = self._plan
        prefetch = self.prefetch_planes and not do_update and rays_o.is_cuda
        # work-list steps drive the IDWT backward themselves (two parts, see SplitIdwtBackward); its gradient-independent
        # part goes to the prefetch stream right away and overlaps the render
        will_split = use_plan and not self.pipelined_tail and all(p.grad is None for p in enc.parameters())
        # (debug mode of the exchange sums the whole gradient buffer, so it needs all of it defined)
        partial_zero = will_split and not (self.reducer is not None and self.reducer.check)
        if use_plan:
            self._plan.defer_clean_abs = will_split
        if prefetch:
            if self._side is None:
                self._side = torch.cuda.Stream()
            planes = enc.prefetch_planes(self._side, partial_zero=partial_zero)
        else:
            planes = enc.get_planes()
        enc.idwt_plan = None   # the cached planes of this step are built; anything reconstructed later is dense again
        abs_sums = enc._last_abs_sums
        self._split = None
        if will_split:
            self._split = self._make_split(enc, opt)
            # completed by the clean part (the forward skipped those blocks); deterministic mode: complete already (torch sums)
            self._split.abs_sums = None if _lib.deterministic() else abs_sums
            # its gradient-independent ("clean") part runs on the side stream: single GPU / NCCL exchange -> right away, under the
            # render; peer exchange -> later, under the exchange (link-bound, few SMs busy), see below
            # (measured at 8 x B200: 6.24 ms with the clean part under the exchange vs 6.33 ms with it under the render;
            #  TNL_OVERLAP_CLEAN=0 selects the latter)
            self._overlap_clean = (self.exch is not None and prefetch and self._split.reg_ready
                                   and os.environ.get("TNL_OVERLAP_CLEAN", "1") == "1")
            if prefetch and self._split.reg_ready and not self._overlap_clean:
                with torch.cuda.stream(self._side):
                    self._split.run_clean()
        if do_update:
            with torch.autocast("cuda", dtype=torch.float16, enabled=opt.fp16):
                model.update_extra_state()
            if self.world_size > 1:
                # every rank refreshed its grid from its own RNG stream (jittered cell samples): the replicas must agree on the
                # occupancy, or the dirty-tile lists (and the all-reduce buffer sizes) derived from it diverge -> rank 0's wins
                parallel.sync_occupancy(model)
            if self.reducer is not None:
                self.reducer.refresh()
                self._reducer_gen = model.bitfield_generation
            if self._plan is not None:
                self.refresh_plan()
        capturing = torch.cuda.is_current_stream_capturing()
        if self.reducer is None and self._split is None:
            # single GPU, dense planes: one backward through render + IDWT
            with torch.autocast("cuda", dtype=torch.float16, enabled=opt.fp16):
                loss = self._render_loss(rays_o, rays_d, images)
                enc._join_prefetch()
                reg = wavelet_regulariser(enc, opt.wavelet_regularization, getattr(opt, "fused_regulariser", True))
                if reg is not None:
                    loss = loss + reg
                enc.reset_cahce()
                self.scaler.scale(loss).backward()
            if self.world_size > 1 and not capturing:
                parallel.allreduce_gradients(model, self.world_size)
        else:
            # cut the graph at the planes: render backward -> plane gradient; (N > 1: exchange its dirty tiles;) IDWT backward
            leaf = planes.detach().requires_grad_(True)
            enc.last_used_planes = leaf
            lam = opt.wavelet_regularization
            have_reg = lam > 0 and len(enc.get_wavelet_features()) > 0
            with torch.autocast("cuda", dtype=torch.float16, enabled=opt.fp16):
                loss = self._render_loss(rays_o, rays_d, images)
                enc._join_prefetch()
                # the autograd fall-back needs the regulariser as a graph node now; the split backward applies its gradient
                # itself and completes the |yh| sums in its clean part, so there the value is formed at the end
                reg = wavelet_regulariser(enc, lam, True) if (self._split is None and have_reg) else None
                enc.reset_cahce()
                self.scaler.scale(loss).backward()                    # -> leaf.grad and the MLP gradients of this shard
            self._cut = (planes, leaf, reg)
            if self.reducer is None:
                split = self._split
                self._idwt_backward()
                if split is not None and have_reg:
                    reg = enc.wavelet_l1(lam, abs_sums)
                self._cut = None
                self._split = None
                if self.world_size > 1 and not capturing:
                    parallel.allreduce_gradients(model, self.world_size)
            else:
                overlap = self._split is not None and getattr(self, "_overlap_clean", False) and not self._split.clean_done
                if overlap:
                    # the scatter is done: the clean part of the IDWT backward (0.6 ms of HBM streaming) shares the machine with the exchange
                    self._side.wait_stream(torch.cuda.current_stream())
                    with torch.cuda.stream(self._side):
                        self._split.run_clean()
                elif self._split is not None and not self._split.clean_done:   # first step of a run (no loss scale yet)
                    self._split.reg_scale = self.scaler._scale if self.scaler.is_enabled() else self._split.reg_scale
                    self._split.run_clean()
                if prefetch and not overlap:   # the early part of the IDWT backward belongs to this segment of the step (graph A)
                    torch.cuda.current_stream().wait_stream(self._side)
                if self._split is not None and have_reg and not overlap:
                    reg = enc.wavelet_l1(lam, abs_sums)
                if not capturing or self.exch is not None:    # (the peer exchange is plain kernels: it is captured with the step)
                    self._exchange_and_finish(join_side=overlap)
                    if overlap and have_reg:
                        reg = enc.wavelet_l1(lam, abs_sums)
            loss = loss.detach() + (reg.detach() if reg is not None else 0.0)
        self.global_step += 1
        return loss.detach()

    def _make_split(self, enc, opt):
        from .triplane_encoder import SplitIdwtBackward
        feats = enc.get_wavelet_features()
        lam = opt.wavelet_regularization
        reg_coef = lam / (sum(v.numel() for v in feats) * len(feats)) if (lam > 0 and len(feats) > 0) else 0.0
        if not self.scaler.is_enabled():
            if getattr(self, "_one", None) is None:
                self._one = torch.ones(1, device=enc.planes_features.device)
            scale_t = self._one
        else:
            scale_t = getattr(self.scaler, "_scale", None)    # created lazily by the first scaler.scale() call
        sp = SplitIdwtBackward(enc, self._plan, scale_t, reg_coef)
        sp.reg_ready = reg_coef == 0.0 or scale_t is not None
        sp.clean_done = False
        return sp

    def _plan_supported(self):
        enc = self.model.encoder
        n0 = enc.planes_features.shape[2]
        return len(enc.planes_features_wavelet_coefs) >= 1 and n0 % 16 == 0 and enc.plane_resolution % 32 == 0

    def refresh_plan(self):
        """(Re)build the IDWT work lists from the current density bitfield; must follow every change of the bitfield."""
        from .idwt_plan import IdwtPlan
        self._plan = IdwtPlan.from_model(self.model, plan=self._plan)
        self._plan_gen = getattr(self.model, "bitfield_generation", 0)
        return self._plan

    def _exchange_plane_async(self, plane):
        """called by the sampling backward right after it has launched the scatter of `plane`: that plane's exchange starts on the
        communication stream while the next plane scatters on the main stream"""
        self._comm.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self._comm):
            self.exch.exchange_plane_(plane)
        self._planes_exchanged += 1

    def _exchange(self):
        if self.exch is not None:
            planes, leaf, reg = self._cut
            if self._planes_exchanged == 3 and leaf.grad is None:
                self.exch.exchange_mlp_()                                   # (small: 54 KB) on the main stream ...
                torch.cuda.current_stream().wait_stream(self._comm)         # ... while the last plane finishes on the other
                return
            if leaf.grad is not None:       # dense step (grid refresh): the scatter went into an ordinary buffer
                self.exch.g_planes.copy_(leaf.grad)
                leaf.grad = None
            self.exch.exchange_()
            return
        self._exchange_finish(self._exchange_start())

    def _plane_grad(self):
        """the plane gradient of this step: leaf.grad, or the persistent symmetric buffer the scatter wrote (peer exchange)"""
        planes, leaf, reg = self._cut
        return leaf.grad if (self.exch is None or leaf.grad is not None) else self.exch.g_planes

    def _exchange_start(self):
        """pack the dirty tiles of the plane gradient and start their all-reduce (asynchronous: NCCL's own stream)."""
        planes, leaf, reg = self._cut
        return self.reducer.start_(leaf.grad)

    def _exchange_finish(self, work):
        planes, leaf, reg = self._cut
        self.reducer.finish_(leaf.grad, work)
        mlp = [p for n, p in self.model.named_parameters() if not n.startswith("encoder.")]
        parallel.allreduce_small(mlp, self.world_size)

    def _idwt_backward(self):
        planes, leaf, reg = self._cut
        sp = self._split
        if sp is not None:
            if not sp.clean_done:     # first step of a run: the loss scale did not exist yet when the step started
                if sp.reg_scale is None and sp.reg_coef != 0.0:
                    sp.reg_scale = self.scaler._scale
                sp.run_clean()
            if self._side is not None and self.reducer is None:   # (N > 1: forward_backward has already joined the stream)
                torch.cuda.current_stream().wait_stream(self._side)
            sp.run_active(self._plane_grad())
            sp.assign()
            return
        if self._side is not None:   # the reconstruction's autograd node runs on the prefetch stream
            self._side.wait_stream(torch.cuda.current_stream())
        if reg is not None:   # identical on every rank: added once, after the exchange
            torch.autograd.backward([planes, self.scaler.scale(reg)], [self._plane_grad(), None])
        else:
            torch.autograd.backward([planes], [self._plane_grad()])

    def _tail_pipelined(self):
        """N > 1: per-plane gradient exchange on a communication stream, overlapped with the IDWT backward of the previous
        plane on the compute stream:   exch(0) | exch(1) || idwt(0) | exch(2) || idwt(1) | idwt(2).
        The regulariser gradient (identical on every rank) is added inside the IDWT backward kernels, after the exchange."""
        from .triplane_encoder import PlanewiseIdwtBackward
        planes, leaf, reg = self._cut
        enc, opt = self.model.encoder, self.opt
        feats = enc.get_wavelet_features()
        lam = opt.wavelet_regularization
        reg_coef = lam / (sum(v.numel() for v in feats) * len(feats)) if (lam > 0 and len(feats) > 0) else 0.0
        scale_t = getattr(self.scaler, "_scale", None) if self.scaler.is_enabled() else None
        if scale_t is None:
            scale_t = torch.ones(1, device=leaf.device)
        bw = PlanewiseIdwtBackward(enc, leaf.grad, scale_t, reg_coef)
        main = torch.cuda.current_stream()
        if getattr(self, "_comm", None) is None:
            self._comm = torch.cuda.Stream()
        comm = self._comm
        comm.wait_stream(main)
        done = []
        mlp = [p for n, p in self.model.named_parameters() if not n.startswith("encoder.")]
        with torch.cuda.stream(comm):
            for p in range(3):
                self.reducer.reduce_plane_(leaf.grad, p)
                ev = torch.cuda.Event()
                ev.record(comm)
                done.append(ev)
            parallel.allreduce_small(mlp, self.world_size)
            ev_small = torch.cuda.Event()
            ev_small.record(comm)
        import os
        if os.environ.get("TNL_TAIL_SEQ"):      # diagnostic: no overlap (exchange everything, then the IDWT backward)
            main.wait_event(done[2])
        for p in range(3):
            main.wait_event(done[p])
            bw.run(p)
        main.wait_event(ev_small)
        bw.assign()

    def _exchange_and_finish(self, join_side=False):
        if self.pipelined_tail:
            self._tail_pipelined()
        else:
            self._exchange()
            if join_side:
                torch.cuda.current_stream().wait_stream(self._side)
            self._idwt_backward()
        self._cut = None   # drop the autograd graph (and the AccumulateGrad nodes it keeps alive) of this step
        self._split = None

    # ---- CUDA-graph mode: a steady-state step is one (N = 1) or two (N > 1, NCCL in between) graph launches ----------
    def capture(self, rays_o, rays_d, images, warmup=3):
        """Capture forward_backward (steady state: mean_count > 0, no density-grid refresh) into CUDA graphs.
        Inputs are copied into static buffers before each replay; parameter gradients live in the graph's memory pool
        and are overwritten by every replay (equivalent to zero_grad(set_to_none=True) + backward).  The step counter
        ring slot is the one current at capture time."""
        if rays_o.requires_grad or rays_d.requires_grad:
            raise RuntimeError("TrainStep.capture: rays that require grad (camera pose refinement) cannot be captured: the "
                               "graph's static inputs are plain buffers; run the step eagerly with forward_backward()")
        assert self.model.mean_count > 0, "capture needs the steady state (mean_count > 0): run a few eager steps first"
        self._static = tuple(t.clone() for t in (rays_o, rays_d, images))
        if self.reducer is not None:
            self.reducer.refresh()
            self._reducer_gen = getattr(self.model, "bitfield_generation", 0)
        if self.sparse_idwt and self._plan_supported():
            self.refresh_plan()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self.model.zero_grad(set_to_none=True)
                self.forward_backward(*self._static, update_grid=False)
        torch.cuda.current_stream().wait_stream(side)
        self.model.zero_grad(set_to_none=True)
        self._cut = None
        # both captures run on the same side stream: the autograd nodes of the IDWT (created while capturing A) execute
        # on the stream they were recorded on, which must be the stream that is capturing B
        gA = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gA, stream=side):
            self._static_loss = self.forward_backward(*self._static, update_grid=False)
        gB = None
        if self.reducer is not None and self.exch is None:
            gB = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gB, pool=gA.pool(), stream=side):
                self._idwt_backward()
        self._graphs = (gA, gB)
        self._graph_plan_version = self._plan.version if self._plan is not None else None
        # the gradient tensors the captured kernels write into; replay() re-attaches them, so zero_grad(set_to_none=True)
        # between replays (optimizer_step does it) is harmless
        self._graph_grads = [(p, p.grad) for p in self.model.parameters() if p.grad is not None]
        return self

    def replay(self, rays_o, rays_d, images):
        """One captured fwd+bwd on new inputs (device or pinned-host tensors); returns the (static) loss tensor."""
        for dst, src in zip(self._static, (rays_o, rays_d, images)):
            dst.copy_(src, non_blocking=True)
        gA, gB = self._graphs
        gen = getattr(self.model, "bitfield_generation", 0)
        if self._plan is not None and self._plan_gen != gen:
            self.refresh_plan()            # the lists are rewritten in place: the captured graphs stay valid unless they grew
        if self.reducer is not None and self._reducer_gen != gen:
            self.reducer.refresh()
            self._reducer_gen = gen
        if self._plan is not None and self._plan.version != self._graph_plan_version:
            raise RuntimeError("the IDWT work lists were reallocated after capture(): capture the step again")
        gA.replay()
        if gB is not None:
            self._exchange()
            gB.replay()
        elif self.world_size > 1 and self.reducer is None:
            parallel.allreduce_gradients(self.model, self.world_size)
        for p, g in self._graph_grads:
            p.grad = g
        self.global_step += 1
        return self._static_loss

    def replay_from_feeder(self, feeder, batch_idx, batch_size):
        """One captured fwd+bwd whose rays and targets are generated on the device (rays.RayFeeder, SURVEY.md 8f-2): the
        feeder kernel writes straight into the graph's static input buffers -- no host batch, no H2D copy."""
        ids = feeder.batch_ids(batch_idx, batch_size)
        if ids.numel() != self._static[0].shape[0]:
            raise RuntimeError("replay_from_feeder: the batch does not have the captured number of rays (ragged last batch: "
                               "run it through step()/forward_backward instead)")
        feeder.select_batch(batch_idx, batch_size, out=self._static)
        return self.replay(*self._static)

    def optimizer_step(self):
        if self.optimizer is None:
            return
        from .optim import FusedAdam
        if isinstance(self.optimizer, FusedAdam):
            self.optimizer.step(scaler=self.scaler)        # unscale + non-finite check + Adam + loss-scale update, fused
        else:
            self.scaler.step(self.optimizer)
            self.scaler.update()
        self.optimizer.zero_grad(set_to_none=True)

    def step(self, rays_o, rays_d, images, update_grid=None):
        self.optimizer.zero_grad(set_to_none=True) if self.optimizer is not None else self.model.zero_grad(set_to_none=True)
        loss = self.forward_backward(rays_o, rays_d, images, update_grid)
        self.optimizer_step()
        return loss


def make_optimizer(model, lr=1e-2, fused=False):
    """main_nerf.py:119: Adam(model.get_params(lr), betas=(0.9, 0.99), eps=1e-15).  fused=True: the same update as two
    streaming kernels that also absorb GradScaler.step/update (trinerflet_b200/optim.py)."""
    if fused:
        from .optim import FusedAdam
        return FusedAdam(model.get_params(lr), betas=(0.9, 0.99), eps=1e-15)
    return torch.optim.Adam(model.get_params(lr), betas=(0.9, 0.99), eps=1e-15)
