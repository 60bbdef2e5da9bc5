"""Renderer — host-side mirror of ``src/Renderer/Renderer.{h,cpp,cu}``: orchestrates one ray batch
through sampler -> field (no-grad early-stop pass) -> compaction -> field -> shader -> composite.

``Renderer.Render`` returns the reference's ``RenderResult`` (Renderer.h:18-27) and is connected by
ONE autograd node to the four leaves the trainer optimises (``feat_pool_``, the two ``mlp_.params_``,
``app_emb_`` — ExpRunner.cpp:54,129-136); its backward is a fixed sequence of C-ABI kernels
(composite bwd -> shader MLP bwd -> field MLP bwd -> hash scatter) instead of ~60 autograd nodes.
Host syncs per call: 2 (sample total, survivor total) against the reference's >= 11 ``.item()`` calls.
"""
import os
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib, ops
from ._lib import call, stream
from .field import field_backward, field_forward, field_forward_from_features
from .rng import burn_mlp_output, burn_rand
from .sampler import TRAIN, VALIDATE, LazySampleResult, SampleResultFlex

N_EDGE_PTS = 8192
# The tcgen05 MLP backward rebuilds the hidden activations from the 64 B input row instead of reading 128 / 256 B per sample the
# forward saved (f2b_mlp_bwd2 with hidden0 == NULL): bit-identical dL/dinput, no hidden_save traffic.  F2B_MLP_RECOMPUTE=0 saves.
MLP_RECOMPUTE = os.environ.get("F2B_MLP_RECOMPUTE", "1") == "1"


@dataclass
class RenderResult:
    """``struct RenderResult`` (src/Renderer/Renderer.h:18-27)."""
    colors: torch.Tensor
    first_oct_dis: torch.Tensor
    disparity: torch.Tensor
    edge_feats: Optional[torch.Tensor]
    depth: torch.Tensor
    weights: Optional[torch.Tensor]
    idx_start_end: Optional[torch.Tensor]


class ForwardRenderResult:
    """``RenderResult`` of the fused forward-only path (``f2b_render_fwd_fused``): the per-ray fields are plain tensors; the two
    per-sample fields the reference also returns — ``weights [P']`` and ``idx_start_end [R,2]`` (Renderer.h:24-25) — are packed
    out of the kernel's slot-layout weights on first access (one scan, one 4-byte host read, one gather).  Nothing on the
    evaluation path (ExpRunner::RenderWholeImage, ExpRunner.cpp:257-293) reads them."""
    edge_feats = None

    def __init__(self, colors, first_oct_dis, disparity, depth, kept_counts, w_slots, slot, owner, stamp, total_all):
        self.colors, self.first_oct_dis, self.disparity, self.depth = colors, first_oct_dis, disparity, depth
        self.kept_counts = kept_counts
        self._w_slots, self._slot, self._owner, self._stamp, self._packed = w_slots, slot, owner, stamp, None
        self._total_all = total_all                               # device [2]: samples / octree hits of the whole batch (march)

    def _pack(self):
        if self._packed is None:
            if self._owner._fwd_stamp.get(self._stamp[0]) != self._stamp[1]:
                raise RuntimeError("RenderResult.weights: a later Render re-used this result's slot-layout weights")
            n_rays, dev = self.kept_counts.shape[0], self.kept_counts.device
            bounds, total = ops.count_scan(self.kept_counts, n_rays)
            n_kept, n_all = torch.cat([total, self._total_all[:1]]).tolist()
            if n_all <= 0:                                        # the reference's empty-batch result leaves both undefined
                self._packed = (None, None)                       # (Renderer.cpp:83-97)
                return self._packed
            w = torch.empty((int(n_kept),), dtype=torch.float32, device=dev)
            if n_kept > 0:
                call("f2b_gather_kept_weights", self._w_slots, bounds, n_rays, int(self._slot), w, stream())
            self._packed = (w, bounds)
        return self._packed

    @property
    def weights(self):
        return self._pack()[0]

    @property
    def idx_start_end(self):
        return self._pack()[1]


class Renderer:
    def __init__(self, global_data_pool, pts_sampler, scene_field, shader, n_images, use_app_emb=False,
                 bg_color="rand_noise", device="cuda"):
        self.global_data_pool_ = global_data_pool
        self.pts_sampler_, self.scene_field_, self.shader_ = pts_sampler, scene_field, shader
        self.use_app_emb_ = bool(use_app_emb)
        self.app_emb_ = (torch.randn((n_images, 16), dtype=torch.float32, device=device) * .1).requires_grad_(True)
        if bg_color not in ("white", "black", "rand_noise"):
            bg_color = "rand_noise"
        self.bg_color_type_ = bg_color
        self.sample_result_ = None

    # ------------------------------------------------------------------------------------------
    def _bg(self, n_rays, dev):
        gdp = self.global_data_pool_
        if self.bg_color_type_ == "white":
            return torch.ones((n_rays, 3), dtype=torch.float32, device=dev)
        if self.bg_color_type_ == "rand_noise":
            if gdp.mode_ == TRAIN:
                return torch.rand((n_rays, 3), dtype=torch.float32, device=dev)
            return torch.ones((n_rays, 3), dtype=torch.float32, device=dev) * .5
        return torch.zeros((n_rays, 3), dtype=torch.float32, device=dev)

    def Render(self, rays_o, rays_d, bounds, emb_idx=None):
        """Renderer::Render (Renderer.cpp:52-213)."""
        gdp = self.global_data_pool_
        field, shader, sampler = self.scene_field_, self.shader_, self.pts_sampler_
        n_rays, dev = rays_o.shape[0], rays_o.device
        train = gdp.mode_ == TRAIN
        if not train and self._fused_forward_ok(n_rays):
            return self.render_forward(rays_o, rays_d)
        if self._fused_launch_ok(n_rays):
            return self._render_fused_launches(rays_o, rays_d, emb_idx)
        # ---- the same pipeline, one C-ABI call per kernel (per-kernel tracing, the CUDA-core MLP twin, ray / backward chunking)
        # ---- phase 1: march -> early-stop field pass -> survivors, in the march's slot layout (no host sync) ----
        pf = sampler.take_prefetched(rays_o, rays_d) if n_rays > 0 else None
        if pf is not None:                                           # marched during the previous backward (prefetch_next)
            slots = pf["slots"]
            gen = torch.cuda.default_generators[dev.index if dev.index is not None else torch.cuda.current_device()]
            gen.set_offset(gen.get_offset() + pf["noise_inc"])       # the noise draw happened ahead of time (same numbers)
            torch.cuda.current_stream(dev).wait_event(pf["done"])
        else:
            slots = sampler.begin_march(rays_o, rays_d)              # draws the ray noise (RNG order: noise, bg, ...)
        self.sample_result_ = LazySampleResult(slots)                # the reference-layout view, built only on access
        bg = self._bg(n_rays, dev)
        if n_rays <= 0:
            z = torch.zeros
            return RenderResult(bg, z((0, 1), device=dev), z((0,), device=dev), None, z((0,), device=dev), None, None)
        S = slots.slot
        with torch.no_grad():
            table16 = field.table_f16()
            fparams16 = field.mlp_.params_f16()
            # the encoded features of ALL samples are kept: survivors re-use them in the gradient pass instead of
            # gathering the table a second time (identical values: same points, same table)
            logit_s = self._buf("logit", (n_rays * S,), torch.float32, dev)
            feat_s = self._buf("feat", (n_rays * S, 32), torch.float16, dev)
            weights0 = self._buf("w0", (n_rays * S,), torch.float32, dev)
            alphas0 = self._buf("a0", (n_rays * S,), torch.float32, dev)
            keep = self._buf("keep", (n_rays * S,), torch.uint8, dev)
            kept_counts = self._buf("kept", (n_rays,), torch.int32, dev)
            main = torch.cuda.current_stream(dev)
            chunks = self._ray_chunks(n_rays)
            lanes = [main] + [self._side_stream(dev, i) for i in range(1, len(chunks))]
            ready = torch.cuda.Event()
            ready.record(main)                                       # inputs / table / noise are ready here
            for (r0, r1), st in zip(chunks, lanes):                  # ray chunks on their own streams: chunk k's field
                if st is not main:                                   # pass (memory latency) overlaps chunk k+1's march (issue)
                    st.wait_event(ready)
                with torch.cuda.stream(st):
                    if pf is None:
                        sampler.march_rays(slots, r0, r1)
                    ops.field_fwd_slots(table16, field.prim_pool_, field.bias_pool_, field.n_volumes_, field.local_size_,
                                        fparams16, slots.s_pts[r0 * S:r1 * S], slots.s_anchors[r0 * S:r1 * S],
                                        slots.counts[r0:r1], r1 - r0, S, logit_s[r0 * S:r1 * S], feat_s[r0 * S:r1 * S])
                    ops.early_stop_rays(logit_s, 1, slots.s_dt, slots.slot_bounds[r0:r1], weights0, alphas0, keep,
                                        kept_counts[r0:r1])
            for st in lanes[1:]:
                main.wait_stream(st)
            new_bounds, total = ops.count_scan(kept_counts, n_rays)
            cut_rays = self._bwd_cut_rays(n_rays)                    # interior ray boundaries of the backward's chunks
            head = [total] + ([new_bounds[cut_rays, 0]] if cut_rays is not None else [])
            n_head = 1 + (0 if cut_rays is None else cut_rays.numel())
            vals = torch.cat(head + [t.reshape(-1) for t in slots.totals]).tolist()      # THE host sync of the step
            n_kept = int(vals[0])
            n_all, n_all_oct = int(sum(vals[n_head::2])), int(sum(vals[n_head + 1::2]))
            rcut = [0] + ([] if cut_rays is None else self._cut_list) + [n_rays]
            scut = [0] + [int(v) for v in vals[1:n_head]] + [n_kept]
            self._bwd_cuts_ = [(rcut[i], rcut[i + 1], scut[i], scut[i + 1]) for i in range(len(rcut) - 1)]
            sampler.note_totals(n_rays, n_all_oct)
            slots.noted = True
            self.n_sampled_pts_, self.n_kept_pts_ = n_all, n_kept     # host-side counts of this call (no extra sync)
            if train:
                gdp.sampled_pts_per_ray_ = gdp.sampled_pts_per_ray_ * .9 + (n_all / n_rays) * .1
            if n_all <= 0:
                if train:
                    gdp.meaningful_sampled_pts_per_ray_ *= .9
                z = torch.zeros
                return RenderResult(bg, z((n_rays, 1), device=dev), z((n_rays,), device=dev), None,
                                    torch.full((n_rays,), 512., device=dev), None, None)
            burn_mlp_output(n_all, dev)                   # RNG parity: the reference's MLP output is a torch::rand (rng.py)
            side = None
            if train:
                # octree occupancy votes only feed the NEXT iteration's march: run them beside the gradient pass
                side = self._side_stream(dev, 1)
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    sampler.update_oct_nodes_raw(slots.slot_bounds, slots.s_anchors, weights0, alphas0)
                gdp.meaningful_sampled_pts_per_ray_ = gdp.meaningful_sampled_pts_per_ray_ * .9 + (n_kept / n_rays) * .1
            n_edge = 2 * N_EDGE_PTS if train else 0
            feat_q = torch.empty((n_kept + n_edge, 32), dtype=torch.float16, device=dev)
            f32 = lambda *sh: torch.empty(sh, dtype=torch.float32, device=dev)
            pts, dirs, dt, t = f32(n_kept, 3), f32(n_kept, 3), f32(n_kept), f32(n_kept)
            anchors = torch.empty((n_kept, 3), dtype=torch.int32, device=dev)
            ops.compact_slots(keep, slots.slot_bounds, new_bounds, slots.rays_d, slots.s_pts, slots.s_dt, slots.s_t,
                              slots.s_anchors, feat_s, (pts, dirs, dt, t, anchors), feat_q)
            es = SampleResultFlex(pts, dirs, dt, t, anchors, new_bounds, slots.first_oct_dis.clone())
            if train:                                                                 # TV-loss edge points
                edge_pts, edge_anchors = sampler.GetEdgeSamples(N_EDGE_PTS)
                e_pts, e_anc = edge_pts.reshape(N_EDGE_PTS * 2, 3), edge_anchors.reshape(N_EDGE_PTS * 2)
                e_pts, e_anc = e_pts.contiguous(), e_anc.contiguous()
                feat_q[n_kept:] = ops.hash_fwd(table16, field.prim_pool_, field.bias_pool_, field.n_volumes_, field.local_size_,
                                               e_pts, e_anc, 1)
                segments = [(pts, anchors, 3, 0, n_kept), (e_pts, e_anc, 1, n_kept, n_edge)]
            else:
                segments = [(pts, anchors, 3, 0, n_kept)]
            burn_mlp_output(n_kept + n_edge, dev)         # second AnchoredQuery (Renderer.cpp:165/172) ...
            burn_mlp_output(n_kept, dev)                  # ... and the shader MLP (SHShader.cpp:27)
            pt_emb_idx = ray_emb_idx = None
            if train and self.use_app_emb_:
                ray_emb_idx = emb_idx.to(torch.int32).contiguous()
                pt_emb_idx = ops.scatter_idx(n_kept, new_bounds, ray_emb_idx)

        grad_on = torch.is_grad_enabled() and train
        args = (self, es, segments, None, pt_emb_idx, ray_emb_idx, bg, feat_q, n_kept, grad_on)
        colors, disparity, depth, weights, edge_feats = _RenderFunction.apply(
            field.feat_pool_, field.mlp_.params_, shader.mlp_.params_, self.app_emb_, *args)
        if not train:
            edge_feats = None
        if side is not None:
            torch.cuda.current_stream(dev).wait_stream(side)      # joined before weights0 / alphas0 can be recycled
        return RenderResult(colors, es.first_oct_dis, disparity, edge_feats, depth, weights, new_bounds)

    # ------------------------------------------------------------------------------------------
    def _fused_launch_ok(self, n_rays):
        """One foreign call per phase (f2b_render_phase1 / _phase2_fwd / _bwd, csrc/render.cu) instead of one per kernel: the
        default.  The per-kernel path stays for per-kernel tracing (bench.py's breakdown), the CUDA-core MLP twin and the
        experimental ray / backward chunking."""
        if n_rays <= 0 or _lib.TRACE is not None or os.environ.get("F2B_FUSED_LAUNCH", "1") != "1":
            return False
        if _lib.lib.f2b_get_mlp_impl() != 1 or self.scene_field_.mlp_.n_hidden_matmuls != 0 or self.shader_.mlp_.n_hidden_matmuls != 1:
            return False
        return len(self._ray_chunks(n_rays)) == 1 and self._bwd_cut_rays(n_rays) is None

    def _render_fused_launches(self, rays_o, rays_d, emb_idx):
        """Renderer::Render (Renderer.cpp:52-213): identical kernels, order, streams and RNG draws as the per-kernel path below,
        issued through the three launch sequences of csrc/render.cu."""
        gdp = self.global_data_pool_
        field, shader, sampler = self.scene_field_, self.shader_, self.pts_sampler_
        n_rays, dev = rays_o.shape[0], rays_o.device
        train = gdp.mode_ == TRAIN
        main = torch.cuda.current_stream(dev)
        grad_on = torch.is_grad_enabled() and train                  # as the CALLER has it (everything up to the node is grad-free)
        pf = sampler.take_prefetched(rays_o, rays_d)
        if pf is not None:                                           # marched during the previous backward (prefetch_next)
            slots = pf["slots"]
            gen = torch.cuda.default_generators[dev.index if dev.index is not None else torch.cuda.current_device()]
            gen.set_offset(gen.get_offset() + pf["noise_inc"])       # the noise draw happened ahead of time (same numbers)
            main.wait_event(pf["done"])
        else:
            slots = sampler.begin_march(rays_o, rays_d)              # draws the ray noise (RNG order: noise, bg, ...)
        self.sample_result_ = LazySampleResult(slots)
        bg = self._bg(n_rays, dev)
        S = slots.slot
        with torch.no_grad():
            table16 = field.table_f16()
            i32 = lambda *sh: torch.empty(sh, dtype=torch.int32, device=dev)
            f16 = lambda *sh: torch.empty(sh, dtype=torch.float16, device=dev)
            f32 = lambda *sh: torch.empty(sh, dtype=torch.float32, device=dev)
            fparams16, sparams16 = f16(field.mlp_.params_.numel()), f16(shader.mlp_.params_.numel())
            logit_s = self._buf("logit", (n_rays * S,), torch.float32, dev)
            feat_s = self._buf("feat", (n_rays * S, 32), torch.float16, dev)
            weights0 = self._buf("w0", (n_rays * S,), torch.float32, dev)
            alphas0 = self._buf("a0", (n_rays * S,), torch.float32, dev)
            keep = self._buf("keep", (n_rays * S,), torch.uint8, dev)
            kept_counts = self._buf("kept", (n_rays,), torch.int32, dev)
            new_bounds, heads = i32(n_rays, 2), i32(3)                # heads = [n_kept, n_all, n_all_oct]
            ra = _lib.RenderArgs()
            ra.set(tree_nodes=sampler.tree_nodes_gpu_, n_nodes=sampler.n_nodes, trans=sampler.pers_trans_gpu_,
                   n_trans=sampler.pers_trans_gpu_.numel() // 544, edge_pool=sampler.edge_pool_gpu_ if sampler.n_edges else None,
                   near_t=float(sampler.global_near_), far_t=1e8, sample_l=float(sampler.sample_l_),
                   scale_by_dis=int(sampler.scale_by_dis_), max_hits=int(sampler.max_oct_intersect_per_ray_),
                   count_all_hits=int(bool(sampler.exact_oct_stat_)),
                   table16=table16, prim=field.prim_pool_, bias=field.bias_pool_, n_volumes=int(field.n_volumes_),
                   local_size=int(field.local_size_), field_params=field.mlp_.params_.detach(), n_field_params=fparams16.numel(),
                   shader_params=shader.mlp_.params_.detach(), n_shader_params=sparams16.numel(), fparams16=fparams16,
                   sparams16=sparams16, n_rays=n_rays, rays_o=slots.rays_o, rays_d=slots.rays_d, noise=slots.noise, bg=bg,
                   skip_march=int(pf is not None), s_pts=slots.s_pts, s_dt=slots.s_dt, s_t=slots.s_t, s_anchors=slots.s_anchors,
                   counts=slots.counts, chunk_bounds=slots.chunk_bounds, slot_bounds=slots.slot_bounds,
                   first_oct_dis=slots.first_oct_dis, totals=heads[1:], logit_s=logit_s, feat_s=feat_s, w0=weights0, a0=alphas0,
                   keep=keep, kept_counts=kept_counts, new_bounds=new_bounds, total_kept=heads, stream=stream())
            if pf is not None:
                heads[1:].copy_(slots.totals[0])                      # the prefetched march's own totals
            call("f2b_render_phase1", ra)
            if pf is not None:
                _lib.LAUNCHES -= 3                                    # march (2 kernels) + slot bounds ran with the prefetch
            n_pairs = N_EDGE_PTS if train else 0
            n_edge = 2 * n_pairs
            side = votes_done = None

            def launch_votes():
                # octree occupancy votes only feed the NEXT march: on the side stream, device-ordered behind phase 1 (no host value)
                nonlocal side, votes_done
                side = self._side_stream(dev, 1)
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    sampler.update_oct_nodes_raw(slots.slot_bounds, slots.s_anchors, weights0, alphas0)
                votes_done = torch.cuda.Event()
                votes_done.record(side)                               # (the next batch's march may follow on the same stream)

            def phase2_buffers(rows):
                """Buffers of the second half for up to ``rows`` surviving samples + the TV-loss edge draws (the reference's RNG
                order: after the early-stop query's output draw, before the second query's)."""
                T = dict(pts=f32(rows, 3), dirs=f32(rows, 3), dt=f32(rows), t=f32(rows), anchors=i32(rows, 3),
                         feat_q=f16(rows + n_edge, 32), logit=f32(rows), mlp_in=f16(rows, 32), raw=f16(rows, 16),
                         rgb=f32(rows, 3), edge32=f32(n_edge, 16), colors=f32(n_rays, 3), disparity=f32(n_rays), depth=f32(n_rays),
                         weights=f32(rows))
                if grad_on and not MLP_RECOMPUTE:
                    T.update(f_hidden=f16(1, rows + n_edge, 64), s_hidden=f16(2, rows, 64))
                if train:                                             # TV-loss edge points: the reference's draws
                    if sampler.n_edges <= 0:
                        raise RuntimeError("GetEdgeSamples: empty edge pool (needs >= 2 face-adjacent valid leaves)")
                    T.update(edge_idx=torch.randint(0, sampler.n_edges, (n_pairs,), dtype=torch.int32, device=dev),
                             edge_coord=torch.rand((n_pairs, 2), dtype=torch.float32, device=dev) * 2. - 1.,
                             e_pts=f32(n_edge, 3), e_anc=i32(n_edge))
                if train and self.use_app_emb_:
                    T.update(ray_emb_idx=emb_idx.to(torch.int32).contiguous(), pt_emb_idx=i32(rows))
                return T

            # A prefetched march brought its sample total to the host long ago (pinned copy behind the march): everything that
            # needs only that total — the early-stop query's RNG draw, the votes, the edge draws, the phase-2 buffers (sized for
            # all marched samples, an upper bound of the survivors) — is issued NOW, while the GPU runs phase 1, instead of in
            # the gap behind the sync.
            pre_all = None
            if pf is not None and pf.get("host_totals") is not None:
                pf["done"].synchronize()                  # the march (and the pinned copy behind it) finished during the last backward
                pre_all = int(pf["host_totals"][0])
            T = None
            if pre_all is not None and pre_all > 0 and os.environ.get("F2B_PRESYNC_HOST", "1") == "1":
                burn_mlp_output(pre_all, dev)             # RNG parity: the reference's MLP output is a torch::rand (rng.py)
                if train:
                    launch_votes()
                T = phase2_buffers(pre_all)
            n_kept, n_all, n_all_oct = heads.tolist()                 # THE host sync of the step
            self._bwd_cuts_ = None
            sampler.note_totals(n_rays, n_all_oct)
            slots.noted = True
            slots.totals = [heads[1:]]
            self.n_sampled_pts_, self.n_kept_pts_ = n_all, n_kept
            if train:
                gdp.sampled_pts_per_ray_ = gdp.sampled_pts_per_ray_ * .9 + (n_all / n_rays) * .1
            if n_all <= 0:
                if train:
                    gdp.meaningful_sampled_pts_per_ray_ *= .9
                z = torch.zeros
                return RenderResult(bg, z((n_rays, 1), device=dev), z((n_rays,), device=dev), None,
                                    torch.full((n_rays,), 512., device=dev), None, None)
            if T is None:
                burn_mlp_output(n_all, dev)               # RNG parity: the reference's MLP output is a torch::rand (rng.py)
                if train:
                    launch_votes()
                T = phase2_buffers(n_kept)
            elif pre_all != n_all:
                raise RuntimeError(f"Renderer.Render: prefetched march total {pre_all} != {n_all}")
            T["weights"] = T["weights"][:n_kept]          # the one per-sample tensor handed out (RenderResult.weights)
            if train:
                gdp.meaningful_sampled_pts_per_ray_ = gdp.meaningful_sampled_pts_per_ray_ * .9 + (n_kept / n_rays) * .1
            burn_mlp_output(n_kept + n_edge, dev)         # second AnchoredQuery (Renderer.cpp:165/172) ...
            burn_mlp_output(n_kept, dev)                  # ... and the shader MLP (SHShader.cpp:27)
            if train and self.use_app_emb_:
                ra.set(app_emb=self.app_emb_.detach(), n_emb=self.app_emb_.shape[0])
            ra.set(n_kept=n_kept, n_edge_pairs=n_pairs, **T)
            keepalive = (slots, table16, fparams16, sparams16, new_bounds, heads, bg, T)
        colors, disparity, depth, weights, edge_feats = _FusedRenderFunction.apply(
            field.feat_pool_, field.mlp_.params_, shader.mlp_.params_, self.app_emb_, self, ra, keepalive, grad_on)
        if train and getattr(self, "next_rays_", None) is not None:
            # Software-pipelined march of the NEXT batch (set_next_rays): launched as soon as phase 2 is enqueued, behind the
            # occupancy votes on the side stream, into the other march scratch set — it runs under this batch's phase 2 / loss /
            # backward.  Its noise is drawn at the Philox position the next Render will find: behind the coming backward's
            # GradientScaling draws (rng.py).
            pending = [n_kept * 3, n_kept] if (gdp.gradient_scaling_progress_ < 1. and n_kept > 0) else []
            nxt, self.next_rays_ = self.next_rays_, None
            sampler.prefetch_march(nxt[0], nxt[1], side, pending)
        if side is not None:
            main.wait_event(votes_done)                           # votes joined before weights0 / alphas0 can be recycled
        return RenderResult(colors, slots.first_oct_dis.clone(), disparity, edge_feats if train else None, depth, weights, new_bounds)

    def _fused_forward_ok(self, n_rays):
        """VALIDATE mode takes no gradient, no occupancy votes and no TV-loss edge points: march + ONE kernel
        (f2b_render_fwd_fused).  F2B_FUSED_FORWARD=0 (or per-kernel tracing / the CUDA-core MLP twin) keeps the operator pipeline."""
        if n_rays <= 0 or _lib.TRACE is not None or os.environ.get("F2B_FUSED_FORWARD", "1") != "1":
            return False
        return (_lib.lib.f2b_get_mlp_impl() == 1 and self.scene_field_.mlp_.n_hidden_matmuls == 0
                and self.shader_.mlp_.n_hidden_matmuls == 1)

    def render_forward(self, rays_o, rays_d, out=None, lane=0):
        """Renderer::Render (Renderer.cpp:52-213) for a batch that takes no gradient (VALIDATE mode): the march, then hash encode
        -> field MLP -> early stop -> SH + shader MLP -> composite in ONE kernel that walks each ray front to back and stops at
        the first opaque sample (csrc/fused_fwd.cu).  No host sync, no per-sample tensor in HBM; values bit-identical to the
        operator pipeline.  ``out`` = (colors [R,3], disparity [R], depth [R]) views to write into (whole-image rendering writes
        its image buffers directly); ``lane`` > 0 uses that extra scratch set so two chunks can be in flight on two streams.
        Not reproduced: the reference's torch::rand draws for the MLP outputs (rng.py) — their sizes would need the host sync."""
        field, shader, sampler = self.scene_field_, self.shader_, self.pts_sampler_
        n_rays, dev = rays_o.shape[0], rays_o.device
        slots = sampler.begin_march(rays_o, rays_d, lane=lane)
        sampler.march_rays(slots, 0, n_rays)
        if lane == 0:
            self.sample_result_ = LazySampleResult(slots)
        bg = self._bg(n_rays, dev)
        S = slots.slot
        with torch.no_grad():
            table16 = field.table_f16()
            fparams16, sparams16 = field.mlp_.params_f16(), shader.mlp_.params_f16()
            f32 = lambda *sh: torch.empty(sh, dtype=torch.float32, device=dev)
            colors, disparity, depth = out if out is not None else (f32(n_rays, 3), f32(n_rays), f32(n_rays))
            kept = torch.empty((n_rays,), dtype=torch.int32, device=dev)
            ticket = torch.empty((1,), dtype=torch.int32, device=dev)
            w_slots = self._buf(f"w_fwd{lane}", (n_rays * S,), torch.float32, dev)
            stamps = self.__dict__.setdefault("_fwd_stamp", {})
            stamps[lane] = stamps.get(lane, 0) + 1
            call("f2b_render_fwd_fused", table16, field.prim_pool_, field.bias_pool_, int(field.n_volumes_), int(field.local_size_),
                 fparams16, sparams16, slots.s_pts, slots.s_dt, slots.s_t, slots.s_anchors, slots.counts, slots.rays_d, bg, n_rays, S,
                 slots.totals[0], ticket, colors, disparity, depth, kept, w_slots, stream())
        res = ForwardRenderResult(colors, slots.first_oct_dis, disparity, depth, kept, w_slots, S, self, (lane, stamps[lane]),
                                  slots.totals[0])
        res._keep = (slots, table16, fparams16, sparams16, bg, ticket)          # alive until the result dies (stream-ordered reuse)
        return res

    def set_next_rays(self, rays_o, rays_d):
        """Hand over the ray tensors of the NEXT ``Render`` before calling this one (TRAIN mode): ``Render`` then launches their
        march itself, right behind this batch's occupancy votes (earliest point at which the octree is final for it), instead of
        the caller doing so afterwards through :meth:`prefetch_next`.  Results are bit-identical either way."""
        self.next_rays_ = (rays_o, rays_d)

    def prefetch_next(self, rays_o, rays_d):
        """Software-pipeline the NEXT batch's ray march behind this batch's loss + backward.  Call right after ``Render``
        returned (TRAIN mode), with the ray tensors the next ``Render`` will be given: the march reads no trainable state, only
        the octree as this iteration's votes leave it, so it is queued on the votes' side stream and its ~1 ms of per-ray
        dependent latency disappears from the critical path.  Results are bit-identical to an unpipelined run (same noise
        numbers, same octree state); a next ``Render`` with different rays simply ignores the prefetch."""
        gdp = self.global_data_pool_
        dev = rays_o.device
        pf = getattr(self.pts_sampler_, "_prefetched", None)
        if pf is not None and pf["key"][:3] == (rays_o.data_ptr(), rays_d.data_ptr(), rays_o.shape[0]):
            return                                                  # Render already launched it (set_next_rays)
        self.next_rays_ = None
        pending = ()
        if gdp.gradient_scaling_progress_ < 1. and getattr(self, "n_kept_pts_", 0) > 0:      # the coming backward's burns
            pending = (self.n_kept_pts_ * 3, self.n_kept_pts_)
        self.pts_sampler_.prefetch_march(rays_o, rays_d, self._side_stream(dev, 1), pending)

    def _table_grad_buffer(self, shape, dev):
        """The fp32 table gradient handed to autograd.  Only floats [0, 17*S) of it are ever written (the half-overlapping level
        layout leaves the other 15/32 of the pool without gradient for ever), so the STORAGE is kept across steps and only that
        live prefix is zero-filled per backward (34 of 64 MB at log2 19, 272 of 512 MB at log2 22) — as long as no tensor on last
        step's gradient is alive any more (storage use count): a trainer that keeps ``.grad`` (zero_grad(set_to_none=False),
        gradient accumulation) gets a fresh, fully zeroed tensor instead.  Every backward returns a NEW tensor object on the
        storage, so autograd still takes it as ``.grad`` without a copy."""
        self._table_grad_tail_zero = False
        n = 1
        for d in shape:
            n *= int(d)
        st = getattr(self, "_d_table_storage_", None)
        try:
            if st is not None and st.nbytes() == 4 * n and st.device == torch.device(dev) and torch._C._storage_Use_Count(st._cdata) == 1:
                self._table_grad_tail_zero = True              # the dead tail has been zero since the storage was created
                return torch.empty(0, dtype=torch.float32, device=dev).set_(st, 0, tuple(shape))
            buf = torch.zeros(tuple(shape), dtype=torch.float32, device=dev)
            self._d_table_storage_ = buf.untyped_storage()
            self._table_grad_tail_zero = True                  # just zeroed as a whole
            return buf
        except (AttributeError, RuntimeError):                 # private use-count API missing: a plain per-step allocation, zeroed as a whole
            self._d_table_storage_ = None
            return torch.empty(tuple(shape), dtype=torch.float32, device=dev)

    def _side_stream(self, dev, i=1):
        pool = self.__dict__.setdefault("_streams_", {})
        key = (torch.device(dev).index, i)
        if key not in pool:
            pool[key] = torch.cuda.Stream(device=dev)
        return pool[key]

    def _buf(self, name, shape, dtype, dev):
        """Persistent slot-layout work buffers (grown on demand; no allocator traffic in steady state)."""
        pool = self.__dict__.setdefault("_bufs_", {})
        n = 1
        for d in shape:
            n *= d
        t = pool.get(name)
        if t is None or t.numel() < n or t.dtype != dtype or t.device != torch.device(dev):
            t = pool[name] = torch.empty((max(n, 1),), dtype=dtype, device=dev)
        return t[:n].view(*shape)

    def _bwd_cut_rays(self, n_rays):
        """Device index tensor of the interior ray boundaries of the backward chunks (F2B_BWD_CHUNKS / ``bwd_chunks_``)."""
        if not hasattr(self, "bwd_chunks_"):
            self.bwd_chunks_ = int(os.environ.get("F2B_BWD_CHUNKS", "1"))
        k = max(1, min(int(self.bwd_chunks_), 16, (n_rays + 255) // 256))
        if k <= 1:
            self._cut_list = []
            return None
        key = (n_rays, k)
        if getattr(self, "_cut_key", None) != key:
            step = -(-n_rays // k)
            self._cut_list = [r for r in range(step, n_rays, step)]
            self._cut_dev = torch.tensor(self._cut_list, dtype=torch.int64, device=self.app_emb_.device) if self._cut_list else None
            self._cut_key = key
        return self._cut_dev

    def _ray_chunks(self, n_rays):
        """Ray ranges marched on separate streams (F2B_RAY_CHUNKS / ``ray_chunks_``; 1 = single stream)."""
        if not hasattr(self, "ray_chunks_"):
            self.ray_chunks_ = int(os.environ.get("F2B_RAY_CHUNKS", "1"))
        k = max(1, min(int(self.ray_chunks_), 4, (n_rays + 255) // 256))
        step = -(-n_rays // k)
        return [(r0, min(r0 + step, n_rays)) for r0 in range(0, n_rays, step)]

    # ------------------------------------------------------------------------------------------
    def States(self):
        out = []
        for p in (self.pts_sampler_, self.scene_field_, self.shader_):
            out += p.States()
        return out + [self.app_emb_.data]

    def LoadStates(self, states, idx=0):
        for p in (self.pts_sampler_, self.scene_field_, self.shader_):
            idx = p.LoadStates(states, idx)
        self.app_emb_.data.copy_(states[idx].to(self.app_emb_.device)); idx += 1
        return idx

    def OptimParamGroups(self):
        lr = self.global_data_pool_.learning_rate_
        groups = self.scene_field_.OptimParamGroups() + self.shader_.OptimParamGroups()
        return groups + [dict(params=[self.app_emb_], lr=lr, betas=(0.9, 0.99), eps=1e-15, weight_decay=1e-6)]

    def Reset(self):
        self.scene_field_.Reset()
        self.shader_.Reset()


class _FusedRenderFunction(torch.autograd.Function):
    """Second half of Renderer::Render (Renderer.cpp:127-208) with its whole backward, each ONE launch sequence of csrc/render.cu.
    ``ra`` (the filled f2b_render block) and the tensors it points to travel in ``keepalive``."""

    @staticmethod
    def forward(ctx, feat_pool, field_params, shader_params, app_emb, renderer, ra, keepalive, grad_on):
        T = keepalive[-1]
        call("f2b_render_phase2_fwd", ra)
        if ra.n_edge_pairs == 0:
            _lib.LAUNCHES -= 3
        ctx.renderer, ctx.ra, ctx.keepalive, ctx.grad_on = renderer, ra, keepalive, grad_on
        ctx.gs_progress = renderer.global_data_pool_.gradient_scaling_progress_
        ctx.table_shape, ctx.emb_shape = feat_pool.shape, app_emb.shape
        return T["colors"], T["disparity"], T["depth"], T["weights"], T["edge32"].reshape(-1, 2, 16)

    @staticmethod
    def backward(ctx, d_colors, d_disp, d_depth, d_weights, d_edge):
        renderer, ra = ctx.renderer, ctx.ra
        if ctx.keepalive is None:
            raise RuntimeError("Renderer.Render backward: the saved activations were released by a previous backward "
                               "(like tiny-cuda-nn's context, TCNNWP.cpp:207, the graph can be traversed once)")
        if not ctx.grad_on:
            raise RuntimeError("Renderer.Render backward: forward ran without grad (VALIDATE mode / no_grad)")
        field, shader = renderer.scene_field_, renderer.shader_
        T = ctx.keepalive[-1]
        dev = T["colors"].device
        n_kept, n_edge, n_rays = ra.n_kept, 2 * ra.n_edge_pairs, ra.n_rays
        main = torch.cuda.current_stream(dev)
        c = lambda g: None if g is None else g.contiguous()
        d_colors = c(d_colors) if d_colors is not None else torch.zeros((n_rays, 3), dtype=torch.float32, device=dev)
        d_disp, d_depth, d_weights = c(d_disp), c(d_depth), c(d_weights)
        d_edge = None if d_edge is None else d_edge.reshape(-1, 16).contiguous()
        if ctx.gs_progress < 1.:                          # GradientScaling::backward draws an unused rand_like (CustomOps.cu:154)
            burn_rand(n_kept * 3, dev)
            burn_rand(n_kept, dev)
        f16 = lambda *sh: torch.empty(sh, dtype=torch.float16, device=dev)
        f32 = lambda *sh: torch.empty(sh, dtype=torch.float32, device=dev)
        emb_on = "ray_emb_idx" in T
        slab_hook = getattr(renderer, "grad_slab_hook_", None)
        f_scale = field.mlp_.loss_scale_
        grad_mul = (1.0 / f_scale) * (getattr(renderer, "grad_premul_", 1.0) if slab_hook is not None else 1.0)
        # dfeat16: the field MLP's fp16 dL/dfeatures, in memory only when the scatter is a separate kernel (level slabs, A/B runs)
        two_kernel = slab_hook is not None or not _lib.FIELD_BWD_SCATTER
        B = dict(d_logit=f32(n_kept), d_raw=f16(n_kept, 16), d_in16=f16(n_kept, 32), d_scene16=f16(n_kept + n_edge, 16),
                 dfeat16=f16(n_kept + n_edge, 32) if two_kernel else None, d_sparams=f32(ra.n_shader_params), d_fparams=f32(ra.n_field_params),
                 d_table=renderer._table_grad_buffer(ctx.table_shape, dev),
                 nonfinite=torch.empty((2,), dtype=torch.int32, device=dev))
        if emb_on:
            B["d_app"] = torch.empty(ctx.emb_shape, dtype=torch.float32, device=dev)
        side = renderer._side_stream(dev, 2)
        ra.set(d_colors=d_colors, d_disparity=d_disp, d_depth=d_depth, d_weights=d_weights, d_edge=d_edge,
               gs_progress=float(ctx.gs_progress), shader_loss_scale=float(shader.mlp_.loss_scale_), field_loss_scale=float(f_scale),
               table_grad_mul=float(grad_mul),
               # floats to zero-fill: the live prefix only when the buffer's dead tail is known to be zero already
               table_numel=min(B["d_table"].numel(), 17 * int(field.local_size_)) if renderer._table_grad_tail_zero else B["d_table"].numel(),
               table_live=min(B["d_table"].numel(), 17 * int(field.local_size_)), scatter_mode=int(slab_hook is not None),
               stream=main.cuda_stream, side_stream=side.cuda_stream, **B)
        call("f2b_render_bwd", ra)
        if slab_hook is not None:                         # data parallel: level slabs top-down, all-reduce of each behind it (dist.py)
            hash_args = (field.prim_pool_, field.bias_pool_, int(field.n_volumes_), int(field.local_size_))
            jobs = [(T["pts"], T["anchors"], 3, 0, n_kept)] + ([(T["e_pts"], T["e_anc"], 1, n_kept, n_kept + n_edge)] if n_edge else [])
            ev = torch.cuda.Event()
            ev.record(main)
            side.wait_event(ev)
            with torch.cuda.stream(side):
                for lo, nl in slab_groups():
                    for pts_j, anc_j, stride_j, s0, s1 in jobs:
                        if s1 > s0:
                            call("f2b_hash_bwd_levels", *hash_args, pts_j, anc_j, int(stride_j), int(s1 - s0), B["dfeat16"][s0:s1], 1,
                                 float(grad_mul), B["d_table"], lo, nl, stream())
                    slab_hook(B["d_table"], lo, int(field.local_size_))
            main.wait_stream(side)
            renderer.grad_slab_finish_()
        call("f2b_render_grad_finalize", ra)
        bad = B["nonfinite"] != 0                          # [shader, field], device-side, no sync here
        prev = getattr(renderer, "nonfinite_flag_", None)
        renderer.nonfinite_flag_ = bad if prev is None else (prev | bad)
        ctx.keepalive = None                              # saved activations die with the backward, not with `res`
        return B["d_table"], B["d_fparams"], B["d_sparams"], B.get("d_app"), None, None, None, None


class _RenderFunction(torch.autograd.Function):
    """Second half of Renderer::Render (Renderer.cpp:152-208) with its whole backward."""

    @staticmethod
    def forward(ctx, feat_pool, field_params, shader_params, app_emb, renderer, es, q_pts, q_anchors, pt_emb_idx,
                ray_emb_idx, bg, feat16, n_kept, grad_on):
        field, shader = renderer.scene_field_, renderer.shader_
        fparams16 = ops.cast_f32_to_f16(field_params)
        sparams16 = ops.cast_f32_to_f16(shader_params)
        dev = bg.device
        n_q = feat16.shape[0]
        emb = app_emb if pt_emb_idx is not None else None
        if _lib.lib.f2b_get_mlp_impl() == 1 and field.mlp_.n_hidden_matmuls == 0 and shader.mlp_.n_hidden_matmuls == 1:
            # fused epilogues (tcgen05 kernels): field MLP -> [logit | shader-MLP input row], shader MLP -> [raw | rgb];
            # the fp32 scene_feat of the ray samples is never materialised (edge points still need all 16 channels)
            save = grad_on and not MLP_RECOMPUTE
            f_hidden = torch.empty((1, n_q, 64), dtype=torch.float16, device=dev) if save else None
            logit = torch.empty((n_kept,), dtype=torch.float32, device=dev)
            mlp_in = torch.empty((n_kept, 32), dtype=torch.float16, device=dev)
            call("f2b_field_shade_fwd", feat16, fparams16, es.dirs, emb, pt_emb_idx, n_kept, logit, mlp_in, f_hidden, stream())
            if n_q > n_kept:
                edge32 = torch.empty((n_q - n_kept, 16), dtype=torch.float32, device=dev)
                call("f2b_mlp_fwd_f32", feat16[n_kept:], fparams16, 0, n_q - n_kept, edge32, None,
                     f_hidden[0, n_kept:] if save else None, stream())
            else:
                edge32 = torch.empty((0, 16), dtype=torch.float32, device=dev)
            s_hidden = torch.empty((2, n_kept, 64), dtype=torch.float16, device=dev) if save else None
            raw = torch.empty((n_kept, 16), dtype=torch.float16, device=dev)
            rgb = torch.empty((n_kept, 3), dtype=torch.float32, device=dev)
            call("f2b_shader_mlp_rgb_fwd", mlp_in, sparams16, n_kept, raw, rgb, s_hidden, stream())
            logit_stride = 1
        else:
            scene_feat, f_hidden = field_forward_from_features(field, fparams16, feat16, save=grad_on)
            mlp_in = ops.shader_prep(scene_feat[:n_kept], es.dirs, emb, pt_emb_idx) if n_kept > 0 else \
                torch.empty((0, 32), dtype=torch.float16, device=bg.device)
            raw, s_hidden = ops.mlp_fwd(mlp_in, sparams16, shader.mlp_.n_hidden_matmuls, save_hidden=grad_on)
            rgb = ops.shader_act(raw)
            logit, logit_stride, edge32 = scene_feat, 16, scene_feat[n_kept:]
        colors, disparity, depth, weights = ops.composite_fwd(logit, logit_stride, rgb, es.dt, es.t, es.pts_idx_bounds, bg)
        scene_feat = (logit, logit_stride)
        edge_feats = edge32.reshape(-1, 2, 16)
        ctx.renderer, ctx.es, ctx.n_kept = renderer, es, n_kept
        ctx.cuts = renderer._bwd_cuts_ if getattr(renderer, "_bwd_cuts_", None) else [(0, es.pts_idx_bounds.shape[0], 0, n_kept)]
        ctx.pack = (fparams16, sparams16, q_pts, q_anchors, ray_emb_idx, bg, scene_feat, feat16, f_hidden, mlp_in, raw,
                    s_hidden, rgb)
        ctx.gs_progress = renderer.global_data_pool_.gradient_scaling_progress_
        ctx.grad_on = grad_on
        return colors, disparity, depth, weights, edge_feats

    @staticmethod
    def backward(ctx, d_colors, d_disp, d_depth, d_weights, d_edge):
        renderer, es, n_kept = ctx.renderer, ctx.es, ctx.n_kept
        field, shader, gdp = renderer.scene_field_, renderer.shader_, renderer.global_data_pool_
        if ctx.pack is None:
            raise RuntimeError("Renderer.Render backward: the saved activations were released by a previous backward "
                               "(like tiny-cuda-nn's context, TCNNWP.cpp:207, the graph can be traversed once)")
        (fparams16, sparams16, q_pts, q_anchors, ray_emb_idx, bg, scene_feat, feat16, f_hidden, mlp_in, raw, s_hidden,
         rgb) = ctx.pack
        if not ctx.grad_on:
            raise RuntimeError("Renderer.Render backward: forward ran without grad (VALIDATE mode / no_grad)")
        segments = q_pts
        n_q, dev = feat16.shape[0], feat16.device
        n_rays = es.pts_idx_bounds.shape[0]
        zeros = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)
        d_colors = d_colors.contiguous() if d_colors is not None else zeros(n_rays, 3)
        d_disp = d_disp.contiguous() if d_disp is not None else None
        d_depth = d_depth.contiguous() if d_depth is not None else None
        d_weights = d_weights.contiguous() if d_weights is not None else None
        if ctx.gs_progress < 1.:                          # GradientScaling::backward draws an unused rand_like (CustomOps.cu:154)
            burn_rand(n_kept * 3, dev)
            burn_rand(n_kept, dev)
        # ---- backward, optionally in ray chunks (bwd_chunks_ / F2B_BWD_CHUNKS): the dense chain (composite -> sigmoid ->
        # shader MLP -> input assembly -> field MLP; HBM streaming) of chunk k+1 on the main stream, the hash scatter of
        # chunk k (L2 reductions) on a side stream.  Measured on B200 (r01): co-running them is SLOWER (6.05 ms at 1
        # chunk, 6.5 / 6.8 / 7.7 ms at 2 / 4 / 8: the scatter's 260 k small blocks crowd out the persistent tcgen05 CTAs),
        # so the default is one chunk; the scatter still runs on the side stream behind an event.
        s_scale, f_scale = shader.mlp_.loss_scale_, field.mlp_.loss_scale_
        nh_s, nh_f = shader.mlp_.n_hidden_matmuls, field.mlp_.n_hidden_matmuls
        f16 = lambda *sh: torch.empty(sh, dtype=torch.float16, device=dev)
        d_logit = torch.empty((n_kept,), dtype=torch.float32, device=dev)
        d_raw, d_in16, d_scene16 = f16(n_kept, 16), f16(n_kept, 32), f16(n_q, 16)
        d_sparams, d_fparams = zeros(sparams16.numel()), zeros(fparams16.numel())
        d_table = torch.zeros_like(field.feat_pool_)
        d_app = torch.zeros_like(renderer.app_emb_) if ray_emb_idx is not None else None
        if n_q > n_kept:
            if d_edge is not None:
                d_scene16[n_kept:] = (d_edge.reshape(-1, 16) * f_scale).to(torch.float16)
            else:
                d_scene16[n_kept:].zero_()
        main = torch.cuda.current_stream(dev)
        side = renderer._side_stream(dev, 2)
        bounds = es.pts_idx_bounds
        hash_args = (field.prim_pool_, field.bias_pool_, int(field.n_volumes_), int(field.local_size_))

        # Data parallel: ``grad_slab_hook_`` (f2nerf_b200.dist.install_grad_overlap) wants the table gradient slab by slab, so that
        # the NCCL all-reduce of a finished slab runs while the lower level groups still scatter.  Level l only writes floats
        # [l*S, (l+2)*S): the scatter then runs per level group, top-down, after the dense chain; the hook is called after each.
        slab_hook = getattr(renderer, "grad_slab_hook_", None)
        grad_mul = (1.0 / f_scale) * (getattr(renderer, "grad_premul_", 1.0) if slab_hook is not None else 1.0)
        jobs = []

        def scatter(pts, anc, stride, s0, s1):            # on the side stream, behind everything queued on main so far
            if slab_hook is not None:
                jobs.append((pts, anc, stride, s0, s1))
                return
            ev = torch.cuda.Event()
            ev.record(main)
            side.wait_event(ev)
            with torch.cuda.stream(side):
                ops.hash_bwd(*hash_args, pts, anc, stride, dfeat16[s0:s1], grad_mul, d_table)

        # one chunk, no slab hook: the field-MLP backward and the scatter of both segments as ONE kernel (f2b_field_bwd_scatter)
        fused = (_lib.FIELD_BWD_SCATTER and slab_hook is None and len(ctx.cuts) == 1 and nh_f == 0
                 and _lib.lib.f2b_get_mlp_impl() == 1)
        dfeat16 = None if fused else f16(n_q, 32)
        for r0, r1, s0, s1 in ctx.cuts:
            if s1 <= s0:
                continue
            nr, ns = r1 - r0, s1 - s0
            # composite backward with the colour activation's backward applied on the way out (fp16 d_raw directly)
            call("f2b_composite_act_bwd", scene_feat[0], int(scene_feat[1]), rgb, es.dt, es.t, bounds[r0:r1], bg[r0:r1], nr,
                 d_colors[r0:r1], None if d_disp is None else d_disp[r0:r1], None if d_depth is None else d_depth[r0:r1],
                 d_weights, float(ctx.gs_progress), raw, float(s_scale), d_logit, 1, d_raw, stream())
            call("f2b_mlp_bwd2", d_raw[s0:s1], mlp_in[s0:s1], None if s_hidden is None else s_hidden[0, s0:s1],
                 s_hidden[1, s0:s1] if (nh_s and s_hidden is not None) else None, sparams16, int(nh_s), ns, d_in16[s0:s1], d_sparams,
                 stream())
            ops.shader_prep_bwd_f16(d_in16, d_logit, bounds[r0:r1], None if ray_emb_idx is None else ray_emb_idx[r0:r1],
                                    1.0 / s_scale, f_scale, d_scene16, d_app)
            if fused:
                continue
            call("f2b_mlp_bwd2", d_scene16[s0:s1], feat16[s0:s1], None if f_hidden is None else f_hidden[0, s0:s1],
                 f_hidden[1, s0:s1] if (nh_f and f_hidden is not None) else None, fparams16, int(nh_f), ns, dfeat16[s0:s1], d_fparams,
                 stream())
            scatter(segments[0][0][s0:s1], segments[0][1][s0:s1], segments[0][2], s0, s1)
        if fused:
            edge = segments[1] if len(segments) > 1 else (None, None, 1, n_kept, 0)
            ops.field_bwd_scatter(d_scene16, feat16, fparams16, segments[0][0], segments[0][1], edge[0], edge[1], *hash_args,
                                  grad_mul, d_fparams, d_table)
        for pts_e, anc_e, stride_e, first, rows in ([] if fused else segments[1:]):   # TV-loss edge points: field MLP + scatter only
            if rows > 0:
                call("f2b_mlp_bwd2", d_scene16[first:first + rows], feat16[first:first + rows],
                     None if f_hidden is None else f_hidden[0, first:first + rows],
                     f_hidden[1, first:first + rows] if (nh_f and f_hidden is not None) else None, fparams16, int(nh_f), rows,
                     dfeat16[first:first + rows], d_fparams, stream())
                scatter(pts_e, anc_e, stride_e, first, first + rows)
        if slab_hook is not None:
            ev = torch.cuda.Event()
            ev.record(main)
            side.wait_event(ev)
            with torch.cuda.stream(side):
                for lo, nl in slab_groups():
                    for pts_j, anc_j, stride_j, s0, s1 in jobs:
                        call("f2b_hash_bwd_levels", *hash_args, pts_j, anc_j, int(stride_j), int(s1 - s0), dfeat16[s0:s1], 1, float(grad_mul),
                             d_table, lo, nl, stream())
                    slab_hook(d_table, lo, int(field.local_size_))          # issued on the side stream: NCCL orders itself behind it
        main.wait_stream(side)
        if slab_hook is not None:
            renderer.grad_slab_finish_()                  # the main stream waits for the slab all-reduces: d_table leaves here averaged
        d_sparams = d_sparams / s_scale
        d_fparams = d_fparams / f_scale
        # NaN back-off of TCNNWPFunction::backward (TCNNWP.cpp:231-240): the reference tests dL/dparams AND dL/dinput of
        # each MLP.  The shader MLP's input gradient reaches d_app (and the field MLP's dL/dout), the field MLP's input
        # gradient reaches every table-gradient entry its samples touch, so those stand in for the fp16 tensors
        # themselves (a non-finite fp16 element cannot disappear on the way: w * inf / NaN stays non-finite).
        live = min(d_table.shape[0], (17 * int(field.local_size_)) // 2)
        ok_s = torch.isfinite(d_sparams).all()
        if d_app is not None:
            ok_s = ok_s & torch.isfinite(d_app).all()
        ok_f = torch.isfinite(d_fparams).all() & torch.isfinite(d_table[:live]).all()
        bad = torch.stack([~ok_s, ~ok_f])                          # [shader, field], device-side, no sync here
        prev = getattr(renderer, "nonfinite_flag_", None)
        renderer.nonfinite_flag_ = bad if prev is None else (prev | bad)      # OR: a second backward must not erase a hit
        ctx.pack = None                               # saved activations (~1 GB at 4 M samples) die with the backward, not with `res`
        return d_table, d_fparams, d_sparams, d_app, None, None, None, None, None, None, None, None, None, None


def slab_groups():
    """Level groups (first level, count) of the data-parallel scatter, top-down; the table-gradient slab above a group's lower
    boundary is all-reduced behind it while the next group scatters (dist.install_grad_overlap).  F2B_DP_SLABS = 4 (default:
    12-15 | 8-11 | 4-7 | 0-3), 2 (8-15 | 0-7: fewer launch tails, a larger exposed last slab) or 1."""
    n = int(os.environ.get("F2B_DP_SLABS", "4"))
    return {4: ((12, 4), (8, 4), (4, 4), (0, 4)), 2: ((8, 8), (0, 8)), 1: ((0, 16),)}.get(n, ((12, 4), (8, 4), (4, 4), (0, 4)))


def check_backward_nan(renderer):
    """Host read of the device-side NaN flags accumulated by the backward passes since the last call (one sync);
    applies the reference's loss-scale halving to the MLP(s) that produced the non-finite values and sets
    ``global_data_pool_.backward_nan_`` — the flag ExpRunner.cpp:131-134 reads right after ``loss.backward()``.
    A trainer MUST call this between ``backward()`` and ``optimizer.step()`` (FusedAdam.step(renderer=...) does)."""
    flag = getattr(renderer, "nonfinite_flag_", None)
    renderer.nonfinite_flag_ = None
    if flag is None:
        return False
    hit = flag.reshape(-1).tolist()
    if len(hit) == 1:
        hit = [hit[0], hit[0]]
    for m, h in ((renderer.shader_.mlp_, hit[0]), (renderer.scene_field_.mlp_, hit[1])):
        if h:
            m.loss_scale_ = max(m.loss_scale_ / 2.0, 1.0)
    if any(hit):
        renderer.global_data_pool_.backward_nan_ = True
        return True
    return False
