"""Fused training steps: one forward, the minimal backward, gradient exchange and the optimizer update, all as
launches of libfmri_b200.so kernels on raw device buffers (no autograd graph, no host round trip inside the step).

VaeGanStage1 follows the reference's train/train_vgan_stage1.py:316-432 (all four loss mixes of :359-388) and computes
exactly the three gradients its optimizers consume -- g_enc = d loss_encoder / d encoder, g_dec = d loss_decoder / d decoder,
g_dis = d loss_discriminator / d discriminator at the pre-step weights (SURVEY.md 0-7) -- with ONE discriminator forward
(the reference runs it twice on the same inputs, vae_gan.py:284-285; BN running statistics are updated twice to match)
and no discarded gradient (the reference's three full autograd sweeps execute 2.35x the necessary FLOPs).

WaeGanStage1 follows /root/reference/train/train_wae_stage1.py:259-311.

Data parallelism (SURVEY.md 8e): every rank holds full replicas; each parameter bucket's flat fp32 gradient buffer is
all-reduced (SUM, no averaging: the losses are batch sums) on a side stream as soon as its last gradient kernel has
been issued, overlapping the rest of the backward; BatchNorm statistics stay per rank; the equilibrium gate is decided
on the device from the all-reduced BCE sums so every rank takes the same branch.
"""
from __future__ import annotations

from collections import OrderedDict

import torch

from . import lib as L
from . import nets as NN
from .dp import FlatBucket
from .nets import BF16, F32, E, Z


def _split(full, prefix):
    return OrderedDict((k[len(prefix):], v) for k, v in full.items() if k.startswith(prefix))


class _TrainerBase:
    # Adam's step count lives in a device int32 (advanced by fmri_step_increment, read by fmri_multi_tensor_adam_dev): the step has
    # no host-side scalar that changes from call to call, so it can be captured in a CUDA graph (GraphedStep).
    t_dev = None

    @property
    def t(self):
        return int(self.t_dev.item()) if self.t_dev is not None else 0

    @t.setter
    def t(self, v):
        if self.t_dev is None:
            self.t_dev = torch.zeros(1, dtype=torch.int32, device="cuda")
        self.t_dev.fill_(int(v))

    def _setup(self, params, buffers, nets, n_states, lr, dist_group):
        """Device state of a trainer of `nets` (prefix -> network, in bucket order): one flat bucket per network with its
        reference-named parameters and n_states[prefix] optimizer-state buffers, learning rates `lr`, device copies of the
        BatchNorm buffers, 16 loss-sum / gate slots `sc`, the exchange state and the operand packs."""
        self.nets = nets
        self.buckets = OrderedDict()
        for pre, net in nets.items():
            named = _split(params, pre)
            diff = set(net.param_names()) ^ set(named)
            if diff:
                raise L.FmriError(f"parameter names of {pre} differ from the reference layout: {sorted(diff)}")
            self.buckets[pre] = FlatBucket(pre, OrderedDict((k, named[k].to("cuda", F32)) for k in named), n_states[pre],
                                           "cuda")
        self.S = OrderedDict((k, v.to("cuda").clone()) for k, v in buffers.items())
        self.Ssub = {pre: _split(self.S, pre) for pre in self.buckets}
        self.nbt = {}
        self.sc = Z(16)
        self.lr = lr
        self._ones_buf = None
        self.dist = dist_group
        self.world = 1
        if dist_group is not None:
            import torch.distributed as td

            self.td = td
            self.world = td.get_world_size(group=dist_group)
            self.comm_stream = torch.cuda.Stream()
        self.refresh()

    def refresh(self):
        """Re-derive the bf16 operand packs from the fp32 master weights."""
        for pre, net in self.nets.items():
            net.refresh(self.buckets[pre].P, inplace=True)

    def _ones(self, n):
        """At least n fp32 ones on the device: the upstream gradient of a loss sum."""
        if self._ones_buf is None or self._ones_buf.numel() < n:
            self._ones_buf = torch.ones(n, device="cuda")
        return self._ones_buf

    def _count_bn_updates(self, pre, counts):
        """Add one forward's BatchNorm running-statistics updates (name -> count, names under `pre`) to the pending
        num_batches_tracked increments. Reads self.nbt on every call: GraphedStep swaps it around a capture."""
        for k, v in counts.items():
            self.nbt[pre + k] = self.nbt.get(pre + k, 0) + v

    def _latent_d_phase(self, net, b, z_real, z_fake, scale, sums):
        """Discriminator phase of a latent WaeDiscriminator `net` (bucket `b`): L_fake = -scale sum log(d(z_fake) + 1e-3)
        into sums[0], L_real = -scale sum log(1 - d(z_real) + 1e-3) into sums[1], and their gradient in b.G.
        Returns d(z_real), d(z_fake) and the [2B] loss / score-gradient scratch, which the G-phase reuses."""
        B = z_real.shape[0]
        ones = self._ones(B)
        p_real, cr = net.forward(b.P, z_real)
        p_fake, cf = net.forward(b.P, z_fake)
        l, gp = E(2 * B), E(2 * B)
        L.bce_fwd(p_fake, l[:B], B, True, scale)
        L.bce_fwd(p_real, l[B:], B, False, scale)
        L.vecsum(l[:B], B, 1.0, sums[0:1])
        L.vecsum(l[B:], B, 1.0, sums[1:2])
        L.bce_bwd(p_fake, ones, gp[:B], B, True, scale)
        L.bce_bwd(p_real, ones, gp[B:], B, False, scale)
        net.backward(b.P, cf, gp[:B], b.G, False, True, False)
        net.backward(b.P, cr, gp[B:], b.G, True, True, False)
        return p_real, p_fake, l, gp

    def _allreduce_async(self, tensors):
        """SUM all-reduce on the side stream, ordered after everything issued so far on the compute stream."""
        if self.world == 1:
            return
        cur = torch.cuda.current_stream()
        self.comm_stream.wait_stream(cur)
        NN.side_into(self.comm_stream)   # weight gradients are produced on nets' side stream
        with torch.cuda.stream(self.comm_stream):
            for t in tensors:
                self.td.all_reduce(t, op=self.td.ReduceOp.SUM, group=self.dist)
                t.record_stream(self.comm_stream)
            ev = torch.cuda.Event()
            ev.record(self.comm_stream)
        return ev   # everything reduced so far on the exchange stream (update() may wait for a prefix of the exchanges)

    def _wait_comm(self):
        NN.join_side()
        if self.world > 1:
            torch.cuda.current_stream().wait_stream(self.comm_stream)

    def _flush_nbt(self):
        for name, n in self.nbt.items():
            self.S[name] += n
        self.nbt.clear()

    def end_epoch(self, epoch=None, **kw):
        """Per-epoch schedules of the reference scripts, applied to this trainer's learning rates / gate constants:
        VAE/GAN trainers -> hp.epoch_end_vgan (ExponentialLR 0.98, margin / equilibrium / lambda_mse decay,
        train_vgan_stage1.py:446-457); WAE trainers -> hp.epoch_end_wae (StepLR(30, 0.5), needs `epoch`)."""
        from . import hp as _hp

        if "beta1" in self.hp:
            _hp.epoch_end_wae(self.lr, int(epoch), **kw)
        else:
            _hp.epoch_end_vgan(self.lr, self.hp, **kw)

    def state_dict(self):
        """Checkpoint of the whole trainer (host tensors). `model` holds parameters and BatchNorm buffers under the
        reference's state_dict keys (torch.save(sd["model"]) is a checkpoint the reference's load_state_dict accepts);
        `optimizer` holds every bucket's per-parameter state (RMSprop square_avg, or Adam exp_avg / exp_avg_sq, named like the
        parameters); plus learning rates, hyper-parameters (the decayed margin / equilibrium / lambda_mse) and Adam's step count."""
        self._wait_comm()
        model = OrderedDict((k, v.detach().cpu().clone()) for k, v in self.named_parameters().items())
        model.update((k, v.detach().cpu().clone()) for k, v in self.named_buffers().items())
        opt = OrderedDict()
        for pre, b in self.buckets.items():
            opt[pre] = [OrderedDict((pre + k, b.state_view(i, k).detach().cpu().clone()) for k in b.names)
                        for i in range(len(b.states))]
        return dict(model=model, optimizer=opt, lr=dict(self.lr), hp=dict(self.hp), t=self.t)

    def load_state_dict(self, sd):
        """Resume from state_dict(): copies into the flat device buckets, then re-derives the bf16 operand packs."""
        self._wait_comm()
        for k, v in self.named_parameters().items():
            v.copy_(sd["model"][k])
        self.nbt.clear()
        for k, v in self.S.items():
            v.copy_(sd["model"][k])
        for pre, b in self.buckets.items():
            for i, st in enumerate(sd["optimizer"].get(pre, [])):
                for k in b.names:
                    b.state_view(i, k).copy_(st[pre + k])
        self.lr.update(sd["lr"])
        self.hp.update(sd["hp"])
        if self.t_dev is not None:
            self.t = int(sd["t"])
        self.refresh()

    def named_parameters(self):
        out = OrderedDict()
        for b in self.buckets.values():
            for k, v in b.P.items():
                out[b.prefix + k] = v
        return out

    def named_grads(self):
        NN.join_side()
        out = OrderedDict()
        for b in self.buckets.values():
            for k, v in b.G.items():
                out[b.prefix + k] = v
        return out

    def named_buffers(self):
        self._flush_nbt()
        return self.S


class VaeGanStage1(_TrainerBase):
    """Stage-I VAE/GAN trainer (image -> image): visual Encoder, Decoder, Discriminator, three RMSprop optimizers.

    mode: the loss mix of train_vgan_stage1.py:359-388. 'vae-gan' and 'beta-vae' use the discriminator's feature MSE;
    'dcgan' (:374-380) and 'vae' (:382-387) use the pixel NLE instead and leave bce_p out of loss_discriminator. 'dcgan'
    trains no encoder; 'vae' drops the discriminator term from loss_decoder and sets train_dis = False before the gate.
    gate=False applies the mix's own flags without the gate: 'vae' trains the decoder only, every other mix trains both."""

    MODES = ("vae-gan", "beta-vae", "dcgan", "vae")
    LATENT_DISCRIMINATOR = False

    def __init__(self, params, buffers, cfg, z=128, adt=BF16, hp=None, dist_group=None, gate=True, mode="vae-gan", beta=1.0):
        from .hp import HP_VGAN

        if mode not in self.MODES:
            raise L.FmriError(f"unknown Stage-I loss mix {mode!r}: the fused step implements {', '.join(self.MODES)} "
                              "(train_vgan_stage1.py:359-388)")
        self.mode, self.beta, self._klw = mode, float(beta), 1.0
        self.cfg, self.z, self.adt = cfg, z, adt
        self.hp = dict(HP_VGAN if hp is None else hp)
        self.gate_on = gate
        self.enc = NN.EncoderNet(cfg, z, adt)
        self.dec = NN.DecoderNet(cfg, z, adt)
        self.dis = NN.DiscriminatorNet(cfg, adt)
        nets = OrderedDict((("encoder.", self.enc), ("decoder.", self.dec), ("discriminator.", self.dis)))
        if self.LATENT_DISCRIMINATOR:
            self.ldis = NN.WaeDiscriminatorNet(z, adt)
            nets["latent_discriminator."] = self.ldis
        self._ev_dec = None   # exchange of the loss sums, discriminator and decoder, issued by backward()
        # sc: [0..5] = sum bce_o, bce_p, bce_s, kl, mse, nle ; [8],[9] = gates (train_dis, train_dec)
        self._setup(params, buffers, nets, dict.fromkeys(nets, 1), dict.fromkeys(nets, float(self.hp["lr"])), dist_group)

    def forward_backward(self, x, eps, z_p):
        """x [B,3,H,W] fp32 NCHW, eps / z_p [B,z] fp32, all on the device. Leaves gradients in the buckets' flat_g and the
        loss sums in self.sc. Returns a dict of the forward tensors (device)."""
        st = self.forward(x, eps, z_p)
        self.backward(st)
        return st.out

    def forward(self, x, eps, z_p):
        """Forward + losses (vae_gan.py:276-286, 302-320; train_vgan_stage1.py:369-372). Returns the saved state the backward
        consumes (tests/test_teacher_forced_gpu.py overwrites it with the oracle's activations before calling backward)."""
        B, z = x.shape[0], self.z
        be, bd, bc = self.buckets["encoder."], self.buckets["decoder."], self.buckets["discriminator."]
        Se, Sd, Sc = self.Ssub["encoder."], self.Ssub["decoder."], self.Ssub["discriminator."]
        nbe, nbd, nbc = {}, {}, {}
        sc = self.sc
        ycat, ce = self.enc.forward(be.P, Se, x, True, self._enc_bn_updates, nbe)
        mu, lv = ycat[:, :z], ycat[:, z:]
        zz, kl = E(B, z), E(B)
        L.reparam_kl_fwd(mu, lv, eps, zz, kl, B, z, ld=2 * z)
        x_tilde, cd1 = self.dec.forward(bd.P, Sd, zz, True, 1, nbd)
        x_p, cd2 = self.dec.forward(bd.P, Sd, z_p, True, 1, nbd)
        raw3, p, cc = self.dis.forward(bc.P, Sc, [x, x_tilde, x_p], True, 2, True, nbc)  # REC + GAN passes -> 2 BN updates
        for pre, d in (("encoder.", nbe), ("decoder.", nbd), ("discriminator.", nbc)):
            self._count_bn_updates(pre, d)
        # ------------------------------------------------------------------ losses (vae_gan.py:302-320, stage1 :369-372)
        Fd = raw3[0].numel()
        mse, nle = E(B), E(B)
        L.rowsqdiff_fwd(raw3[:B], raw3[B:2 * B], mse, B, Fd, 0.5)
        L.rowsqdiff_fwd(x, x_tilde, nle, B, x[0].numel(), 0.5)
        bce = E(3 * B)
        L.bce_fwd(p[:B], bce[:B], B, True, 1.0)
        L.bce_fwd(p[B:], bce[B:], 2 * B, False, 1.0)
        L.vecsum(bce[:B], B, 1.0, sc[0:1])
        L.vecsum(bce[B:2 * B], B, 1.0, sc[1:2])
        L.vecsum(bce[2 * B:], B, 1.0, sc[2:3])
        L.vecsum(kl, B, 1.0, sc[3:4])
        L.vecsum(mse, B, 1.0, sc[4:5])
        L.vecsum(nle, B, 1.0, sc[5:6])
        self._allreduce_async([sc[:8]])  # global loss sums: the gate must agree on every rank (SURVEY.md 0-10)
        out = dict(x_tilde=x_tilde, x_p=x_p, disc_layer_nhwc=raw3, disc_class=p, mu=mu, logvar=lv, z=zz, kl=kl, mse=mse,
                   bce=bce, nle=nle)
        return NN.Ctx(B=B, x=x, eps=eps, ce=ce, cd1=cd1, cd2=cd2, cc=cc, raw3=raw3, p=p, mu=mu, lv=lv, out=out)

    def backward(self, st):
        """The three used gradients (SURVEY.md 0-7) from the saved forward state. Four sweeps, run as two paired ones: the
        discriminator's class path (1) and feature tap (2), and the decoder's sweeps (3) and (4) on decoder call 1, each walk
        back through one saved forward state, and train-mode BatchNorm is linear in its upstream once that state is fixed, so
        each pair shares every BatchNorm backward (x read once for both upstreams) and stacks its data gradients."""
        if self.mode in ("dcgan", "vae"):
            return self._backward_pixel_nle(st)
        hp, B = self.hp, st.B
        lam = float(hp["lambda_mse"])
        bd, bc = self.buckets["decoder."], self.buckets["discriminator."]
        cd1, cd2, cc, raw3, p = st.cd1, st.cd2, st.cc, st.raw3, st.p
        Fd = raw3[0].numel()
        # (1) discriminator, class-score path: g_dis = d loss_discriminator / d discriminator, plus d loss_dis / d(x_tilde, x_p)
        gp = E(3 * B)
        ones = self._ones(3 * B)
        L.bce_bwd(p[:B], ones, gp[:B], B, True, 1.0)
        L.bce_bwd(p[B:], ones, gp[B:], 2 * B, False, 1.0)
        # (2) discriminator, feature-tap path: d sum(mse) / d x_tilde (data gradient only; BN couples the whole 3B batch)
        draw3 = torch.empty_like(raw3)
        draw3[2 * B:].zero_()
        L.rowsqdiff_bwd(raw3[:B], raw3[B:2 * B], ones, draw3[:B], draw3[B:2 * B], B, Fd, 0.5)
        dimg_bce, dimg_mse = self.dis.backward_pair(bc.P, cc, gp, draw3, bc.G, False, live=(0, 2),
                                                    after_dw=lambda: self._allreduce_async([bc.flat_g]))
        # (3) decoder: g_dec = d [lambda * mse - (1 - lambda) * loss_dis] / d decoder over both decoder calls, paired on call 1
        # with (4): the mse term flows x_tilde -> decoder (data gradient) -> z. Call 1 accumulates first, as in four sweeps.
        dz = self.dec.backward_pair(bd.P, cd1, lam, dimg_mse, -(1.0 - lam), dimg_bce[:B], 1.0, dimg_mse, bd.G, False)
        self.dec.backward(bd.P, cd2, -(1.0 - lam), dimg_bce[B:], 0.0, None, bd.G, True, True, False)
        self._ev_dec = self._allreduce_async([bd.flat_g])   # loss sums, discriminator and decoder buckets are reduced here
        # (4, continued) encoder: g_enc = d [sum kl + sum mse] / d encoder
        dycat = self._encoder_backward(st, dz)
        st.sweeps = dict(dimg_bce=dimg_bce, dimg_mse=dimg_mse, dz=dz, dycat=dycat)

    def _backward_pixel_nle(self, st):
        """Modes 'dcgan' (train_vgan_stage1.py:374-380) and 'vae' (:382-387): no feature-tap sweep (2), because the pixel NLE
        replaces the feature MSE; bce_p is not in loss_discriminator, but train-mode BatchNorm couples the whole 3B batch, so
        its gradient slot is zero while x_tilde still receives an image gradient from the class path."""
        hp, B = self.hp, st.B
        lam = float(hp["lambda_mse"])
        bd, bc = self.buckets["decoder."], self.buckets["discriminator."]
        x, x_tilde, p = st.x, st.out["x_tilde"], st.p
        dcgan = self.mode == "dcgan"
        # (1) class path: g_dis = d [sum bce_o + sum bce_s] / d discriminator; image gradients only where loss_decoder has
        # the discriminator term ('dcgan'). 'vae' runs it every step: its gate is decided on the device.
        gp = E(3 * B)
        ones = self._ones(3 * B)
        L.bce_bwd(p[:B], ones, gp[:B], B, True, 1.0)
        gp[B:2 * B].zero_()
        L.bce_bwd(p[2 * B:], ones, gp[2 * B:], B, False, 1.0)
        dimg_bce = self.dis.backward_gan(bc.P, st.cc, gp, bc.G, False, True, (1, 3) if dcgan else None)
        self._allreduce_async([bc.flat_g])
        dnle = torch.empty_like(x_tilde)
        L.rowsqdiff_bwd(x_tilde, x, ones, dnle, None, B, x[0].numel(), 0.5)   # d sum(nle) / d x_tilde = x_tilde - x
        if dcgan:
            # (3) g_dec = d [lambda * sum nle - (1 - lambda) * loss_dis] / d decoder over both decoder calls; no encoder
            self.dec.backward(bd.P, st.cd1, lam, dnle, -(1.0 - lam), dimg_bce[:B], bd.G, False, True, False)
            self.dec.backward(bd.P, st.cd2, -(1.0 - lam), dimg_bce[B:], 0.0, None, bd.G, True, True, False)
            self._ev_dec = self._allreduce_async([bd.flat_g])
            st.sweeps = dict(dimg_bce=dimg_bce, dnle=dnle)
            return
        # 'vae': one decoder sweep over call 1 gives d sum(nle) / d decoder and dz; the backward is linear in its upstream,
        # so g_dec = lambda * those weight gradients and dz is the encoder's upstream at unit weight. x_p gets no gradient.
        dz = self.dec.backward(bd.P, st.cd1, 1.0, dnle, 0.0, None, bd.G, False, True, True)
        NN.join_side()
        L.scale_f32(bd.flat_g, lam)
        self._ev_dec = self._allreduce_async([bd.flat_g])
        dycat = self._encoder_backward(st, dz)
        st.sweeps = dict(dnle=dnle, dz=dz, dycat=dycat)

    def _encoder_backward(self, st, dz):
        """Reparameterisation / KL backward from dz, then the encoder sweep with its gradient exchange. Returns dycat."""
        be, B, z = self.buckets["encoder."], st.B, self.z
        mu, lv, eps = st.mu, st.lv, st.eps
        dycat = E(B, 2 * z, dtype=self.adt)
        # 'beta-vae' (:359-362): loss_encoder = beta / batch_size * sum kl + sum mse, the batch being the global one here
        self._klw = self.beta / float(B * self.world) if self.mode == "beta-vae" else 1.0
        L.reparam_kl_bwd(mu, lv, eps, dz, None, dycat[:, :z], dycat[:, z:], B, z, ld=2 * z, ldd=2 * z, gkl_const=self._klw)
        self._before_encoder_backward(mu, dycat)   # hook: DualWaeVaeGanStage1 adds the latent penalty gradient here
        # encoder bucket in two parts (SURVEY.md section 5): fc.0 / fc.1 / l_mu / l_var (67.6 MB, the tail of the flat buffer)
        # are complete after the first three backward kernels and reduce while the conv backward still runs; only the conv
        # part (4.1 MB) is exchanged after the last kernel
        split = min(off for k, (off, _) in be.offsets.items() if not k.startswith("conv."))
        if self.world > 1 and all(off < split for k, (off, _) in be.offsets.items() if k.startswith("conv.")):
            self.enc.backward(be.P, st.ce, dycat, be.G, False, True, True,
                              after_fc=lambda: self._allreduce_async([be.flat_g[split:]]))
            self._allreduce_async([be.flat_g[:split]])
        else:
            self.enc.backward(be.P, st.ce, dycat, be.G, False, True, True)
            self._allreduce_async([be.flat_g])
        return dycat

    _enc_bn_updates = 1

    def _before_encoder_backward(self, mu, dycat):
        pass

    def update(self, B_global):
        """Equilibrium gate (device side) + the three RMSprop updates (train_vgan_stage1.py:396-432), then repack."""
        hp = self.hp
        # Data parallel: the loss sums, the discriminator and the decoder buckets were exchanged during the encoder sweep, so
        # the gate, their two updates and their repacks run while the last exchange (the encoder's conv part, issued after the
        # final backward kernel: 0.2 ms exposed at 8 GPUs in profiles/r2_nccl_overlap_N8_B512_per_rank.txt) is still in flight;
        # only the encoder update waits for it. The three buckets are independent, so the order changes nothing numerically.
        ev = self._ev_dec
        staged = self.world > 1 and ev is not None
        if staged:
            NN.join_side()
            torch.cuda.current_stream().wait_event(ev)
            self._ev_dec = None
        else:
            self._wait_comm()
        gates = self.sc[8:10]
        dis_in = self.mode != "vae"   # 'vae' sets train_dis = False before the gate (train_vgan_stage1.py:387)
        if self.gate_on:
            L.vgan_gate_mix(self.sc, float(B_global), hp["margin"], hp["equilibrium"], dis_in, gates)
        else:
            gates[0:1].fill_(1.0 if dis_in else 0.0)
            gates[1:2].fill_(1.0)
        for pre, g in (("decoder.", gates[1:2]), ("discriminator.", gates[0:1]), ("encoder.", None)):
            if pre == "encoder." and self.mode == "dcgan":
                continue   # :374-380 trains no encoder: its parameters, square_avg and operand packs stay as they are
            if pre == "encoder." and staged:
                self._wait_comm()
            b = self.buckets[pre]
            L.multi_tensor_rmsprop([b.flat_p], [b.flat_g], [b.states[0]], self.lr[pre], hp["alpha"], hp["eps"], 0.0,
                                   None, g)
            self.nets[pre].refresh(b.P, inplace=True)

    def step(self, x, eps, z_p):
        """One full training iteration on device-resident inputs. Returns the device tensor of loss sums."""
        out = self.forward_backward(x, eps, z_p)
        self.update(x.shape[0] * self.world)
        return out

    def losses(self):
        """Host view of the last step's (globally reduced) loss sums, as the reference logs them (stage1 :391-394)."""
        s = self.sc.tolist()
        lam = float(self.hp["lambda_mse"])
        if self.mode in ("dcgan", "vae"):   # train_vgan_stage1.py:374-387 (the 'dcgan' loss_encoder is logged, not trained)
            loss_dis = s[0] + s[2]
            loss_enc = s[3] + s[5]
            loss_dec = lam * s[5] - ((1 - lam) * loss_dis if self.mode == "dcgan" else 0.0)
        else:
            loss_dis = s[0] + s[1] + s[2]
            loss_enc = self._klw * s[3] + s[4]
            loss_dec = lam * s[4] - (1 - lam) * loss_dis
        return dict(loss_encoder=loss_enc, loss_discriminator=loss_dis, loss_decoder=loss_dec,
                    nle=s[5], bce_o=s[0], bce_p=s[1], bce_s=s[2], kl=s[3], mse=s[4], train_dis=s[8] != 0,
                    train_dec=s[9] != 0)


class _WaeTrainer(_TrainerBase):
    """The Adam-trained WAE trainers: buckets "encoder." (the encoder that gives the latent z), "decoder." and the latent
    "discriminator."; sc[0..3] = L_fake, L_real, L_rec, L_pen."""

    def _adam(self, pre):
        b, hp = self.buckets[pre], self.hp
        L.multi_tensor_adam_dev([b.flat_p], [b.flat_g], [b.states[0]], [b.states[1]], self.lr[pre], hp["beta1"], hp["beta2"],
                                hp["eps"], self.t_dev)
        self.nets[pre].refresh(b.P, inplace=True)

    def _encoder_tail(self, ce, dmu):
        """End of the G-phase: the encoder sweep from dmu = d loss / d z (fp32 [B, z]; l_var receives no gradient), its
        exchange together with the loss sums, and the encoder's Adam step."""
        B, z = dmu.shape[0], self.z
        be = self.buckets["encoder."]
        dycat = Z(B, 2 * z, dtype=self.adt)
        L.cast2d(dmu, z, dycat[:, :z], 2 * z, B, z)
        be.flat_g.zero_()  # l_var receives no gradient (logvar unused): its slots stay zero and Adam leaves it unchanged
        self.nets["encoder."].backward(be.P, ce, dycat, be.G, False, True, False)
        self._allreduce_async([be.flat_g, self.sc[:8]])
        self._wait_comm()
        self._adam("encoder.")

    def losses(self):
        s = self.sc.tolist()
        return dict(loss_discriminator_fake=s[0], loss_discriminator_real=s[1], loss_reconstruction=s[2],
                    loss_penalty=s[3])


class WaeGanStage1(_WaeTrainer):
    """Stage-I WAE/GAN trainer (/root/reference/train/train_wae_stage1.py:259-311): visual Encoder, Decoder, latent
    WaeDiscriminator, three Adam(betas=(0.5, 0.999)) optimizers (the discriminator at lr / 2).

    D-phase: z_real = encoder(x) (encoder / decoder frozen), L_fake = -10 sum log(d(z_fake) + 1e-3),
    L_real = -10 sum log(1 - d(z_real) + 1e-3), Adam step on the discriminator. G-phase: the reference runs the encoder a
    second time on unchanged weights (:296) -- same z_real, so it is computed once and the BN running statistics are
    updated twice; x_recon = decoder(z_real), d(z_real) with the UPDATED discriminator, L_rec = sum 0.5 (x_recon - x)^2,
    L_pen = -10 sum log(d + 1e-3); Adam on the encoder (grad of L_rec + L_pen; l_var gets none) and the decoder (L_rec).

    penalty='mmd' (EXTENSION, parity unpinned: the reference has no MMD, SURVEY.md 0-3): no latent discriminator and no
    D-phase; L_pen = lambda_mmd * B * MMD_IMQ(z_real, z_fake) over this rank's batch (per-rank, like BatchNorm), one encoder
    forward. Everything else as train_wae_stage1.py:292-311.
    """

    def __init__(self, params, buffers, cfg, z=128, adt=BF16, hp=None, dist_group=None, penalty="gan", lambda_mmd=10.0,
                 sigma2=0.25):
        from .hp import HP_WAE

        if penalty not in ("gan", "mmd"):
            raise L.FmriError("penalty must be 'gan' (the reference's latent discriminator) or 'mmd'")
        self.cfg, self.z, self.adt = cfg, z, adt
        self.penalty, self.lambda_mmd, self.sigma2 = penalty, float(lambda_mmd), float(sigma2)
        self.hp = dict(HP_WAE if hp is None else hp)
        self.enc = NN.EncoderNet(cfg, z, adt)
        self.dec = NN.DecoderNet(cfg, z, adt)
        nets = OrderedDict((("encoder.", self.enc), ("decoder.", self.dec)))
        if penalty == "gan":
            self.dis = NN.WaeDiscriminatorNet(z, adt)
            nets["discriminator."] = self.dis
        lr = {"encoder.": float(self.hp["lr"]), "decoder.": float(self.hp["lr"]), "discriminator.": 0.5 * float(self.hp["lr"])}
        self._setup(params, buffers, nets, dict.fromkeys(nets, 2), lr, dist_group)
        self.t = 0
        self._mmd_ws = torch.empty(3, dtype=torch.float64, device="cuda")

    def step(self, x, z_fake):
        """x [B,3,H,W] fp32 NCHW, z_fake [B,z] fp32 (= 0.5 * N(0,1), train_wae_stage1.py:276), device resident."""
        B, z, gan = x.shape[0], self.z, self.penalty == "gan"
        be, bd = self.buckets["encoder."], self.buckets["decoder."]
        L.step_increment(self.t_dev)
        sc, ones = self.sc, self._ones(B)
        nbe, nbd = {}, {}
        ycat, ce = self.enc.forward(be.P, self.Ssub["encoder."], x, True, 2 if gan else 1, nbe)
        z_real = ycat[:, :z]
        if gan:   # ---------------- discriminator phase (:271-288)
            bc = self.buckets["discriminator."]
            p_real, p_fake, l, gp = self._latent_d_phase(self.dis, bc, z_real, z_fake, 10.0, sc)
            self._allreduce_async([bc.flat_g])
            self._wait_comm()
            self._adam("discriminator.")
        # ---------------- generator phase (:292-311)
        x_recon, cd = self.dec.forward(bd.P, self.Ssub["decoder."], z_real, True, 1, nbd)
        out = dict(z_real=z_real, x_recon=x_recon)
        if gan:
            p_real2, cr2 = self.dis.forward(bc.P, z_real)
            out.update(d_real=p_real, d_fake=p_fake, d_real_g=p_real2)
        rec = E(B)
        L.rowsqdiff_fwd(x_recon, x, rec, B, x[0].numel(), 0.5)
        L.vecsum(rec, B, 1.0, sc[2:3])
        if gan:
            L.bce_fwd(p_real2, l[:B], B, True, 10.0)
            L.vecsum(l[:B], B, 1.0, sc[3:4])
        else:
            lam = self.lambda_mmd * B
            L.mmd_imq_fwd(z_real, z_fake, B, z, self.sigma2, lam, sc[3:4], self._mmd_ws)
        dxr = torch.empty_like(x_recon)
        L.rowsqdiff_bwd(x_recon, x, ones, dxr, None, B, x[0].numel(), 0.5)
        if gan:
            L.bce_bwd(p_real2, ones, gp[:B], B, True, 10.0)
            dz_pen = self.dis.backward(bc.P, cr2, gp[:B], None, False, False, True)
        dz_rec = self.dec.backward(bd.P, cd, 1.0, dxr, 0.0, None, bd.G, False, True, True)
        self._allreduce_async([bd.flat_g])
        if gan:
            dmu = E(B, z)
            L.axpby_tanh_bwd(1.0, dz_rec, 1.0, dz_pen, None, dmu)
        else:
            dmu = dz_rec if dz_rec.dtype == F32 and dz_rec.is_contiguous() else dz_rec.to(F32).contiguous()
            L.mmd_imq_bwd(z_real, z_fake, B, z, self.sigma2, lam, dmu, accumulate=True)
        self._encoder_tail(ce, dmu)
        self._adam("decoder.")
        self._count_bn_updates("encoder.", nbe)
        self._count_bn_updates("decoder.", nbd)
        return out


class VaeGanCognitiveStage(_TrainerBase):
    """Stage-II / Stage-III cognitive VAE/GAN trainer (/root/reference/train/train_vgan_stage2.py:321-407,
    train_vgan_stage3.py:324-411) over VaeGanCognitive (models/vae_gan.py:323-432, mode 'vae').

    stage 2: trains {CognitiveEncoder, Discriminator}; the decoder is frozen; the discriminator's "real" batch is the
             teacher's reconstruction decoder(reparameterize(teacher.encoder(image))) (train-mode BN, frozen weights);
             no gate (train_dis=True, train_dec=False). Backward: class-score sweep (g_dis only), feature-tap data-gradient
             sweep -> decoder data-gradient sweep -> reparam/KL -> cognitive encoder.
    stage 3: trains {Decoder, Discriminator} with the equilibrium gate; the cognitive encoder is frozen.
    Both clamp gradients to [-1, 1] inside the fused RMSprop launch (stage2 :391,406; stage3 :402,410).
    Parameter keys: encoder.* (CognitiveEncoder), decoder.*, discriminator.*, teacher_net.encoder.* (stage 2 only)."""

    LATENT_DISCRIMINATOR = False
    mode, _klw = "vae-gan", 1.0   # losses() is VaeGanStage1's, with the 'vae-gan' formulas

    def __init__(self, params, buffers, cfg, stage, z=128, adt=BF16, hp=None, dist_group=None, voxels=None):
        from .hp import HP_VGAN, NUM_VOXELS

        if stage not in (2, 3):
            raise L.FmriError("stage must be 2 or 3")
        self.cfg, self.z, self.adt, self.stage = cfg, z, adt, stage
        self.hp = dict(HP_VGAN if hp is None else hp)
        self.cog = NN.CognitiveEncoderNet(voxels or NUM_VOXELS, z, adt)
        self.dec = NN.DecoderNet(cfg, z, adt)
        self.dis = NN.DiscriminatorNet(cfg, adt)
        nets = OrderedDict((("encoder.", self.cog), ("decoder.", self.dec), ("discriminator.", self.dis)))
        if stage == 2 or self.LATENT_DISCRIMINATOR:
            self.tenc = NN.EncoderNet(cfg, z, adt)
            nets["teacher_net.encoder."] = self.tenc
        if self.LATENT_DISCRIMINATOR:
            self.ldis = NN.WaeDiscriminatorNet(z, adt)
            nets["latent_discriminator."] = self.ldis
        # sc: [0..5] as VaeGanStage1; [8], [9] = gates
        self._setup(params, buffers, nets, {pre: 2 if pre == "latent_discriminator." else 1 for pre in nets},
                    dict.fromkeys(nets, float(self.hp["lr"])), dist_group)

    def forward_backward(self, fmri, image, eps, eps_t, z_p):
        """fmri [B,V], image [B,3,H,W], eps / eps_t / z_p [B,z]: fp32, device resident (eps_t is used in stage 2 only)."""
        hp, B, z, stage = self.hp, fmri.shape[0], self.z, self.stage
        lam = float(hp["lambda_mse"])
        be, bd, bc = self.buckets["encoder."], self.buckets["decoder."], self.buckets["discriminator."]
        nb = {pre: {} for pre in self.buckets}
        sc = self.sc
        ycat, ce = self.cog.forward(be.P, self.Ssub["encoder."], fmri, True, 1, nb["encoder."])
        mu, lv = ycat[:, :z], ycat[:, z:]
        zz, kl = E(B, z), E(B)
        L.reparam_kl_fwd(mu, lv, eps, zz, kl, B, z, ld=2 * z)
        x_tilde, cd1 = self.dec.forward(bd.P, self.Ssub["decoder."], zz, True, 1, nb["decoder."])
        gt_x = image
        if stage == 2:
            bt = self.buckets["teacher_net.encoder."]
            yt, _ = self.tenc.forward(bt.P, self.Ssub["teacher_net.encoder."], image, True, 1, nb["teacher_net.encoder."])
            zt = E(B, z)
            L.reparam_kl_fwd(yt[:, :z], yt[:, z:], eps_t, zt, None, B, z, ld=2 * z)
            gt_x, _ = self.dec.forward(bd.P, self.Ssub["decoder."], zt, True, 1, nb["decoder."])
        x_p, cd2 = self.dec.forward(bd.P, self.Ssub["decoder."], z_p, True, 1, nb["decoder."])
        raw3, p, cc = self.dis.forward(bc.P, self.Ssub["discriminator."], [gt_x, x_tilde, x_p], True, 2, True,
                                       nb["discriminator."])
        for pre, d in nb.items():
            self._count_bn_updates(pre, d)
        Fd = raw3[0].numel()
        mse, nle, bce = E(B), E(B), E(3 * B)
        L.rowsqdiff_fwd(raw3[:B], raw3[B:2 * B], mse, B, Fd, 0.5)
        L.rowsqdiff_fwd(gt_x, x_tilde, nle, B, gt_x[0].numel(), 0.5)
        L.bce_fwd(p[:B], bce[:B], B, True, 1.0)
        L.bce_fwd(p[B:], bce[B:], 2 * B, False, 1.0)
        for i, (v, n) in enumerate(((bce[:B], B), (bce[B:2 * B], B), (bce[2 * B:], B), (kl, B), (mse, B), (nle, B))):
            L.vecsum(v, n, 1.0, sc[i:i + 1])
        self._allreduce_async([sc[:8]])
        ones = self._ones(3 * B)
        gp = E(3 * B)
        L.bce_bwd(p[:B], ones, gp[:B], B, True, 1.0)
        L.bce_bwd(p[B:], ones, gp[B:], 2 * B, False, 1.0)
        # discriminator class-score sweep: g_dis; image gradients only when the decoder is trained (stage 3)
        dimg_bce = self.dis.backward_gan(bc.P, cc, gp, bc.G, False, True, (1, 3) if stage == 3 else None)
        self._allreduce_async([bc.flat_g])
        # feature-tap sweep (data gradient only): d sum(mse) / d x_tilde
        draw3 = torch.empty_like(raw3)
        draw3[2 * B:].zero_()
        L.rowsqdiff_bwd(raw3[:B], raw3[B:2 * B], ones, draw3[:B], draw3[B:2 * B], B, Fd, 0.5)
        dimg_mse = self.dis.backward_rec(bc.P, cc, draw3, None, False, False, (1, 2), live=(0, 2))
        if stage == 2:
            dz = self.dec.backward(bd.P, cd1, 1.0, dimg_mse, 0.0, None, None, False, False, True)
            dycat = E(B, 2 * z, dtype=self.adt)
            L.reparam_kl_bwd(mu, lv, eps, dz, None, dycat[:, :z], dycat[:, z:], B, z, ld=2 * z, ldd=2 * z, gkl_const=1.0)
            self.cog.backward(be.P, ce, dycat, be.G, False, True, True)
            self._allreduce_async([be.flat_g])
        else:
            self.dec.backward(bd.P, cd1, lam, dimg_mse, -(1.0 - lam), dimg_bce[:B], bd.G, False, True, False)
            self.dec.backward(bd.P, cd2, -(1.0 - lam), dimg_bce[B:], 0.0, None, bd.G, True, True, False)
            self._allreduce_async([bd.flat_g])
        return dict(gt_x=gt_x, x_tilde=x_tilde, x_p=x_p, disc_layer_nhwc=raw3, disc_class=p, mu=mu, logvar=lv, kl=kl,
                    mse=mse, bce=bce, nle=nle)

    def update(self, B_global):
        hp = self.hp
        self._wait_comm()
        gates = self.sc[8:10]
        if self.stage == 3:
            L.vgan_gate(self.sc, float(B_global), hp["margin"], hp["equilibrium"], gates)
            plan = (("decoder.", gates[1:2]), ("discriminator.", gates[0:1]))
        else:
            gates[0:1].fill_(1.0)   # stage 2: train_dis = True, train_dec = False, no gate (train_vgan_stage2.py:375-376)
            gates[1:2].fill_(0.0)
            plan = (("encoder.", None), ("discriminator.", None))
        for pre, g in plan:
            b = self.buckets[pre]
            L.multi_tensor_rmsprop([b.flat_p], [b.flat_g], [b.states[0]], self.lr[pre], hp["alpha"], hp["eps"], 1.0, None, g)
            self.nets[pre].refresh(b.P, inplace=True)

    def step(self, fmri, image, eps, eps_t, z_p):
        out = self.forward_backward(fmri, image, eps, eps_t, z_p)
        self.update(fmri.shape[0] * self.world)
        return out

    losses = VaeGanStage1.losses


class DualCognitiveStage3(VaeGanCognitiveStage):
    """BASELINE.json configs[3], "Stage III cognitive WAE/Dual-GAN with two discriminators and fixed cognitive encoder": a
    composite, not a single reference script (SURVEY.md 8d, C4). The image side is the Stage-III VAE/GAN update
    (/root/reference/train/train_vgan_stage3.py:324-411: decoder + image Discriminator, gate, gradient clamp, RMSprop); the
    latent side is the discriminator phase of /root/reference/train/train_wae_stage3.py:308-326: z_fake = the cognitive
    encoder's mu (the same forward), z_real = teacher.encoder(image) (train-mode BN, frozen weights),
    L_fake = -10 sum log(d(z_fake) + 1e-3), L_real = -10 sum log(1 - d(z_real) + 1e-3), Adam(5e-4, betas (0.5, 0.999)) on
    the latent WaeDiscriminator. Extra parameter keys: teacher_net.encoder.*, latent_discriminator.main.*."""

    LATENT_DISCRIMINATOR = True

    def __init__(self, params, buffers, cfg, z=128, adt=BF16, hp=None, hp_latent=None, dist_group=None, voxels=None):
        from .hp import HP_WAE23

        super().__init__(params, buffers, cfg, 3, z, adt, hp, dist_group, voxels)
        self.hp_lat = dict(HP_WAE23 if hp_latent is None else hp_latent)
        self.t = 0
        self.lsc = Z(2)  # latent L_fake, L_real (sums); all-reduced with the latent discriminator's gradient bucket

    def forward_backward(self, fmri, image, eps, z_p):
        out = super().forward_backward(fmri, image, eps, None, z_p)
        bt, bl = self.buckets["teacher_net.encoder."], self.buckets["latent_discriminator."]
        nbt = {}
        yt, _ = self.tenc.forward(bt.P, self.Ssub["teacher_net.encoder."], image, True, 1, nbt)
        self._count_bn_updates("teacher_net.encoder.", nbt)
        z_fake, z_real = out["mu"], yt[:, :self.z]
        p_real, p_fake, _, _ = self._latent_d_phase(self.ldis, bl, z_real, z_fake, 10.0, self.lsc)
        self._allreduce_async([bl.flat_g, self.lsc])
        out.update(z_real=z_real, d_real=p_real, d_fake=p_fake)
        return out

    def update(self, B_global):
        super().update(B_global)
        L.step_increment(self.t_dev)
        b, hp = self.buckets["latent_discriminator."], self.hp_lat
        L.multi_tensor_adam_dev([b.flat_p], [b.flat_g], [b.states[0]], [b.states[1]], float(hp["lr_dis"]), hp["beta1"],
                                hp["beta2"], hp["eps"], self.t_dev)
        self.ldis.refresh(b.P, inplace=True)

    def step(self, fmri, image, eps, z_p):
        out = self.forward_backward(fmri, image, eps, z_p)
        self.update(fmri.shape[0] * self.world)
        return out

    def losses(self):
        d = super().losses()
        lf, lr = self.lsc.tolist()
        d.update(loss_discriminator_fake=lf, loss_discriminator_real=lr)
        return d


class WaeCognitiveStage(_WaeTrainer):
    """Stage-II / Stage-III cognitive WAE/GAN trainer (/root/reference/train/train_wae_stage2.py:274-328,
    train_wae_stage3.py:295-347) over WaeGanCognitive (models/vae_gan.py:532-578) and the Stage-I teacher's visual encoder.

    Both stages: D-phase on z_fake = cognitive_encoder(fmri) vs z_real = teacher.encoder(image) (train-mode BN, frozen
    weights), L_fake = -10 sum log(d(z_fake) + 1e-3), L_real = -10 sum log(1 - d(z_real) + 1e-3), Adam(5e-4) on the latent
    discriminator. G-phase: the scripts run the cognitive encoder a second time on unchanged weights (same output: computed
    once, BN running statistics updated twice), x_recon = decoder(z), d from the UPDATED discriminator,
    L_rec = nn.MSELoss()(x_recon, image) (a MEAN over all elements), L_pen = -10 mean log(d + 1e-3).
      stage 2 (:274-328): an extra, unused teacher reconstruction decoder(teacher.encoder(image)) runs first for its BN side
               effects (:284-285); trains the cognitive encoder on L_rec + L_pen with Adam(1e-3); decoder frozen.
      stage 3 (:295-347): trains the DECODER on L_rec only (:338-347) with Adam(1e-3); cognitive encoder frozen.
    Data parallel: the two means are taken over the GLOBAL batch (each rank scales by 1 / (world * B_local)), so the SUM
    all-reduce of the gradient buckets reproduces the single-process step on the concatenated batch up to per-rank BatchNorm.
    Parameter keys: encoder.* (CognitiveEncoder), decoder.*, discriminator.main.*, teacher_net.encoder.*."""

    def __init__(self, params, buffers, cfg, stage, z=128, adt=BF16, hp=None, dist_group=None, voxels=None):
        from .hp import HP_WAE23, NUM_VOXELS

        if stage not in (2, 3):
            raise L.FmriError("stage must be 2 or 3")
        self.cfg, self.z, self.adt, self.stage = cfg, z, adt, stage
        self.hp = dict(HP_WAE23 if hp is None else hp)
        self.cog = NN.CognitiveEncoderNet(voxels or NUM_VOXELS, z, adt)
        self.dec = NN.DecoderNet(cfg, z, adt)
        self.dis = NN.WaeDiscriminatorNet(z, adt)
        self.tenc = NN.EncoderNet(cfg, z, adt)
        nets = OrderedDict((("encoder.", self.cog), ("decoder.", self.dec), ("discriminator.", self.dis),
                            ("teacher_net.encoder.", self.tenc)))
        # sc: [0..3] = L_fake, L_real (sums), L_rec, L_pen (global means)
        lr = {"encoder.": float(self.hp["lr"]), "decoder.": float(self.hp["lr"]), "discriminator.": float(self.hp["lr_dis"])}
        self._setup(params, buffers, nets, dict.fromkeys(nets, 2), lr, dist_group)
        self.t = 0

    def step(self, fmri, image):
        """fmri [B,V], image [B,3,H,W]: fp32, device resident."""
        B, z, stage = fmri.shape[0], self.z, self.stage
        Bg = float(B * self.world)
        be, bd, bc = self.buckets["encoder."], self.buckets["decoder."], self.buckets["discriminator."]
        bt = self.buckets["teacher_net.encoder."]
        L.step_increment(self.t_dev)
        sc, ones = self.sc, self._ones(B)
        nb = {pre: {} for pre in self.buckets}
        # teacher encoder: stage 2 runs it twice on the same input (:284 and the D-phase), stage 3 once
        yt, _ = self.tenc.forward(bt.P, self.Ssub["teacher_net.encoder."], image, True, 2 if stage == 2 else 1,
                                  nb["teacher_net.encoder."])
        z_real = yt[:, :z]
        if stage == 2:   # unused teacher reconstruction: BatchNorm running statistics of the decoder only
            self.dec.forward(bd.P, self.Ssub["decoder."], z_real, True, 1, nb["decoder."])
        # cognitive encoder: D-phase and G-phase forwards see the same weights -> one forward, two BN updates
        ycat, ce = self.cog.forward(be.P, self.Ssub["encoder."], fmri, True, 2, nb["encoder."])
        z_fake = ycat[:, :z]
        # ---------------- discriminator phase
        p_real, p_fake, l, gp = self._latent_d_phase(self.dis, bc, z_real, z_fake, 10.0, sc)
        self._allreduce_async([bc.flat_g])
        self._wait_comm()
        self._adam("discriminator.")
        # ---------------- generator phase
        x_recon, cd = self.dec.forward(bd.P, self.Ssub["decoder."], z_fake, True, 1, nb["decoder."])
        p2, c2 = self.dis.forward(bc.P, z_fake)
        Fimg = image[0].numel()
        rec = E(B)
        L.rowsqdiff_fwd(x_recon, image, rec, B, Fimg, 1.0 / (Bg * Fimg))
        L.vecsum(rec, B, 1.0, sc[2:3])
        L.bce_fwd(p2, l[:B], B, True, 10.0 / Bg)
        L.vecsum(l[:B], B, 1.0, sc[3:4])
        dxr = torch.empty_like(x_recon)
        L.rowsqdiff_bwd(x_recon, image, ones, dxr, None, B, Fimg, 1.0 / (Bg * Fimg))
        if stage == 2:
            L.bce_bwd(p2, ones, gp[:B], B, True, 10.0 / Bg)
            dz_pen = self.dis.backward(bc.P, c2, gp[:B], None, False, False, True)
            dz_rec = self.dec.backward(bd.P, cd, 1.0, dxr, 0.0, None, None, False, False, True)
            dmu = E(B, z)
            L.axpby_tanh_bwd(1.0, dz_rec, 1.0, dz_pen, None, dmu)
            self._encoder_tail(ce, dmu)
        else:
            self.dec.backward(bd.P, cd, 1.0, dxr, 0.0, None, bd.G, False, True, False)
            self._allreduce_async([bd.flat_g, sc[:8]])
            self._wait_comm()
            self._adam("decoder.")
        for pre, d in nb.items():
            self._count_bn_updates(pre, d)
        return dict(z_fake=z_fake, z_real=z_real, x_recon=x_recon, d_real=p_real, d_fake=p_fake, d_real_g=p2)


class GraphedStep:
    """One training step captured in a CUDA graph and replayed: for launch-bound batch sizes (Stage I at batch 64 is 276
    kernel launches in 5 ms, i.e. the host's launch rate, not the GPU, sets the step time). Every trainer of this module is
    capturable on one GPU: the equilibrium gate is decided on the device (fmri_vgan_gate) and Adam's step count lives in
    device memory (fmri_step_increment / fmri_multi_tensor_adam_dev), so no host-side scalar changes from step to step.

        g = GraphedStep(trainer, x, eps, z_p)      # warms up (3 eager steps), then captures
        out = g(x, eps, z_p)                       # copies the inputs into the graph's static buffers and replays

    The tensors in `out` live in the graph's memory pool and are overwritten by the next replay."""

    def __init__(self, trainer, *inputs, warmup=3):
        if not isinstance(trainer, _TrainerBase) or trainer.world != 1:
            raise L.FmriError("GraphedStep captures a single-GPU trainer of this module (NCCL collectives are not captured)")
        if isinstance(trainer, VaeGanStage1) and not trainer.gate_on:
            raise L.FmriError("GraphedStep needs the device-side gate (gate=True)")
        self.tr = trainer
        self.static = [t.clone() if t is not None else None for t in inputs]
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):   # eager warm-up: lazy workspaces, function attributes, tensor-map cache
            for _ in range(warmup):
                trainer.step(*self.static)
        cur.wait_stream(side)
        self.recaptures = -1
        self._capture()

    def _capture(self):
        """Capture one step. Learning rates, margin / equilibrium and lambda_mse are HOST scalars baked into the captured
        kernel arguments, so the values captured are remembered and __call__ re-captures when the trainer's differ
        (end_epoch() and load_state_dict() change them: ExponentialLR 0.98 per epoch, train_vgan_stage1.py:446-457)."""
        trainer = self.tr
        torch.cuda.synchronize()
        nbt0 = dict(trainer.nbt)
        n0 = L.launch_count()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = trainer.step(*self.static)
        self.launches = L.launch_count() - n0           # kernels per replay (the host counter only saw the capture)
        self.nbt_inc = {k: v - nbt0.get(k, 0) for k, v in trainer.nbt.items()}
        trainer.nbt = nbt0                               # the capture itself executed nothing
        self.captured = (dict(trainer.lr), dict(trainer.hp))
        self.recaptures += 1

    def __call__(self, *inputs):
        if (self.tr.lr, self.tr.hp) != self.captured:
            self._capture()
        for s, t in zip(self.static, inputs):
            if s is not None and t is not s:
                s.copy_(t, non_blocking=True)
        self.graph.replay()
        nbt = self.tr.nbt
        for k, v in self.nbt_inc.items():
            nbt[k] = nbt.get(k, 0) + v
        return self.out


class DualWaeVaeGanStage1(VaeGanStage1):
    """The dual WAE/GAN Stage-I step of /root/reference/train/wae_vgan_stage1.py:282-441 (mode 'vae-gan'; SURVEY.md 8a row a16),
    TORCH >= 2 SEMANTICS (the decoder `step()` of :417 acts on None gradients and is a no-op): the Stage-I VAE/GAN step plus a
    latent WaeDiscriminator (RMSprop) that is trained on z_real = encoder(x) vs z_fake (:380-397) and whose penalty
    -lam sum log(d(z_real) + 1e-3), evaluated with the UPDATED latent discriminator (:401-411), is accumulated into the
    encoder's gradient (:421). The script's second and third encoder forwards see unchanged weights, so the encoder runs once
    and its BatchNorm running statistics are updated three times; the unused decoder(z_real) forward of :405 runs for its
    BatchNorm side effects. NOTE: the latent discriminator is updated inside forward_backward (the penalty needs it).
    Extra parameter keys: latent_discriminator.main.*; step(x, eps, z_p, z_fake)."""

    _enc_bn_updates = 3
    LATENT_DISCRIMINATOR = True

    def __init__(self, params, buffers, cfg, z=128, adt=BF16, hp=None, dist_group=None, gate=True, lam=1.0):
        super().__init__(params, buffers, cfg, z, adt, hp, dist_group, gate)
        self.lam = float(lam)
        self.lsc = Z(4)   # L_fake, L_real, L_pen (batch sums)
        self._z_fake = None

    def _before_encoder_backward(self, mu, dycat):
        hp, z, lam = self.hp, self.z, self.lam
        B = mu.shape[0]
        bl, bd = self.buckets["latent_discriminator."], self.buckets["decoder."]
        ones = self._ones(B)
        # ---- latent discriminator phase (:380-397)
        p_real, p_fake, l, gp = self._latent_d_phase(self.ldis, bl, mu, self._z_fake, lam, self.lsc)
        if self.world > 1:   # the penalty needs the globally updated latent discriminator
            self._allreduce_async([bl.flat_g])
            torch.cuda.current_stream().wait_stream(self.comm_stream)
        L.multi_tensor_rmsprop([bl.flat_p], [bl.flat_g], [bl.states[0]], self.lr["latent_discriminator."], hp["alpha"],
                               hp["eps"], 0.0, None, None)
        self.ldis.refresh(bl.P, inplace=True)
        # ---- penalty (:401-417): the unused reconstruction forward (BatchNorm running statistics), then d with the new weights
        nbd = {}
        self.dec.forward(bd.P, self.Ssub["decoder."], mu, True, 1, nbd)
        self._count_bn_updates("decoder.", nbd)
        p2, c2 = self.ldis.forward(bl.P, mu)
        L.bce_fwd(p2, l[:B], B, True, lam)
        L.vecsum(l[:B], B, 1.0, self.lsc[2:3])
        L.bce_bwd(p2, ones, gp[:B], B, True, lam)
        dz_pen = self.ldis.backward(bl.P, c2, gp[:B], None, False, False, True)
        dycat[:, :z].add_(dz_pen.to(dycat.dtype))   # :421 the encoder sweep accumulates onto the penalty gradient
        self._allreduce_async([self.lsc])   # logged sums are global, like sc[0..5] (waited on in update())
        self._d = dict(z_real=mu, d_real=p_real, d_fake=p_fake, d_real_g=p2)

    def forward_backward(self, x, eps, z_p, z_fake):
        self._z_fake = z_fake
        out = super().forward_backward(x, eps, z_p)
        out.update(self._d)
        return out

    def step(self, x, eps, z_p, z_fake):
        out = self.forward_backward(x, eps, z_p, z_fake)
        self.update(x.shape[0] * self.world)
        return out

    def losses(self):
        d = super().losses()
        lf, lr, lp, _ = self.lsc.tolist()
        d.update(loss_discriminator_fake=lf, loss_discriminator_real=lr, loss_penalty=lp)
        return d
