"""Loss graph of the Swapping Autoencoder on the B200 operator surface.

Restates reference ``models/swapping_autoencoder_model.py`` (+ the command dispatch of ``models/base_model.py``)
so the training step can run on a box where the reference checkout is absent; the reference's own file also
runs unchanged on this operator surface (INTEGRATION.md).  Method names, the ``command=`` dispatch, loss keys,
loss weights and the order of random draws follow the reference so that, given the same parameters and RNG
state, both produce the same numbers.
"""
import os

import torch

from . import networks, util
from .stylegan2_op import filter_reuse
from .stylegan2_op.blocks import data_gradients_only


class BaseModel(torch.nn.Module):
    """reference models/base_model.py: option holder, checkpoint I/O and ``forward(command=...)`` dispatch."""

    @staticmethod
    def modify_commandline_options(parser, is_train):
        return parser

    def __init__(self, opt):
        super().__init__()
        self.opt = opt
        # one process per GPU: the model lives on THIS process's device (torch.cuda.current_device(), set from LOCAL_RANK by
        # parallel.init_distributed), never on cuda:0 of every rank (the reference's single-process DataParallel uses
        # cuda:0, models/base_model.py:18)
        self.device = torch.device('cuda', torch.cuda.current_device()) if opt.num_gpus > 0 else torch.device('cpu')

    def initialize(self):
        pass

    def per_gpu_initialize(self):
        pass

    def get_parameters_for_mode(self, mode):
        return {}

    def _checkpoint_dir(self, name=None):
        return os.path.join(self.opt.checkpoints_dir, name or self.opt.name)

    def save(self, total_steps_so_far):
        """``<N>k_checkpoint.pth`` + ``latest_checkpoint.pth`` symlink (reference base_model.py:33-41)."""
        savedir = self._checkpoint_dir()
        os.makedirs(savedir, exist_ok=True)
        fname = "%dk_checkpoint.pth" % (total_steps_so_far // 1000)
        torch.save(self.state_dict(), os.path.join(savedir, fname))
        link = os.path.join(savedir, "latest_checkpoint.pth")
        if os.path.lexists(link):
            os.remove(link)
        os.symlink(fname, link)

    def load(self, path=None, strict_shapes=True, partial_shapes=None):
        """Copy tensors by key from a (reference-format) state_dict (reference base_model.py:43-112).  Keys missing from the
        checkpoint are reported and skipped, as in the reference.  A tensor whose shape differs raises unless partial loading
        is asked for (``strict_shapes=False`` or ``opt.partial_shape_loading``): the reference asks yes / no / all on the
        terminal for every such key; there, as here, only tensors of rank 1, 2 or 4 are eligible and only the corner the
        checkpoint does not cover is zeroed."""
        if partial_shapes is None:
            partial_shapes = (not strict_shapes) or bool(getattr(self.opt, "partial_shape_loading", False))
        if path is None:
            pretrained = getattr(self.opt, "pretrained_name", None)
            name = pretrained if (self.opt.isTrain and pretrained is not None) else self.opt.name
            path = os.path.join(self._checkpoint_dir(name), "%s_checkpoint.pth" % self.opt.resume_iter)
        if not os.path.exists(path):
            assert self.opt.isTrain, "In test mode, the checkpoint file must exist"
            print("checkpoint %s does not exist; training starts from scratch" % path)
            return False
        ckpt = torch.load(path, map_location="cpu")        # copied parameter by parameter onto this rank's own device
        with torch.no_grad():
            for name, own in self.state_dict().items():
                if not self.opt.isTrain and (name.startswith("D.") or name.startswith("Dpatch.")):
                    continue
                if name not in ckpt:
                    print("Key %s does not exist in checkpoint. Skipping..." % name)
                    continue
                src = ckpt[name]
                if own.shape == src.shape:
                    own.copy_(src)
                    continue
                message = "Key [%s]: Shape does not match the created model (%s) and loaded checkpoint (%s)" % (
                    name, tuple(own.shape), tuple(src.shape))
                if not partial_shapes:
                    raise ValueError(message + " — pass strict_shapes=False (or opt.partial_shape_loading) to force-load the "
                                     "common sub-block, the reference's interactive 'all' answer")
                print(message)
                ms = [min(a, b) for a, b in zip(own.shape, src.shape)]
                if own.dim() != src.dim() or len(ms) not in (1, 2, 4):
                    print("Skipping min_shape of %s" % str(ms))           # e.g. the 5-D ModulatedConv2d weights
                    continue
                common = tuple(slice(0, m) for m in ms)
                corner = tuple(slice(m, None) for m in ms)
                own[common].copy_(src[common].to(own.device))
                own[corner].zero_()                                  # only the far corner is cleared (reference :75-83)
        return True

    def forward(self, *args, command=None, **kwargs):
        if command is None:
            raise ValueError(command)
        method = getattr(self, command)
        assert callable(method), "[%s] is not a method of %s" % (command, type(self).__name__)
        # one command = one loss evaluation on fixed parameters: derived filter tensors are shared between the
        # several passes each network makes inside it (stylegan2_op/conv.py filter_reuse)
        with filter_reuse():
            return method(*args, **kwargs)


class SwappingAutoencoderModel(BaseModel):
    @staticmethod
    def modify_commandline_options(parser, is_train):
        BaseModel.modify_commandline_options(parser, is_train)
        parser.add_argument("--spatial_code_ch", default=8, type=int)
        parser.add_argument("--global_code_ch", default=2048, type=int)
        parser.add_argument("--lambda_R1", default=10.0, type=float)
        parser.add_argument("--lambda_patch_R1", default=1.0, type=float)
        parser.add_argument("--lambda_L1", default=1.0, type=float)
        parser.add_argument("--lambda_GAN", default=1.0, type=float)
        parser.add_argument("--lambda_PatchGAN", default=1.0, type=float)
        parser.add_argument("--patch_min_scale", default=1 / 8, type=float)
        parser.add_argument("--patch_max_scale", default=1 / 4, type=float)
        parser.add_argument("--patch_num_crops", default=8, type=int)
        parser.add_argument("--patch_use_aggregation", type=util.str2bool, default=True)
        return parser

    # ------------------------------------------------------------------ construction
    def initialize(self):
        opt = self.opt
        self.E = networks.create_network(opt, opt.netE, "encoder")
        self.G = networks.create_network(opt, opt.netG, "generator")
        if opt.lambda_GAN > 0.0:
            self.D = networks.create_network(opt, opt.netD, "discriminator")
        if opt.lambda_PatchGAN > 0.0:
            self.Dpatch = networks.create_network(opt, opt.netPatchD, "patch_discriminator")
        # discriminator iteration counter for lazy R1 (StyleGAN2 appendix B); part of the state_dict contract
        self.register_buffer("num_discriminator_iters", torch.zeros(1, dtype=torch.long))
        self.l1_loss = torch.nn.L1Loss()
        if (not opt.isTrain) or opt.continue_train:
            self.load()
        if opt.num_gpus > 0:
            self.to(self.device)

    # ------------------------------------------------------------------ helpers
    def swap(self, x):
        """exchange the two members of every consecutive pair of the minibatch (reference :53-60)"""
        assert x.shape[0] % 2 == 0, "Minibatch size must be a multiple of 2"
        return x.reshape(x.shape[0] // 2, 2, *x.shape[1:]).flip(1).reshape(x.shape)

    def get_random_crops(self, x, crop_window=None):
        opt = self.opt
        return util.apply_random_crop(x, opt.patch_size, (opt.patch_min_scale, opt.patch_max_scale),
                                      num_crops=opt.patch_num_crops)

    # ------------------------------------------------------------------ discriminator side
    def compute_image_discriminator_losses(self, real, rec, mix):
        lam = self.opt.lambda_GAN
        if lam == 0.0:
            return {}
        if getattr(self.opt, "batch_discriminator_passes", False):
            # extension: D has no cross-sample operation, so one pass over the concatenated batch gives the same
            # per-sample predictions with a third of the launches and fuller tiles on the small late layers
            pred_real, pred_rec, pred_mix = self.D(torch.cat([real, rec, mix])).split([real.size(0), rec.size(0), mix.size(0)])
        else:
            pred_real, pred_rec, pred_mix = self.D(real), self.D(rec), self.D(mix)
        return {
            "D_real": util.gan_loss(pred_real, should_be_classified_as_real=True) * lam,
            "D_rec": util.gan_loss(pred_rec, should_be_classified_as_real=False) * (0.5 * lam),
            "D_mix": util.gan_loss(pred_mix, should_be_classified_as_real=False) * (0.5 * lam),
        }

    def compute_patch_discriminator_losses(self, real, mix):
        opt = self.opt
        if getattr(opt, "batch_discriminator_passes", False):
            # same three crop draws in the same order (the feature extractor draws nothing), one pass over all of them
            if real.size(1) <= 4 and real.is_cuda == mix.is_cuda:
                crops, sizes = util.apply_random_crops_multi([real, real, mix], opt.patch_size,
                                                             (opt.patch_min_scale, opt.patch_max_scale), opt.patch_num_crops)
            else:
                parts = [self.get_random_crops(real), self.get_random_crops(real), self.get_random_crops(mix)]
                crops, sizes = torch.cat(parts), [c.size(0) for c in parts]
            n = crops.size(1)
            real_feat, target_feat, mix_feat = self.Dpatch.extract_features(crops).split([b * n for b in sizes])
            if opt.patch_use_aggregation:
                real_feat = self.Dpatch.aggregate_features(real_feat, sizes[0], n)
        else:
            real_feat = self.Dpatch.extract_features(self.get_random_crops(real), aggregate=opt.patch_use_aggregation)
            target_feat = self.Dpatch.extract_features(self.get_random_crops(real))
            mix_feat = self.Dpatch.extract_features(self.get_random_crops(mix))
        return {
            "PatchD_real": util.gan_loss(self.Dpatch.discriminate_features(real_feat, target_feat),
                                         should_be_classified_as_real=True) * opt.lambda_PatchGAN,
            "PatchD_mix": util.gan_loss(self.Dpatch.discriminate_features(real_feat, mix_feat),
                                        should_be_classified_as_real=False) * opt.lambda_PatchGAN,
        }

    def compute_discriminator_losses(self, real):
        self.num_discriminator_iters.add_(1)
        sp, gl = self.E(real)
        b = real.size(0)
        assert b % 2 == 0, "Batch size must be even on each GPU."
        rec = self.G(sp[:b // 2], gl[:b // 2])        # reconstruction of the first half only
        mix = self.G(self.swap(sp), gl)
        losses = self.compute_image_discriminator_losses(real, rec, mix)
        if self.opt.lambda_PatchGAN > 0.0:
            losses.update(self.compute_patch_discriminator_losses(real, mix))
        return losses, {}, sp.detach(), gl.detach()

    def compute_R1_loss(self, real):
        """R1 gradient penalty on D (w.r.t. the image) and on Dpatch (w.r.t. both crop sets); needs the
        second-order autograd of every op in D / Dpatch (reference :138-185)."""
        # both autograd.grad calls below ask for gradients with respect to images / crops only: the recorded backward skips
        # weight gradients and the fused blocks take their closed-form double backward (stylegan2_op/blocks.py)
        with data_gradients_only():
            return self._compute_R1_loss(real)

    def _compute_R1_loss(self, real):
        opt = self.opt
        penalty = 0.0
        if opt.lambda_R1 > 0.0:
            real.requires_grad_()
            pred = self.D(real).sum()
            g, = torch.autograd.grad(outputs=pred, inputs=[real], create_graph=True, retain_graph=True)
            penalty = g.pow(2).sum(list(range(1, g.ndim))) * (opt.lambda_R1 * 0.5)
        crop_penalty = 0.0
        if opt.lambda_patch_R1 > 0.0:
            real_crop = self.get_random_crops(real).detach().requires_grad_()
            target_crop = self.get_random_crops(real).detach().requires_grad_()
            real_feat = self.Dpatch.extract_features(real_crop, aggregate=opt.patch_use_aggregation)
            target_feat = self.Dpatch.extract_features(target_crop)
            pred = self.Dpatch.discriminate_features(real_feat, target_feat).sum()
            g_real, g_target = torch.autograd.grad(outputs=pred, inputs=[real_crop, target_crop],
                                                   create_graph=True, retain_graph=True)
            dims = list(range(1, g_real.ndim))
            crop_penalty = (g_real.pow(2).sum(dims) + g_target.pow(2).sum(dims)) * (0.5 * opt.lambda_patch_R1 * 0.5)
        return {"D_R1": penalty + crop_penalty}

    # ------------------------------------------------------------------ generator side
    def compute_generator_losses(self, real, sp_ma=None, gl_ma=None):
        opt = self.opt
        losses, metrics = {}, {}
        b = real.size(0)
        sp, gl = self.E(real)
        rec = self.G(sp[:b // 2], gl[:b // 2])
        sp_mix = self.swap(sp)
        metrics["L1_dist"] = self.l1_loss(rec, real[:b // 2])
        if opt.lambda_L1 > 0.0:
            losses["G_L1"] = metrics["L1_dist"] * opt.lambda_L1
        if opt.crop_size >= 1024:
            # memory-saving rule of the reference (:201-205): only the second half goes through the mix branch
            real, gl, sp_mix = real[b // 2:], gl[b // 2:], sp_mix[b // 2:]
        mix = self.G(sp_mix, gl)
        if opt.lambda_GAN > 0.0:
            if getattr(opt, "batch_discriminator_passes", False):
                pred_rec, pred_mix = self.D(torch.cat([rec, mix])).split([rec.size(0), mix.size(0)])
            else:
                pred_rec, pred_mix = self.D(rec), self.D(mix)
            losses["G_GAN_rec"] = util.gan_loss(pred_rec, should_be_classified_as_real=True) * (opt.lambda_GAN * 0.5)
            losses["G_GAN_mix"] = util.gan_loss(pred_mix, should_be_classified_as_real=True) * (opt.lambda_GAN * 1.0)
        if opt.lambda_PatchGAN > 0.0:
            real_feat = self.Dpatch.extract_features(self.get_random_crops(real),
                                                     aggregate=opt.patch_use_aggregation).detach()
            mix_feat = self.Dpatch.extract_features(self.get_random_crops(mix))
            losses["G_mix"] = util.gan_loss(self.Dpatch.discriminate_features(real_feat, mix_feat),
                                            should_be_classified_as_real=True) * opt.lambda_PatchGAN
        return losses, metrics

    # ------------------------------------------------------------------ inference callers (SURVEY.md §8 f4)
    def get_visuals_for_snapshot(self, real):
        if self.opt.isTrain:
            real = real[:2] if self.opt.num_gpus > 1 else real[:4]
        sp, gl = self.E(real)
        layout = util.resize2d_tensor(util.visualize_spatial_code(sp), real)
        return {"real": real, "layout": layout, "rec": self.G(sp, gl), "mix": self.G(sp, self.swap(gl))}

    def fix_noise(self, sample_image=None):
        if sample_image is not None:
            sp, gl = self.E(sample_image)
            self.G(sp, gl)          # one pass so every NoiseInjection knows its map size
        return self.G.fix_and_gather_noise_parameters()

    def encode(self, image, extract_features=False):
        return self.E(image, extract_features=extract_features)

    def decode(self, spatial_code, global_code):
        return self.G(spatial_code, global_code)

    def decode_regions(self, spatial_code, texture_codes, masks):
        """Region-wise texture editing: decode with texture code k inside region k.  texture_codes [N, K, C]; masks [N, K, hm, wm],
        non-negative and summing to 1 over K at every pixel (soft masks blend codes).  The code map sum_k masks[:, k] texture_codes[:, k]
        is built at the masks' resolution and handed to G, which interpolates it to each layer."""
        if texture_codes.dim() != 3 or masks.dim() != 4 or tuple(masks.shape[:2]) != tuple(texture_codes.shape[:2]):
            raise ValueError("decode_regions: texture_codes [N, K, C] and masks [N, K, h, w] expected, got %s and %s"
                             % (tuple(texture_codes.shape), tuple(masks.shape)))
        if bool((masks < 0).any()) or not torch.allclose(masks.sum(dim=1), masks.new_ones(()), rtol=0.0, atol=1e-4):
            raise ValueError("decode_regions: masks must be non-negative and sum to 1 over the regions at every pixel")
        code_map = torch.einsum("nkc,nkhw->nchw", texture_codes, masks.to(texture_codes.dtype))
        return self.G(spatial_code, code_map)

    def get_parameters_for_mode(self, mode):
        if mode == "generator":
            return list(self.G.parameters()) + list(self.E.parameters())
        if mode == "discriminator":
            params = []
            if self.opt.lambda_GAN > 0.0:
                params += list(self.D.parameters())
            if self.opt.lambda_PatchGAN > 0.0:
                params += list(self.Dpatch.parameters())
            return params
        raise ValueError(mode)
