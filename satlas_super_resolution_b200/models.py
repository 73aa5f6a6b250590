"""MODEL_REGISTRY['SSRESRGANModel'] -- the training-step object `ssr/train.py` drives (ssr/train.py:62-145).

Same constructor (`opt` dict from the YAML), the same methods the loop calls (update_learning_rate, feed_data,
optimize_parameters, get_current_learning_rate, get_current_log, save, validation, resume_training, test,
get_current_visuals) and the same attributes (net_g, net_g_ema, net_d, optimizer_g/d, output, log_dict, lr, gt) as
/root/reference/ssr/models/ssr_esrgan_model.py (on basicsr SRGANModel / SRModel / BaseModel).  The arithmetic of
feed_data / optimize_parameters / test runs in ESRGANTrainer (trainer.py) over libssr_b200.
"""
import os
from collections import OrderedDict
from copy import deepcopy

import torch

from . import archs, losses  # noqa: F401  (registers the archs and losses)
from .registry import MODEL_REGISTRY, _register, build_network
from .trainer import ESRGANTrainer
from . import weights


class _OptimizerHandle:
    """The torch.optim surface basicsr touches (param_groups for the LR schedule, state_dict for checkpoints), backed by
    the fused Adam(+EMA) state of the trainer."""

    def __init__(self, state, net):
        self._state, self._net = state, net
        self.param_groups = [{"lr": state.lr, "initial_lr": state.lr, "betas": state.betas, "eps": state.eps,
                              "weight_decay": state.wd, "params": list(net.parameters())}]

    def sync(self):
        g = self.param_groups[0]
        self._state.lr, self._state.betas, self._state.eps, self._state.wd = g["lr"], tuple(g["betas"]), g["eps"], g["weight_decay"]

    def zero_grad(self, set_to_none=False):
        self._state.g.flat.zero_()

    def state_dict(self):
        return {"step": self._state.step_count, "exp_avg": self._state.m.flat.detach().cpu(),
                "exp_avg_sq": self._state.v.flat.detach().cpu(), "param_groups": [{k: v for k, v in self.param_groups[0].items()
                                                                                   if k != "params"}]}

    def load_state_dict(self, sd):
        self._state.step_count = int(sd["step"])
        self._state.m.flat.copy_(sd["exp_avg"])
        self._state.v.flat.copy_(sd["exp_avg_sq"])
        for k, v in sd["param_groups"][0].items():
            self.param_groups[0][k] = v
        self.sync()


class SSRESRGANModel:
    def __init__(self, opt):
        self.opt = opt
        self.is_train = opt.get("is_train", True)
        if opt.get("num_gpu", 1) == 0:
            raise RuntimeError("SSRESRGANModel (B200 engine): num_gpu == 0 / CPU execution is not available")
        rank = int(os.environ.get("LOCAL_RANK", 0))
        self.device = torch.device("cuda", rank if opt.get("dist") else torch.cuda.current_device())
        train_opt = opt.get("train") or {}
        # ---- networks (registry-built, reference key schema); the trainer then owns their storage
        self.net_g = build_network(opt["network_g"])
        self._load_if_given(self.net_g, "pretrain_network_g", "param_key_g", "strict_load_g", "params")
        self.log_dict = OrderedDict()
        self.optimizers, self.schedulers = [], []
        self.trainer = None
        if not self.is_train:
            # basicsr SRModel with is_train False builds net_g only (no D, losses, optimizers, EMA copy): forward-only engine
            self.net_g.to(self.device).eval()
            return
        if "network_d" not in opt:
            raise ValueError("SSRESRGANModel (is_train): the option file has no network_d")
        self.net_d = build_network(opt["network_d"])
        self._load_if_given(self.net_d, "pretrain_network_d", "param_key_d", "strict_load_d", "params")
        for unsupported in ("ldl_opt", "clip_opt"):
            if train_opt.get(unsupported):
                raise NotImplementedError(f"train.{unsupported}: this loss is outside the built hot path (SURVEY.md section 2 rows 5, 13)")
        pix, per, gan = train_opt.get("pixel_opt") or {}, train_opt.get("perceptual_opt") or {}, train_opt.get("gan_opt") or {}
        ssim = train_opt.get("ssim_opt") or {}                       # ssr_esrgan_model.py:87-90
        if ssim and ssim.get("type", "SSIMLoss") != "SSIMLoss":
            raise NotImplementedError(f"train.ssim_opt.type '{ssim.get('type')}' is not built (ssr/losses/basic_loss.py:50 SSIMLoss is)")
        if gan and gan.get("gan_type", "vanilla") != "vanilla":
            raise NotImplementedError("only gan_type 'vanilla' is built")
        optim_g = dict(train_opt.get("optim_g", {"type": "Adam", "lr": 1e-4, "betas": [0.9, 0.99]}))
        optim_d = dict(train_opt.get("optim_d", optim_g))
        for o in (optim_g, optim_d):
            if o.get("type", "Adam") != "Adam":
                raise NotImplementedError("only Adam is built (esrgan_s2naip_urban.yml:98-107)")
            extra = set(o) - {"type", "lr", "betas", "weight_decay", "eps"}
            if extra:
                raise NotImplementedError(f"Adam options {sorted(extra)} are not built")
        if optim_g.get("eps", 1e-8) != 1e-8 or optim_d.get("eps", 1e-8) != 1e-8:
            raise NotImplementedError("Adam eps other than 1e-8 is not built")
        vgg_sd = weights.resolve_vgg19_state(per.get("vgg_seed", opt.get("vgg_seed")), per.get("vgg_path")) if per else None
        cfg = dict(network_g=dict(num_in_ch=self.net_g.num_in_ch, num_block=self.net_g.num_block, scale=self.net_g.scale),
                   ema_decay=train_opt.get("ema_decay", 0), lr=optim_g.get("lr", 1e-4), betas=tuple(optim_g.get("betas", (0.9, 0.99))),
                   weight_decay=optim_g.get("weight_decay", 0.0),
                   lr_d=optim_d.get("lr", 1e-4), betas_d=tuple(optim_d.get("betas", (0.9, 0.99))),
                   weight_decay_d=optim_d.get("weight_decay", 0.0),
                   pixel_weight=pix.get("loss_weight", 1.0) if pix else 0.0, gan_weight=gan.get("loss_weight", 0.1),
                   ssim_weight=ssim.get("loss_weight", 1.0) if ssim else 0.0,
                   perceptual=bool(per), layer_weights=per.get("layer_weights"), perceptual_weight=per.get("perceptual_weight", 1.0),
                   use_input_norm=per.get("use_input_norm", True), range_norm=per.get("range_norm", False),
                   feed_disc_lr=bool(opt.get("feed_disc_lr")), l1_gt_usm=opt.get("l1_gt_usm", True) is not False,
                   percep_gt_usm=opt.get("percep_gt_usm", True) is not False, gan_gt_usm=opt.get("gan_gt_usm", True) is not False,
                   net_d_iters=train_opt.get("net_d_iters", 1), net_d_init_iters=train_opt.get("net_d_init_iters", 0),
                   cuda_graph=bool(opt.get("cuda_graph", True)), overlap=opt.get("overlap"))   # overlap: None = $SSR_OVERLAP (ops.overlap_enabled)
        if per and not cfg["layer_weights"]:
            raise ValueError("perceptual_opt needs layer_weights")
        pg = torch.distributed.group.WORLD if (opt.get("dist") and torch.distributed.is_initialized()) else None
        # ESRGANTrainer broadcasts rank 0's parameters / buffers / EMA to every rank (what DDP does at construction)
        self.trainer = ESRGANTrainer(self.net_g.state_dict(), self.net_d.state_dict(), vgg_sd, cfg, device=self.device,
                                     process_group=pg)
        tr = self.trainer
        self.net_g.to(self.device)
        self.net_g.adopt(tr.gbuf, tr.ggrad)
        self.net_d.to(self.device)
        self.net_d.adopt(tr.dbuf, tr.dgrad)
        for k, b in self.net_d.named_buffers():
            b.data = tr.d_uv[k]
        if tr.gema is not None:
            self.net_g_ema = build_network(opt["network_g"]).to(self.device)
            self.net_g_ema.adopt(tr.gema, tr.gema.like())
            ema_path = opt.get("path", {}).get("pretrain_network_g")
            if ema_path:
                sd = torch.load(ema_path, map_location="cpu")
                if "params_ema" in sd:
                    self.net_g_ema.load_state_dict(sd["params_ema"], strict=opt["path"].get("strict_load_g", True))
            self.net_g_ema.eval()
        self.optimizer_g = _OptimizerHandle(tr.opt_g, self.net_g)
        self.optimizer_d = _OptimizerHandle(tr.opt_d, self.net_d)
        self.optimizers = [self.optimizer_g, self.optimizer_d]
        sched = dict(train_opt.get("scheduler", {"type": "MultiStepLR", "milestones": [400000], "gamma": 0.5}))
        if sched.get("type", "MultiStepLR") not in ("MultiStepLR", "MultiStepRestartLR"):
            raise NotImplementedError("only MultiStepLR is built (esrgan_s2naip_urban.yml:109-112)")
        self._milestones, self._gamma = list(sched.get("milestones", [])), sched.get("gamma", 0.5)
        self._sched_iter = 0
        self.net_g.train()
        self.net_d.train()

    # ------------------------------------------------------------------ basicsr BaseModel surface
    def _load_if_given(self, net, path_key, param_key, strict_key, default_key):
        path = self.opt.get("path", {}).get(path_key)
        if path:
            self.load_network(net, path, self.opt["path"].get(strict_key, True), self.opt["path"].get(param_key, default_key))

    def load_network(self, net, load_path, strict=True, param_key="params"):
        sd = torch.load(load_path, map_location="cpu")
        if param_key is not None:
            if param_key not in sd and "params" in sd:
                param_key = "params"
            sd = sd[param_key]
        sd = OrderedDict((k[7:] if k.startswith("module.") else k, v) for k, v in sd.items())
        net.load_state_dict(sd, strict=strict)

    def update_learning_rate(self, current_iter, warmup_iter=-1):
        """basicsr BaseModel.update_learning_rate with MultiStepLR (+ linear warm-up)"""
        if current_iter > 1:
            self._sched_iter += 1
        factor = self._gamma ** sum(1 for m in self._milestones if self._sched_iter >= m)
        for o in self.optimizers:
            g = o.param_groups[0]
            lr = g["initial_lr"] * factor
            if current_iter < warmup_iter:
                lr = g["initial_lr"] / warmup_iter * current_iter
            g["lr"] = lr
            o.sync()

    def get_current_learning_rate(self):
        return [o.param_groups[0]["lr"] for o in self.optimizers[:1]]

    def feed_data(self, data):
        """ssr_esrgan_model.py:104-117 -- data['lr'] uint8 [B, T*C, h, w], data['hr'] uint8 [B, 3, H, W]"""
        if "hr" not in data or self.trainer is None:
            self.lr = (data["lr"].to(self.device).float() / 255).contiguous()
            if "hr" in data:
                self.gt = (data["hr"].to(self.device).float() / 255).contiguous()
            return
        self.trainer.feed_data(data["lr"], data["hr"], data.get("old_hr"))
        self.lr, self.gt, self.gt_usm = self.trainer.lr, self.trainer.gt, self.trainer.gt_usm

    def optimize_parameters(self, current_iter):
        self.trainer.optimize_parameters(current_iter)
        self.output = self.trainer.output
        self.net_g.mark_weights_changed()

    def get_current_log(self):
        self.log_dict = self.trainer.get_current_log()
        return self.log_dict

    def test(self):
        """ssr_esrgan_model.py:235-244: net_g_ema (eval) when it exists, else net_g in eval mode"""
        if self.trainer is not None:
            self.output = self.trainer.test(self.lr)
            return
        with torch.no_grad():
            self.net_g.eval()
            self.output = self.net_g(self.lr)

    def get_current_visuals(self):
        out = OrderedDict(lr=self.lr.detach().cpu(), result=self.output.detach().cpu())
        if hasattr(self, "gt"):
            out["gt"] = self.gt.detach().cpu()
        return out

    def validation(self, dataloader, current_iter, tb_logger, save_img=False):
        """basicsr BaseModel.validation -> nondist_validation (ssr/models/ssr_esrgan_model.py:269-352)"""
        return self.nondist_validation(dataloader, current_iter, tb_logger, save_img)

    def _initialize_best_metric_results(self, dataset_name, metrics2run):
        """ssr_esrgan_model.py:253-267"""
        if not hasattr(self, "best_metric_results"):
            self.best_metric_results = {}
        if dataset_name in self.best_metric_results:
            return
        record = {}
        for metric, content in metrics2run.items():
            better = content.get("better", "higher")
            record[metric] = dict(better=better, val=float("-inf") if better == "higher" else float("inf"), iter=-1)
        self.best_metric_results[dataset_name] = record

    def _update_best_metric_result(self, dataset_name, metric, val, current_iter):
        rec = self.best_metric_results[dataset_name][metric]
        if (rec["better"] == "higher" and val >= rec["val"]) or (rec["better"] != "higher" and val <= rec["val"]):
            rec["val"], rec["iter"] = val, current_iter

    def _log_validation_metric_values(self, current_iter, dataset_name, tb_logger):
        import logging
        msg = f"Validation {dataset_name}\n"
        for metric, value in self.metric_results.items():
            msg += f"\t # {metric}: {value:.4f}"
            if hasattr(self, "best_metric_results"):
                best = self.best_metric_results[dataset_name][metric]
                msg += f"\tBest: {best['val']:.4f} @ {best['iter']} iter"
            msg += "\n"
        logging.getLogger("basicsr").info(msg)
        if tb_logger:
            for metric, value in self.metric_results.items():
                tb_logger.add_scalar(f"metrics/{dataset_name}/{metric}", value, current_iter)

    def nondist_validation(self, dataloader, current_iter, tb_logger, save_img):
        """The loop of ssr_esrgan_model.py:269-352 with the per-image host work batched on the GPU: EMA-generator forward
        (test()), tensor2img, and PSNR / SSIM / cPSNR / LPIPS for the whole validation batch at once (metrics.py); metric options are
        checked before the first batch.  Any batch size works
        (the reference's loop assumes 1); results are averaged over images.  Image dumps (`save_img`) are PNG IO outside the hot
        path and are not written."""
        from . import metrics as M
        ds = getattr(dataloader, "dataset", None)
        dataset_name = ds.opt["name"] if ds is not None and hasattr(ds, "opt") else "val"
        sect = self.opt.get("test" if dataset_name == "test" else "val") or {}
        metrics2run = sect.get("metrics")
        with_metrics = metrics2run is not None
        if with_metrics:
            for name, mopt in metrics2run.items():
                if mopt["type"] not in M.METRIC_REGISTRY:
                    raise NotImplementedError(f"metric '{mopt['type']}' ({name}) is outside the built path (calculate_psnr / "
                                              "calculate_ssim / calculate_cpsnr / calculate_lpips run batched on the GPU; "
                                              "CLIPScore needs CLIP ViT checkpoints that are not part of this engine)")
                M.check_metric_opt(mopt)
            self.metric_results = {metric: 0.0 for metric in metrics2run}
            self._initialize_best_metric_results(dataset_name, metrics2run)
        n_img = 0
        for val_data in dataloader:
            self.feed_data(val_data)
            self.test()
            if with_metrics and "hr" in val_data:
                data = dict(img=M.to_uint8_images(self.output.float()), img2=M.to_uint8_images(self.gt.float()))
                for name, mopt in metrics2run.items():
                    self.metric_results[name] += float(sum(M.calculate_metric(data, mopt)))
            n_img += int(val_data["lr"].shape[0])
        if with_metrics:
            for metric in self.metric_results:
                self.metric_results[metric] /= max(1, n_img)
                self._update_best_metric_result(dataset_name, metric, self.metric_results[metric], current_iter)
            self._log_validation_metric_values(current_iter, dataset_name, tb_logger)
        return n_img

    def _save_dir(self, sub):
        root = self.opt.get("path", {}).get(sub) or os.path.join(self.opt.get("path", {}).get("experiments_root", "experiments"), sub)
        os.makedirs(root, exist_ok=True)
        return root

    def save(self, epoch, current_iter):
        """basicsr SRGANModel.save: net_g_<iter>.pth = {'params', 'params_ema'}, net_d_<iter>.pth = {'params'}, <iter>.state"""
        tag = "latest" if current_iter == -1 else str(current_iter)
        mdir = self._save_dir("models")
        cpu = lambda sd: OrderedDict((k, v.detach().cpu()) for k, v in sd.items())
        g = {"params": cpu(self.net_g.state_dict())}
        if hasattr(self, "net_g_ema"):
            g["params_ema"] = cpu(self.net_g_ema.state_dict())
        torch.save(g, os.path.join(mdir, f"net_g_{tag}.pth"))
        torch.save({"params": cpu(self.net_d.state_dict())}, os.path.join(mdir, f"net_d_{tag}.pth"))
        if current_iter != -1:
            state = {"epoch": epoch, "iter": current_iter, "optimizers": [o.state_dict() for o in self.optimizers],
                     "schedulers": [{"last_epoch": self._sched_iter}]}
            torch.save(state, os.path.join(self._save_dir("training_states"), f"{current_iter}.state"))

    def resume_training(self, resume_state):
        for o, s in zip(self.optimizers, resume_state["optimizers"]):
            o.load_state_dict(s)
        self._sched_iter = resume_state["schedulers"][0]["last_epoch"]


_register(MODEL_REGISTRY, SSRESRGANModel)
