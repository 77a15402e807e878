"""Training / evaluation driver — drop-in for the reference's train_generative.py.

downsample (:36-42), get_gen_loss (:44-65), train_on_dataset (:67-214),
get_model (:221-240), add_gen_model_parse (:301-318).  get_gen_loss routes the
reconstruction term through the fused catalog cross-entropy so the (B*L, N)
logits, the mask and the soft-max never reach HBM; everything else keeps the
reference's semantics (CE mean over B*L rows, KL summed, Adam without decay).
"""
import numpy as np
import torch

from ._lib import PcvError
from .autograd import CatalogCEFn, KLFn  # noqa: F401
from .env.response_model import sample_users
from .models.listcvae import UserListCVAEWithPrior
from .models.pivotcvae import PIVOTCVAE_MODELS


def downsample(pred, slate, n_neg=1000.0):
    """pred * (onehot(target) U Bernoulli(n_neg/N)) on a materialised logit matrix
    (train_generative.py:36-42).  Kept for API parity; training never calls it."""
    mask = torch.bernoulli(torch.full_like(pred, n_neg / pred.shape[1]))
    mask.scatter_(1, slate.reshape(-1, 1), 1.0)
    return pred * mask


def _as_tensor(x, dtype, device):
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=dtype)
    return torch.as_tensor(np.asarray(x), dtype=dtype, device=device)


def get_gen_loss(batch_data, model, lossFun, beta, n_neg=1000):
    """-> (loss, recLoss, KLD) with autograd attached (train_generative.py:44-65).

    lossFun is accepted for signature parity; the reconstruction term is always the
    mean soft-max CE the reference builds with nn.CrossEntropyLoss (:105)."""
    dev = model.docEmbed.weight.device
    slates = _as_tensor(batch_data["slates"], torch.int64, dev)
    users = _as_tensor(batch_data["users"], torch.int64, dev)
    targets = _as_tensor(batch_data["responses"], torch.float32, dev)
    vp = getattr(model, "_vp", None)
    train_vp = vp is not None and model.docEmbed.weight.requires_grad
    if train_vp and not getattr(model, "_vp_train", False):
        raise PcvError("get_gen_loss: vocab-parallel training with trainable tables (fine_tune=True) needs "
                       "enable_vocab_parallel(train_tables=True)")
    # vocab-parallel: the masked and candidate forwards touch O(n_neg) columns per row and run on the whole catalog;
    # with train_tables their table gradient is computed for this rank's shard only (grad_table)
    grad_table = model.item_table() if train_vp else None
    pMu, pLogvar = model.get_prior(targets, users)
    rx, z, mu, logvar, _ = model.forward_latent(slates, targets, users)
    if model.candidateFlag:
        # sampled soft-max over the data loader's candidates (train_generative.py:52-56): fused gather-dot-CE
        from .autograd import CandidateCEFn
        M = slates.numel()
        cand = _as_tensor(batch_data["sample_candidates"], torch.int64, dev).reshape(M, -1)
        tpos = _as_tensor(batch_data["sample_targets"], torch.int64, dev).reshape(-1)
        recLoss = CandidateCEFn.apply(rx.reshape(M, -1), model.full_table(), cand, tpos, model.docEmbed.weight,
                                      grad_table)
        KLD = KLFn.apply(mu, logvar, pMu, pLogvar)
        model.noise.flush_eager()
        return recLoss + beta * KLD, recLoss, KLD
    N = model.docEmbed.weight.shape[0]
    if n_neg > N:
        raise RuntimeError("n_neg (%d) > number of items (%d): torch.bernoulli would reject p > 1" % (n_neg, N))
    keep = float(n_neg) / float(N)
    bitmask = model.noise.pop("mask")
    M = slates.numel()
    kw = dict(seed=0, offset=0)
    if bitmask is None and keep < 1.0:
        kw = model.noise.stream_args(M)
    if vp is not None and bitmask is None and keep >= 1.0:
        # vocab-parallel full-catalog soft-max: partial records over this rank's shard, one all-gather, merge
        # (SURVEY §8e).  Masked training (keep < 1) touches O(n_neg) columns per row and stays unsharded below.
        from .autograd import VocabParallelCEFn
        recLoss, _, _ = VocabParallelCEFn.apply(rx.reshape(M, -1), model.item_table(), model.docEmbed.weight.detach(),
                                                slates.reshape(-1), vp[0], getattr(model, "ce_engine", "exact"),
                                                model.docEmbed.weight)
    else:
        recLoss, _, _ = CatalogCEFn.apply(rx.reshape(M, -1), model.full_table(), slates.reshape(-1), keep, bitmask, kw["seed"],
                                          kw["offset"], kw.get("offset_dev"), getattr(model, "ce_engine", "exact"),
                                          model.docEmbed.weight, grad_table)
    KLD = KLFn.apply(mu, logvar, pMu, pLogvar)
    loss = recLoss + beta * KLD
    model.noise.flush_eager()
    return loss, recLoss, KLD


def recommendation_test(model, resp_model, bs, n_trial=100, n_context=5):
    """The per-epoch 100 x 5 recommendation test (train_generative.py:168-195):
    -> (min, mean, max) expected click counts per context, each (n_context,)."""
    enc = torch.zeros(n_context, n_trial)
    maxnc = torch.zeros(n_context, n_trial)
    minnc = torch.zeros(n_context, n_trial)
    dev = model.docEmbed.weight.device
    with torch.no_grad():
        for k in range(n_trial):
            users = sample_users(resp_model, bs)
            context = torch.zeros(bs, n_context, device=dev)
            stats = []
            for i in range(n_context):
                context[:, i] = 1
                rSlates, _ = model.recommend(context, users, return_item=True)
                resp = torch.sigmoid(resp_model(rSlates.view(bs, -1), users))
                nc = resp.sum(1)
                stats.append(torch.stack([nc.mean(), nc.max(), nc.min()]))
            st = torch.stack(stats).cpu()  # one device->host sync per trial instead of 15
            enc[:, k], maxnc[:, k], minnc[:, k] = st[:, 0], st[:, 1], st[:, 2]
    return minnc.mean(1), enc.mean(1), maxnc.mean(1)


def train_on_dataset(trainset, valset, model, model_path, logger, resp_model, bs, epochs, lr, decay, beta):
    """Epoch loop of train_generative.py:67-214: Adam(lr) (no weight decay, F10), validation with
    n_neg = trainset.nCandidate, recommendation test, save-best whole-model pickle."""
    from torch.utils.data import DataLoader
    trainLoader = DataLoader(trainset, batch_size=bs, shuffle=True, num_workers=0)
    valLoader = DataLoader(valset, batch_size=bs, shuffle=False, num_workers=0)
    optimizer = torch.optim.Adam(model.parameters(), lr=lr)
    trainHistory, valHistory = [], []
    bestValLoss = float("inf")
    for epoch in range(epochs):
        logger.log("Epoch " + str(epoch + 1))
        losses = []
        for batchData in trainLoader:
            optimizer.zero_grad()
            loss, recLoss, kld = get_gen_loss(batchData, model, None, beta)
            losses.append(loss.detach())
            loss.backward()
            optimizer.step()
        trainHistory.append(float(torch.stack(losses).mean()))
        logger.log("train loss: " + str(trainHistory[-1]))
        vl, vr, vk = [], [], []
        with torch.no_grad():
            for batchData in valLoader:
                loss, recLoss, KLD = get_gen_loss(batchData, model, None, beta, n_neg=trainset.nCandidate)
                vl.append(loss)
                vr.append(recLoss)
                vk.append(KLD)
        valHistory.append(float(torch.stack(vl).mean()))
        logger.log("validation Loss: %s = %s + %s * %s" % (valHistory[-1], float(torch.stack(vr).mean()), beta,
                                                           float(torch.stack(vk).mean())))
        mn, me, mx = recommendation_test(model, resp_model, bs)
        for i in range(len(me)):
            logger.log("Expected response (%d): %s; %s; %s" % (i + 1, mn[i].numpy(), me[i].numpy(), mx[i].numpy()))
        if epoch == 0 or valHistory[-1] < bestValLoss - 1e-3:
            torch.save(model, open(model_path, "wb"))
            logger.log("Save best model")
            bestValLoss = valHistory[-1]
    return trainHistory, valHistory


def get_model(args, response_model):
    """Factory of train_generative.py:221-240 (struct strings like "[54,256,256]")."""
    parse = lambda s: [int(v) for v in s[1:-1].split(",")]
    uemb = None if response_model.noUser else response_model.userEmbed
    if args.model == "listcvae":
        return UserListCVAEWithPrior(response_model.docEmbed, uemb, args.s, args.dim, args.z_size, args.s + 1,
                                     parse(args.enc_struct), parse(args.dec_struct), parse(args.prior_struct),
                                     args.nouser, args.device)
    if args.model in PIVOTCVAE_MODELS:
        return PIVOTCVAE_MODELS[args.model](response_model.docEmbed, uemb, args.s, args.dim, args.z_size, args.s + 1,
                                            parse(args.enc_struct), parse(args.psm_struct), parse(args.scm_struct),
                                            parse(args.prior_struct), args.nouser, args.device)
    return None


def main(args):
    """Orchestration of train_generative.py:242-301: load the environment + datasets, build the generative
    model, train it (one beta, or the beta grid when args.beta <= 0).

    Data IO is NOT part of this package (SURVEY §8: out of scope): `data_extract`, `data_loader`, `my_utils`
    and `settings` are the reference's own modules, imported from the reference checkout on sys.path.
    Two slips of the reference's beta-grid branch are read as intended: the undefined `betaModelPath`
    (:293) is the `modelPath` built two lines above it, and the bare `Logger` (:291) is `utils.Logger`."""
    try:
        import data_extract as dae
        import my_utils as utils
        import settings
        from data_loader import UserSlateResponseDataset
    except ImportError as e:   # pragma: no cover - depends on the host environment
        raise ImportError("train_generative.main needs the reference's data modules (data_extract, data_loader, "
                          "my_utils, settings) on sys.path: %s" % e)
    logger = utils.Logger(utils.make_gen_model_path(args, "log/"))
    if args.dataset not in ("yoochoose", "movielens"):      # simulation environment
        respModel, trainset, valset = dae.load_simulation(args, logger)
    else:
        if args.dataset == "yoochoose":
            train, val, _ = dae.read_yoochoose(entire_set=False)
        else:
            train, val = dae.read_movielens(entire=False)
        trainset = UserSlateResponseDataset(train["features"], train["sessions"], train["responses"], args.nouser)
        if args.dataset == "yoochoose":
            trainset.balance_n_click()
        valset = UserSlateResponseDataset(val["features"], val["sessions"], val["responses"], args.nouser)
        respModel = torch.load(open(args.resp_path, "rb"), weights_only=False)
    trainset.init_sampling(args.nneg)
    valset.init_sampling(args.nneg)
    respModel.to(args.device)
    respModel.device = args.device
    gen_model = get_model(args, respModel)
    if not args.mask_train:
        logger.log("Candidate training")
        gen_model.candidateFlag = True
    else:
        logger.log("Mask training")
    if args.beta > 0:
        modelPath = utils.make_gen_model_path(args, "trained_gen/")
        train_on_dataset(trainset, valset, gen_model, modelPath, logger, respModel,
                         args.batch_size, args.epochs, args.lr, args.wdecay, args.beta)
        return
    logger.log("Beta test")
    for beta in settings.BETA_LIST:
        args.beta = beta
        betaLogger = utils.Logger(utils.make_gen_model_path(args, "log_beta/"))
        modelPath = utils.make_gen_model_path(args, "trained_beta/")
        betaLogger.log("beta = " + str(beta))
        train_on_dataset(trainset, valset, gen_model, modelPath, betaLogger, respModel,
                         args.batch_size, args.epochs, args.lr, args.wdecay, beta)
        logger.log("Done, model saved to: " + modelPath)


def add_gen_model_parse(parser):
    parser.add_argument("--dim", type=int, default=8)
    parser.add_argument("--model", type=str, default="pivotcvae_gt_pi")
    parser.add_argument("--z_size", type=int, default=16)
    parser.add_argument("--mask_train", action="store_true")
    parser.add_argument("--enc_struct", type=str, default="[54,256,256]")
    parser.add_argument("--prior_struct", type=str, default="[14,128,128]")
    parser.add_argument("--beta", type=float, default=-1)
    parser.add_argument("--dec_struct", type=str, default="[30,256,256,40]")
    parser.add_argument("--psm_struct", type=str, default="[30,256,256,8]")
    parser.add_argument("--scm_struct", type=str, default="[38,256,256,32]")
    return parser
