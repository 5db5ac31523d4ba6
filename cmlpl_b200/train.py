"""``python -m cmlpl_b200.train`` -- the reference's train.py on the B200 kernels.

Every flag of train.py:355-380 is kept with its default (``--dataID`` is accepted as int or str).
The mutual-learning step (train.py:149-278) is the function ``mutual_step`` below: two BaseNet2
peers, supervised CE, memory-bank pseudo-label smoothing, masked soft-CE cross supervision and the
pseudo-label-graph contrastive loss, two backward passes and two Adam updates -- every tensor
op on the path is a libcmlpl_sm100.so kernel (torch holds the memory, slices and concatenates).
Reference quirks are reproduced on purpose: the literal 256 pointer stride and the ``queue_ptr1``
update that reads ``queue_ptr`` (train.py:234,237), zero-initialised bank rows entering the softmax
denominator, thr=1 masking everything in epoch 0.
Differences (documented, opt-in free): batches are gathered on the GPU from the PCA cube instead of
a DataLoader over XP.npy; noise / dropout use the device generator; no SVG / CSV reporting.
By default the step runs as ONE ``cmlpl_train_step`` call (cmlpl_b200/fused_step.py: tcgen05 convolutions in fp16
operands / fp32 accumulation, 15 launches in a CUDA graph); ``--fp32_step`` selects ``mutual_step`` below, the fp32
path that meets the reference's 1e-5 bar.
"""
from __future__ import annotations

import argparse
import math
import os
import random
import time
from dataclasses import dataclass, field

import numpy as np
import torch

from . import losses, ops
from .hsi_loader import HSIDataSet
from .tools.hyper_tools import DATASETS, CalAccuracy, test_whole
from .tools.models import BaseNet2


def seed_torch(seed=1088):
    """train.py:50-58."""
    random.seed(seed)
    os.environ['PYTHONHASHSEED'] = str(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    torch.cuda.manual_seed_all(seed)


@dataclass
class MutualState:
    """What train.py keeps across steps (train.py:118-145)."""
    Base: BaseNet2
    Base1: BaseNet2
    opt: torch.optim.Optimizer
    opt1: torch.optim.Optimizer
    queue_feats: torch.Tensor
    queue_probs: torch.Tensor
    queue_feats1: torch.Tensor
    queue_probs1: torch.Tensor
    queue_ptr: int = 0
    queue_ptr1: int = 0
    extras: dict = field(default_factory=dict)


def make_state(num_features, num_classes, args, device, w=20) -> MutualState:
    """Both peers at window ``w`` (the dataset's: 20, or 11 for ``sample_generation --w 11``)."""
    Base = BaseNet2(num_features=num_features, dropout=args.dropout, num_classes=num_classes, w=w).to(device)
    Base1 = BaseNet2(num_features=num_features, dropout=args.dropout, num_classes=num_classes, w=w).to(device)
    qs = 5 * args.labeled_batch_size * 2                                        # train.py:138,142
    z = lambda *s: torch.zeros(*s, device=device)
    return MutualState(Base, Base1, losses.FusedAdam(Base.parameters(), lr=args.lr),
                       losses.FusedAdam(Base1.parameters(), lr=args.lr),
                       z(qs, 1024), z(qs, num_classes), z(qs, 1024), z(qs, num_classes))


def mutual_step(st: MutualState, XP_b_all, X_b_all, XP_e_all, X_e_all, Y_train, epoch, batch_index, args,
                drop_masks=(None, None)):
    """One step of train.py:150-278 given the two peers' (already noise-augmented) input batches
    ``[labelled ; unlabelled]``.  Returns the five loss_hist columns as a CUDA tensor (no host sync)
    plus a dict of intermediates for the parity tests."""
    T = args.temperature
    bs = Y_train.size(0)
    st.opt1.zero_grad()
    st.opt.zero_grad()
    st.Base.train()
    st.Base1.train()
    out_b, feat_b = st.Base(XP_b_all, X_b_all, drop_masks[0])                    # :175
    out_e, feat_e = st.Base1(XP_e_all, X_e_all, drop_masks[1])                   # :185
    labeled_output, x_feature = out_b[:bs], feat_b[:bs]
    un_b_output, xs_feature = out_b[bs:], feat_b[bs:]
    labeled_output1, x_feature1 = out_e[:bs], feat_e[:bs]
    un_e_output, xw_feature = out_e[bs:], feat_e[bs:]
    cls = losses.cross_entropy(labeled_output, Y_train)                          # :191
    cls1 = losses.cross_entropy(labeled_output1, Y_train)                        # :192
    adap_mask = args.thr * math.exp(-0.5 * ((epoch / args.num_epochs) ** 2))     # :147-148,221
    smooth = epoch > 0 or batch_index > args.queue_batch                         # :212
    with torch.no_grad():
        C = out_b.size(1)
        btu = un_b_output.size(0)
        n = bs + btu
        feats_u_w = xw_feature.detach().contiguous()
        feats_u_s = xs_feature.detach().contiguous()
        probs_orig, probs, mask = ops.bank_smooth(un_e_output.detach().contiguous(), feats_u_w, st.queue_feats,
                                                  st.queue_probs, args.alpha, T, smooth, adap_mask)      # :203-222
        probs_orig1, probs1, masks = ops.bank_smooth(un_b_output.detach().contiguous(), feats_u_s, st.queue_feats1,
                                                     st.queue_probs1, args.alpha, T, smooth, adap_mask)  # :209-228
        onehot = torch.zeros(bs, C, device=out_b.device).scatter_(1, Y_train.view(-1, 1), 1)             # :224
        qs = st.queue_feats.size(0)
        st.queue_feats[st.queue_ptr:st.queue_ptr + n] = torch.cat([feats_u_w, x_feature.detach()], 0)    # :232
        st.queue_probs[st.queue_ptr:st.queue_ptr + n] = torch.cat([probs_orig, onehot], 0)
        st.queue_ptr = (st.queue_ptr + 256) % qs                                                         # :234
        st.queue_feats1[st.queue_ptr1:st.queue_ptr1 + n] = torch.cat([feats_u_s, x_feature1.detach()], 0)
        st.queue_probs1[st.queue_ptr1:st.queue_ptr1 + n] = torch.cat([probs_orig1, onehot], 0)
        st.queue_ptr1 = (st.queue_ptr + 256) % qs                                                        # :237 (sic)
    con = losses.soft_cross_entropy(un_b_output, probs, mask)                    # :239,241
    con1 = losses.soft_cross_entropy(un_e_output, probs1, masks)                 # :240,242
    lc = losses.graph_contrast(xs_feature, xw_feature.detach(), probs1, probs, T, 0)      # :243-247,260-262
    lc1 = losses.graph_contrast(xs_feature.detach(), xw_feature, probs1, probs, T, 1)     # :244,257-258,263-265
    total = cls + 0.5 * lc + 4 * con                                             # :266
    total.backward()
    grads = {k: p.grad for k, p in st.Base.named_parameters()} if st.extras.get("keep_grads") else None
    st.opt.step()
    total1 = cls1 + 0.5 * lc1 + 4 * con1                                         # :270
    total1.backward()
    grads1 = {k: p.grad for k, p in st.Base1.named_parameters()} if st.extras.get("keep_grads") else None
    st.opt1.step()
    acc = (ops.argmax_u8(labeled_output1.detach().contiguous()).to(torch.int64) == Y_train).float().mean()   # :194,278
    hist = torch.stack([lc.detach(), total.detach(), cls.detach(), con.detach(), acc])
    return hist, {"logits": out_b.detach(), "logits1": out_e.detach(), "probs": probs, "probs1": probs1,
                  "mask": mask, "masks": masks, "total1": total1.detach(), "lc1": lc1.detach(),
                  "con1": con1.detach(), "cls1": cls1.detach(), "grads": grads, "grads1": grads1}


def noisy_batch(ds, positions, noise_scale, gen=None):
    """Gather a batch on device and add N(0,1)*noise (train.py:157-158): patch noise is fused into the
    gather kernel, spectral noise is one elementwise add."""
    n = positions.numel()
    dev = positions.device
    F, w = ds.cube.shape[2], ds.w
    z = torch.randn((n, F, w, w), device=dev, generator=gen) if noise_scale else None
    XP, X, Y = ds.gather(positions, noise=z, noise_scale=noise_scale)
    if noise_scale:
        X = X + torch.randn(X.shape, device=dev, generator=gen) * noise_scale
    return XP, X, Y


def main(args):
    dataID = int(args.dataID)
    name, num_classes, num_features = DATASETS[dataID]
    device = torch.device("cuda", torch.cuda.current_device())
    root = os.path.join(args.root, name) + "/"
    Yall = np.load(root + 'Y.npy').astype(np.int64) - 1
    test_array = np.load(root + 'test_array.npy')
    Y = Yall[test_array]
    labeled = HSIDataSet(dataID, 'label', max_iters=args.num_unlabel, root=root)                     # train.py:101-104
    unlabeled = HSIDataSet(dataID, 'unlabel', max_iters=args.num_unlabel, num_unlabel=args.num_unlabel, root=root)
    whole = HSIDataSet(dataID, 'wholeset', root=root)
    whole_loader = torch.utils.data.DataLoader(whole, batch_size=args.val_batch_size, shuffle=False)
    st = make_state(num_features, num_classes, args, device, w=labeled.w)
    lb, ub = args.labeled_batch_size, args.unlabeled_batch_size
    num_batches = min(math.ceil(len(labeled) / lb), math.ceil(len(unlabeled) / ub))                 # :134
    hist_dev = []
    fused = None
    if not getattr(args, "fp32_step", False) and labeled.scene_ready and labeled.w in (20, 11):
        # default: the whole step is cmlpl_train_step (gather + Philox noise inside the first kernel, tcgen05
        # convolutions, 15 launches replayed from a CUDA graph); --fp32_step keeps the fp32 reference path below
        from .fused_step import FusedMutualStep
        fused = FusedMutualStep(st.Base, st.Base1, bs=lb, btu=ub, lr=args.lr, temperature=args.temperature,
                                alpha=args.alpha, thr=args.thr, num_epochs=args.num_epochs, queue_batch=args.queue_batch,
                                noise=args.noise, dropout=args.dropout, seed=1088, use_graph=True)
        st.extras["fused"] = fused
        cube = whole.cube_device()
        spectra_all = torch.from_numpy(whole.X.astype(np.float32)).to(device)
        pix_l = torch.from_numpy(labeled.index).to(device)
        pix_u = torch.from_numpy(unlabeled.index).to(device)
        y_all = torch.from_numpy(Yall).to(device)
    for epoch in range(args.num_epochs):
        perm_l = torch.randperm(len(labeled), device=device)
        perm_u = torch.randperm(len(unlabeled), device=device)
        for batch_index in range(num_batches):
            pl = perm_l[batch_index * lb:(batch_index + 1) * lb]
            pu = perm_u[batch_index * ub:(batch_index + 1) * ub]
            if fused is not None:
                pl_pix = pix_l[pl]
                hist = fused.step(y_all[pl_pix], epoch, batch_index, cube=cube, pix=torch.cat([pl_pix, pix_u[pu]]),
                                  spectra=spectra_all)[:5].clone()
                hist_dev.append(hist)
                if (batch_index + 1) % args.print_per_batches == 0:
                    m = torch.stack(hist_dev[-args.print_per_batches:]).mean(0).tolist()
                    print('Epoch %d/%d:  %d/%d loss_contrast= %.2f total_loss = %.4f cls_loss = %.4f con_loss = %.4f acc = %.2f\n'
                          % (epoch + 1, args.num_epochs, batch_index + 1, num_batches, m[0], m[1], m[2], m[3], m[4] * 100))
                continue
            XP_l1, X_l1, Y_train = noisy_batch(labeled, pl, args.noise)          # :157-159
            XP_l2, X_l2, _ = noisy_batch(labeled, pl, args.noise)                # :163-164
            XP_u1, X_u1, _ = noisy_batch(unlabeled, pu, args.noise)              # :170-171
            XP_u2, X_u2, _ = noisy_batch(unlabeled, pu, args.noise)              # :181-182
            hist, _ = mutual_step(st, torch.cat([XP_l1, XP_u1], 0), torch.cat([X_l1, X_u1], 0),
                                  torch.cat([XP_l2, XP_u2], 0), torch.cat([X_l2, X_u2], 0), Y_train,
                                  epoch, batch_index, args)
            hist_dev.append(hist)
            if (batch_index + 1) % args.print_per_batches == 0:                  # :281-289, one sync per print
                m = torch.stack(hist_dev[-args.print_per_batches:]).mean(0).tolist()
                print('Epoch %d/%d:  %d/%d loss_contrast= %.2f total_loss = %.4f cls_loss = %.4f con_loss = %.4f acc = %.2f\n'
                      % (epoch + 1, args.num_epochs, batch_index + 1, num_batches, m[0], m[1], m[2], m[3], m[4] * 100))
    torch.cuda.synchronize()
    time1 = time.time()
    predict_label = test_whole(st.Base, whole_loader, print_per_batches=10)      # :291
    time2 = time.time()
    print('inference time ==', time2 - time1)
    predict_label1 = test_whole(st.Base1, whole_loader, print_per_batches=10)
    results = []
    for tag, pred in (("", predict_label), ("1", predict_label1)):
        OA, Kappa, producerA = CalAccuracy(pred[test_array], Y)                  # :296-299
        print('Result:\n OA%s=%.2f,Kappa=%.2f' % (tag, OA * 100, Kappa * 100))
        print('producerA%s:' % tag, producerA * 100)
        print('AA%s=%.2f' % (tag, np.mean(producerA) * 100))
        results.append((OA, Kappa, producerA))
    return {"loss_hist": torch.stack(hist_dev).cpu().numpy() if hist_dev else np.zeros((0, 5)),
            "predict_label": predict_label, "predict_label1": predict_label1, "results": results, "state": st}


def build_parser():
    parser = argparse.ArgumentParser()
    parser.add_argument('--dataID', type=str, default=1)
    parser.add_argument('--num_label', type=int, default=5)
    parser.add_argument('--save_path_prefix', type=str, default='./')
    parser.add_argument('--labeled_batch_size', type=int, default=128)
    parser.add_argument('--unlabeled_batch_size', type=int, default=128)
    parser.add_argument('--val_batch_size', type=int, default=512)
    parser.add_argument('--num_workers', type=int, default=1)
    parser.add_argument('--lr', type=float, default=5e-4)
    parser.add_argument('--num_epochs', type=int, default=20)
    parser.add_argument('--print_per_batches', type=int, default=10)
    parser.add_argument('--num_unlabel', type=int, default=10000)
    parser.add_argument('--thr', type=float, default=1, help='pseudo label threshold')
    parser.add_argument('--alpha', type=float, default=0.95)
    parser.add_argument('--queue-batch', type=float, default=17, help='number of batches stored in memory bank')
    parser.add_argument('--temperature', default=0.3, type=float, help='softmax temperature')
    parser.add_argument('--teacher_alpha', type=float, default=0.95)
    parser.add_argument('--dropout', type=float, default=0.8)
    parser.add_argument('--noise', type=float, default=0.5)
    parser.add_argument('--m', type=int, default=5, help='number of stochastic augmentations')
    parser.add_argument('--root', type=str, default='./dataset/')
    parser.add_argument('--fp32_step', action='store_true',
                        help='run the step through the fp32 reference-precision kernels instead of cmlpl_train_step')
    return parser


if __name__ == '__main__':
    seed_torch()
    main(build_parser().parse_args())
