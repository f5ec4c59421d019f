"""Drop-in for the reference's training script (SURVEY 8(f) N2 + N3).

``python -m npi_gnn_b200.train_shell --trainingName T --trainingDatasetName A --testingDatasetName B
--fold 0 ...`` accepts the flags of src/train_with_twoDataset.PY:26-43 and leaves the same artefacts:

    result/<trainingName>/log_<fold>.txt                 header, 'Epoch: NNN, training|testing dataset, ...'
                                                         every 5th epoch (not the last), 'result, ...' lines,
                                                         the best-MCC summary and the run time     (:100-222)
    result/<trainingName>/model_<fold>_fold/<epoch>      torch.save(model.state_dict()) at the same cadence (:193-194,213-214)

What runs underneath is this package: the training epochs are ``Trainer`` steps (GPU extraction,
fused forward/backward/Adam replayed from CUDA graphs), the learning rate follows the reference's
rule -- multiply by 0.95 whenever the epoch loss rose (:157-160) -- and the evaluation sweeps are
batched eval-mode forwards with the confusion matrix counted on the GPU (``Scorer.confusion``,
replacing the per-sample loop of src/methods.py:87-127; same TP/FN/TN/FP, same five metrics).
Datasets that only exist as precomputed subgraphs (a PyG ``processed/data.pt``) go through the
module-level route instead: ``Net_1`` + ``torch.optim.Adam`` exactly as the reference's ``train()``.

Differences by design: paths are joined with os.path (the reference hard-codes ``.\\\\data\\\\dataset``
Windows separators, :64-65); ``--seed`` (not in the reference) makes the two ``dataset.shuffle()``
calls (:76-77), the parameter initialisation and dropout reproducible; ``--gpus`` is implied by torchrun.
``--rankMetrics 1`` (not in the reference) adds one line after every testing-dataset metric line:
'<same prefix>, AUROC: x.xxxxx, AP: x.xxxxx, PR-AUC(trapz): x.xxxxx' -- the ROC AUC and PR summaries of
src/compare_withKmer_noKmer.py, from the same sweep (``Scorer.rank_metrics``); with 0 the artefacts are unchanged.
"""
from __future__ import annotations

import argparse
import os
import time

import torch

from . import _lib as L
from .trainer import Scorer, Trainer, metrics, rank_metrics

EVAL_EVERY = 5          # src/train_with_twoDataset.PY:163
GAMMA = 0.95            # ExponentialLR(gamma=0.95) stepped only when the loss rose (:135,158-159)


def build_parser():
    """The reference's flags with its defaults (src/train_with_twoDataset.PY:26-43) + --seed/--dataRoot/--resultRoot/--rankMetrics."""
    p = argparse.ArgumentParser(description="train Net_1 on two enclosing-subgraph datasets")
    p.add_argument("--trainingName", help="the name of this training")
    p.add_argument("--trainingDatasetName", help="the name of this object")
    p.add_argument("--testingDatasetName", help="the name of this object")
    p.add_argument("--inMemory", default=1, type=int, help="in memory dataset or not")
    p.add_argument("--interactionDatasetName", default="NPInter2", help="raw interactions dataset")
    p.add_argument("--fold", type=int, help="this is part of cross validation, the ith fold")
    p.add_argument("--epochNumber", default=50, type=int, help="number of training epoch")
    p.add_argument("--hopNumber", default=1, type=int, help="hop number of subgraph")
    p.add_argument("--node2vecWindowSize", default=5, type=int, help="node2vec window size")
    p.add_argument("--initialLearningRate", default=0.001, type=float, help="Initial learning rate")
    p.add_argument("--l2WeightDecay", default=0.001, type=float, help="L2 weight")
    p.add_argument("--batchSize", default=200, type=int, help="batch size")
    p.add_argument("--seed", default=None, type=int, help="(extension) seed for shuffle / init / dropout")
    p.add_argument("--dataRoot", default=os.path.join("data", "dataset"), help="(extension) where the datasets live")
    p.add_argument("--resultRoot", default="result", help="(extension) where logs and checkpoints go")
    p.add_argument("--rankMetrics", default=0, type=int,
                   help="(extension) 1: log AUROC, AP and trapezoidal PR AUC after every testing-dataset metric line")
    return p


def parse_args(argv=None):
    return build_parser().parse_args(argv)


def metric_line(prefix, m):
    """'<prefix>, Accuracy: ..., MCC: ...' with the reference's 5-decimal formatting (:168,172,199,203)."""
    return "{}, Accuracy: {:.5f}, Precision: {:.5f}, Sensitivity: {:.5f}, Specificity: {:.5f}, MCC: {:.5f}".format(prefix, *m)


def rank_line(prefix, r):
    """'<prefix>, AUROC: ..., AP: ..., PR-AUC(trapz): ...' (--rankMetrics 1) from a ``rank_metrics`` dict."""
    return "{}, AUROC: {:.5f}, AP: {:.5f}, PR-AUC(trapz): {:.5f}".format(prefix, r["auroc"], r["ap"], r["pr_auc_trapz"])


def should_evaluate(epoch1, num_epochs):
    """Intermediate evaluation + checkpoint after epoch ``epoch1`` (1-based)?  (:163)"""
    return epoch1 % EVAL_EVERY == 0 and epoch1 != num_epochs


class LrOnLossIncrease:
    """lr <- lr * gamma after every epoch whose loss exceeded the previous epoch's (:155-160)."""

    def __init__(self, lr, gamma=GAMMA):
        self.lr, self.gamma, self.last = float(lr), float(gamma), float("inf")

    def update(self, loss):
        if loss > self.last:
            self.lr *= self.gamma
        self.last = loss
        return self.lr


class BestByMcc:
    """Tracks the testing-set metrics at the highest MCC seen (:144-149,174-181,205-211)."""

    def __init__(self):
        self.mcc, self.epoch, self.acc, self.pre, self.sen, self.spe = -1, 0, 0, 0, 0, 0

    def offer(self, epoch1, m):
        acc, pre, sen, spe, mcc = m
        if mcc > self.mcc:
            self.mcc, self.epoch, self.acc, self.pre, self.sen, self.spe = mcc, epoch1, acc, pre, sen, spe

    def line(self):
        return "epoch: {}, MCC: {}, ACC: {}, Pre: {}, Sen: {}, Spe: {}".format(self.epoch, self.mcc, self.acc, self.pre,
                                                                              self.sen, self.spe)


class RunLog:
    """log_<fold>.txt writer: the header of :102-112 and one line per event, echoed to stdout."""

    def __init__(self, path, echo=True):
        self.f = open(path, mode="w")
        self.echo = echo

    def header(self, args, lr, wd):
        w = self.f.write
        w("training dataset : {}".format(args.trainingDatasetName))
        w("testing dataset : {}".format(args.testingDatasetName))
        w("database：{}\n".format(args.interactionDatasetName))
        w("node2vec_windowSize = {}\n".format(args.node2vecWindowSize))
        w("number of eopch ：{}\n".format(args.epochNumber))
        w("learn rate：initial = {}，whenever loss increases, multiply by 0.95\n".format(lr))
        w("L2 weight decay = {}\n".format(wd))

    def line(self, text):
        if self.echo:
            print(text)
        self.f.write(text + "\n")

    def close(self):
        self.f.close()


# ---------------------------------------------------------------------------------------------
class _FusedBackend:
    """Pair-set datasets: Trainer (fused step, CUDA graph) + Scorer (GPU confusion counts)."""

    def __init__(self, train_ds, test_ds, args, seed):
        self.tr = Trainer(train_ds.pairset, batch_size=args.batchSize, lr=args.initialLearningRate,
                          weight_decay=args.l2WeightDecay, seed=seed, order=train_ds._index)
        self.train_ds, self.test_ds, self.B = train_ds, test_ds, args.batchSize
        self._scorers = {}

    def train_epoch(self):
        return self.tr.train_epoch()

    def set_lr(self, lr):
        self.tr.set_lr(lr)

    def _scorer(self, which):
        ds = self.train_ds if which == "train" else self.test_ds
        if which not in self._scorers:
            self._scorers[which] = Scorer(ds.pairset, self.tr.params, batch_size=self.B, index=ds._index)
        return self._scorers[which]

    def evaluate(self, which):
        return metrics(*self._scorer(which).confusion())

    def evaluate_ranked(self, which):
        """(metrics, rank_metrics dict) from one sweep of the dataset."""
        r = self._scorer(which).rank_metrics()
        return metrics(*r["confusion"]), r

    def state_dict(self):
        return {k: v.cpu() for k, v in self.tr.params.state_dict().items()}


class _ModuleBackend:
    """Precomputed-subgraph datasets: the reference's own loop shape over the drop-in modules
    (src/train_with_twoDataset.PY:46-57 and src/methods.py:87-127, batched)."""

    def __init__(self, train_ds, test_ds, args, seed):
        from .data import DataLoader
        from .nn import Net_1
        import torch.nn.functional as F
        self.F = F
        self.model = Net_1(train_ds.num_node_features, 2).to("cuda")
        self.opt = torch.optim.Adam(self.model.parameters(), lr=args.initialLearningRate, weight_decay=args.l2WeightDecay)
        self.loaders = {"train": DataLoader(train_ds, batch_size=args.batchSize), "test": DataLoader(test_ds, batch_size=args.batchSize)}
        self.n_train = len(train_ds)

    def train_epoch(self):
        self.model.train()
        loss_all = 0.0
        for data in self.loaders["train"]:
            data = data.to("cuda")
            self.opt.zero_grad()
            loss = self.F.nll_loss(self.model(data), data.y)
            loss.backward()
            loss_all += data.num_graphs * loss.item()
            self.opt.step()
        return loss_all / max(self.n_train, 1)

    def set_lr(self, lr):
        for g in self.opt.param_groups:
            g["lr"] = lr

    def evaluate(self, which):
        return self.evaluate_ranked(which, rank=False)[0]

    def evaluate_ranked(self, which, rank=True):
        from . import ops
        self.model.eval()
        counts = torch.zeros(4, dtype=torch.int64, device="cuda")
        scores, labels = [], []
        with torch.no_grad():
            for data in self.loaders[which]:
                data = data.to("cuda")
                logp = self.model(data).contiguous()
                ops.confusion_counts(logp, data.y.to(torch.int32), data.num_graphs, -1.0, counts)
                if rank:
                    scores.append(torch.exp(logp[:, 1]))
                    labels.append(data.y.to(torch.int32))
        TP, FN, TN, FP = [int(v) for v in counts.cpu()]
        r = rank_metrics(torch.cat(scores), torch.cat(labels)) if rank else None
        return metrics(TP, FN, TN, FP), r

    def state_dict(self):
        return {k: v.detach().cpu() for k, v in self.model.state_dict().items()}


def run(args, train_dataset=None, test_dataset=None, echo=True):
    """The body of the reference script (:60-222).  Datasets may be passed in (tests, notebooks);
    otherwise they are reloaded from ``<dataRoot>/<name>`` like :72-73.  Returns a summary dict."""
    from .data import LncRNA_Protein_Interaction_dataset_1hop_1220_InMemory as DS
    if not torch.cuda.is_available():
        raise L.NPIError("training needs a CUDA device (there is no CPU fallback)")
    if args.inMemory != 1:
        if args.inMemory == 0:
            raise Exception("not ready yet")
        raise Exception("--inMemory has to be 0 or 1")
    if args.seed is not None:
        torch.manual_seed(args.seed)
    if train_dataset is None:
        train_dataset = DS(root=os.path.join(args.dataRoot, args.trainingDatasetName))
    if test_dataset is None:
        test_dataset = DS(root=os.path.join(args.dataRoot, args.testingDatasetName))
    if echo:
        print("shuffle dataset\n")
    train_dataset, test_dataset = train_dataset.shuffle(), test_dataset.shuffle()
    saving_path = os.path.join(args.resultRoot, str(args.trainingName))
    os.makedirs(saving_path, exist_ok=True)
    num_epochs, lr0, wd = args.epochNumber, args.initialLearningRate, args.l2WeightDecay
    model_dir = os.path.join(saving_path, "model_{}_fold".format(args.fold))
    if os.path.exists(model_dir):
        raise Exception("Same fold has been done")
    log = RunLog(os.path.join(saving_path, "log_{}.txt".format(args.fold)), echo=echo)
    log.header(args, lr0, wd)
    start = time.time()
    os.makedirs(model_dir)
    if train_dataset.num_node_features != test_dataset.num_node_features:
        raise Exception("training and testing datasets have different node feature widths")
    if echo:
        print("number of samples in testing dataset：", len(test_dataset), "number of samples in training dataset：", len(train_dataset))
    fused = train_dataset._foreign is None and test_dataset._foreign is None
    seed = args.seed if args.seed is not None else int(torch.initial_seed() & 0x7FFFFFFF)
    be = (_FusedBackend if fused else _ModuleBackend)(train_dataset, test_dataset, args, seed)

    def evaluate_test(prefix):
        """The testing-dataset metric line (+ the rank line under --rankMetrics 1, same sweep); returns the metrics."""
        if not args.rankMetrics:
            m = be.evaluate("test")
            log.line(metric_line(prefix, m))
            return m
        m, r = be.evaluate_ranked("test")
        log.line(metric_line(prefix, m))
        log.line(rank_line(prefix, r))
        return m

    sched, best, losses = LrOnLossIncrease(lr0), BestByMcc(), []
    for epoch in range(num_epochs):
        loss = be.train_epoch()
        losses.append(loss)
        lr = sched.update(loss)
        be.set_lr(lr)
        if should_evaluate(epoch + 1, num_epochs):
            m = be.evaluate("train")
            log.line(metric_line("Epoch: {:03d}, training dataset".format(epoch + 1), m))
            m = evaluate_test("Epoch: {:03d}, testing dataset".format(epoch + 1))
            best.offer(epoch + 1, m)
            torch.save(be.state_dict(), os.path.join(model_dir, str(epoch + 1)))
    m_train = be.evaluate("train")
    log.line(metric_line("result, training dataset", m_train))
    m_test = evaluate_test("result, testing dataset")
    best.offer(num_epochs, m_test)
    torch.save(be.state_dict(), os.path.join(model_dir, str(num_epochs)))
    log.f.write("\n")
    log.line("MCC最大的时候的性能：")
    log.line(best.line())
    elapsed = time.time() - start
    if echo:
        print("Time consuming:", elapsed)
    log.f.write("Time consuming:" + str(elapsed) + "\n")
    log.close()
    return dict(losses=losses, final_train=m_train, final_test=m_test, best_epoch=best.epoch, best_mcc=best.mcc,
                lr=sched.lr, log=os.path.join(saving_path, "log_{}.txt".format(args.fold)), model_dir=model_dir,
                backend="fused" if fused else "module", seconds=elapsed)


def main(argv=None):
    run(parse_args(argv))
    print("\nexit\n")


if __name__ == "__main__":
    main()
