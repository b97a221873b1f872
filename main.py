#!/usr/bin/env python
"""Training / evaluation driver with the reference's flag surface (reference main.py:42-86) and call protocol
(main.py:94-251): partition -> model -> sampler -> epochs of `num_batch` steps -> every 20 epochs checkpoint +
evaluate(test) + evaluate_valid, writing the same `params.txt` / `log.txt` files under
`saved_models/<dataset>/<train_dir>_<timestamp>/`.  The TF session is gone: a step is `model.train_step(...)`
(hand-written sm_100a kernels through the C ABI).

    python main.py --dataset data/ml-1m.txt --train_dir run1 --model sasrec --maxlen 200 --dropout_rate 0.2
    python -m torch.distributed.run --nproc-per-node 8 main.py ...        # data parallel, one process per GPU

New flags have new names (`--eval_mode`, `--eval_every`, `--eval_batch`); every reference flag keeps its name,
default and quirks (`--max_norm` takes effect only with the new `--clip_grad`, `--log_scale` / `--input_context` are `type=bool`, `--seed 0` = unseeded,
`num_batch = round(len(train) / batch_size)`).
"""
from __future__ import annotations

import argparse
import json
import logging
import os
import random
import sys
import time
from datetime import datetime

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODELS = ["cast_1", "cast_2", "cast_3", "cast_4", "cast_5", "cast_6", "cast_7", "cast_8", "cast_9", "sasrec",
          "sasrec_static"]


def build_parser():
    p = argparse.ArgumentParser()
    p.add_argument("--dataset", required=True, help="Location of pre-processed dataset")
    p.add_argument("--maxlen", default=50, type=int, help="Maximum length of user item sequence, for zero-padding")
    p.add_argument("--train_dir", required=True)
    p.add_argument("--batch_size", default=128, type=int, help="Batch size")
    p.add_argument("--lr", type=float, default=1e-3, help="Learning rate")
    p.add_argument("--num_epochs", type=int, default=201, help="Number of epochs")
    p.add_argument("--max_norm", type=float, default=5.0,
                   help="global gradient norm threshold; takes effect only with --clip_grad (unused by the reference)")
    p.add_argument("--hidden_units", default=50, type=int)
    p.add_argument("--num_blocks", default=2, type=int)
    p.add_argument("--num_heads", default=1, type=int)
    p.add_argument("--dropout_rate", default=0.5, type=float)
    p.add_argument("--l2_emb", default=0.0, type=float)
    p.add_argument("--bin_in_hours", default=24, type=int)
    p.add_argument("--max_bins", default=200, type=int)
    p.add_argument("--num_context_blocks", default=2, type=int)
    p.add_argument("--test_model", type=str, default=None, help="Test the specified model with saved parameters")
    p.add_argument("--test_seq_len", type=int, default=None,
                   help="Test the specified model with another sequence length")
    p.add_argument("--saved_model", default="model.pt", type=str, help="(unused, as in the reference)")
    p.add_argument("--seed", default=42, type=int)
    p.add_argument("--log_scale", type=bool, default=False)
    p.add_argument("--input_context", type=bool, default=False)
    p.add_argument("--model", default="cast_1", required=True, help="model to use from" + str(MODELS))
    # additions (new names only)
    p.add_argument("--eval_mode", default="101", choices=["101", "full"],
                   help="101 = the reference's target + 100 sampled negatives; full = rank against the whole catalog")
    p.add_argument("--eval_every", default=20, type=int, help="epochs between checkpoint + evaluation (reference: 20)")
    p.add_argument("--eval_batch", default=256, type=int, help="users scored per device batch")
    p.add_argument("--model_path", default=os.path.abspath("saved_models"))
    p.add_argument("--device_time_features", action="store_true", help="CAST models: the sampler and the evaluation "
                   "hand raw timestamps to the device, which derives time bins / hours / weekdays there")
    p.add_argument("--recommend", default=0, type=int, help="with --test_model: after the evaluation, write the top K "
                   "items of every user (whole history excluded) to recommendations_top{K}.npz next to the checkpoint")
    p.add_argument("--similar_items", default=0, type=int, help="with --test_model: after the evaluation, write the "
                   "top K most similar items of every item to similar_items_top{K}.npz next to the checkpoint")
    p.add_argument("--similarity", default="cosine", choices=["cosine", "dot"],
                   help="item-to-item score of --similar_items: cosine of the item_emb rows, or their dot product")
    p.add_argument("--item_bias", default=None, help="with --recommend / --similar_items: a .npy of itemnum + 1 "
                   "reals (entry 0 ignored) added to every score of item j (-inf removes item j: deny / allow lists; "
                   "e.g. -a*log(1+count) corrects for popularity); NaN or +inf is rejected")
    p.add_argument("--optimizer", default="adam", choices=["adam", "lazy_adam"],
                   help="adam = the reference's dense TF-Adam; lazy_adam = LazyAdam on the item table (only the rows a "
                   "batch touches are updated; step cost no longer grows with the catalog), dense TF-Adam elsewhere")
    p.add_argument("--clip_grad", action="store_true", help="clip the gradient to global norm --max_norm before Adam "
                   "(tf.clip_by_global_norm); the epoch log line then also reports TRAIN/grad_norm of its last step")
    return p


def load_item_bias(args, itemnum):
    """--item_bias FILE.npy -> validated float32 tensor (None without the flag); raises ValueError on a wrong shape, a
    non-real dtype, NaN or +inf"""
    if not getattr(args, "item_bias", None):
        return None
    from cast_b200.models import check_item_bias
    return check_item_bias(np.load(args.item_bias), itemnum)


def write_recommendations(model, dataset, args, rank, world):
    """--recommend K: exact top-K of every user from the last maxlen events of train + valid + test, the whole history
    excluded; users are sharded over the ranks and gathered; rank 0 writes users / items / scores."""
    from cast_b200 import dist as cdist
    from cast_b200.evaluation import build_recommend_inputs, recommend_users
    K = int(args.recommend)
    rec = build_recommend_inputs(dataset, args)
    lo, hi = cdist.shard_users(len(rec["u"]), rank, world)
    ids, scores = recommend_users(model, rec, K, args.eval_batch, lo, hi,
                                  item_bias=load_item_bias(args, model.itemnum))
    if world > 1:
        import torch.distributed as tdist
        parts = [None] * world
        tdist.all_gather_object(parts, (ids, scores))
        ids = np.concatenate([p[0] for p in parts])
        scores = np.concatenate([p[1] for p in parts])
    if rank == 0:
        np.savez(os.path.join(args.test_model, "recommendations_top{}.npz".format(K)), users=rec["u"], items=ids,
                 scores=scores)


def write_similar_items(model, args, rank, world):
    """--similar_items K: exact top-K neighbours (--similarity) of every item; the items are sharded over the ranks and
    gathered; rank 0 writes items / neighbours / scores."""
    from cast_b200 import dist as cdist
    from cast_b200.evaluation import similar_items_all
    K = int(args.similar_items)
    lo, hi = cdist.shard_users(model.itemnum, rank, world)
    items, nbr, scores = similar_items_all(model, K, args.eval_batch, lo, hi, args.similarity,
                                           item_bias=load_item_bias(args, model.itemnum))
    if world > 1:
        import torch.distributed as tdist
        parts = [None] * world
        tdist.all_gather_object(parts, (items, nbr, scores))
        items, nbr, scores = (np.concatenate([p[j] for p in parts]) for j in range(3))
    if rank == 0:
        np.savez(os.path.join(args.test_model, "similar_items_top{}.npz".format(K)), items=items, neighbours=nbr,
                 scores=scores)


def save_checkpoint(model, args, path):
    """reference main.py:226-228 `saver.save(sess, save_path)`: a TensorFlow tensor bundle with the reference's
    variable names, Adam slots, beta powers and global_step (models whose TF scopes are pinned by a shipped checkpoint:
    checkpoint.CKPT_MODELS); the role-named .npz next to it covers every model."""
    from cast_b200 import checkpoint as ck
    if args.model.lower() in ck.CKPT_MODELS:
        ck.save_model(path, model, args.model.lower(), args.num_blocks)
    eng = model.engine
    np.savez(path + ".npz", **{k: v.numpy() for k, v in model.state_dict().items()},
             **{"__adam_m": eng.m.cpu().numpy(), "__adam_v": eng.v.cpu().numpy(),
                "__adam_state": eng.adam_state.cpu().numpy()})
    return path


def load_checkpoint(model, args, directory):
    """reference main.py:153-159 `saver.restore`: reads a bundle written by the reference itself or by this driver"""
    import torch
    from cast_b200 import checkpoint as ck
    prefix = os.path.join(directory, "model.ckpt")
    if os.path.isfile(prefix + ".index") and args.model.lower() in ck.CKPT_MODELS:
        ck.restore_model(prefix, model, args.model.lower(), args.num_blocks)
        return
    g = np.load(prefix + ".npz")
    model.load_state_dict({k: g[k] for k in g.files if not k.startswith("__")})
    if "__adam_m" in g.files:
        eng = model.engine
        eng.m.copy_(torch.from_numpy(g["__adam_m"]).to(eng.device))
        eng.v.copy_(torch.from_numpy(g["__adam_v"]).to(eng.device))
        eng.adam_state.copy_(torch.from_numpy(g["__adam_state"]).to(eng.device))


def run(args, device=None, lib=None, logger=None):
    import cast_b200
    from cast_b200 import dist as cdist
    from cast_b200.data import data_partition
    from cast_b200.evaluation import evaluate, evaluate_valid
    from cast_b200.sampler import WarpSampler

    logger = logger or logging.getLogger("ir2")
    if args.model.lower() not in MODELS:
        print("provide model from", MODELS)
        return 0
    if not os.path.exists(args.dataset):
        logger.info("Pre-process the data first using the --preprocess flag")
        return 0
    rank, world, local = cdist.init_from_env() if device is None else (0, 1, 0)
    dataset = data_partition(args.dataset, args.log_scale)
    train, valid, test, usernum, itemnum, ratingnum = dataset
    load_item_bias(args, itemnum)    # a bad --item_bias fails here, before any training or evaluation
    num_batch = round(len(train) / args.batch_size)
    print("usernum", usernum, "itemnum", itemnum)
    cc = sum(len(v) for v in train.values())
    logger.info("Average sequence length: {:.2f}".format(cc / len(train)))
    seed = int(args.seed or 0)
    if world > 1:   # one seed for the whole job (--seed 0 = "unseeded": drawn once, on rank 0)
        import torch
        import torch.distributed as tdist
        box = [seed if seed else int(np.random.SeedSequence().generate_state(1)[0] % (2 ** 31 - 1)) + 1]
        tdist.broadcast_object_list(box, src=0)
        seed = box[0]
    if seed:        # evaluation draws its user sample and negatives from these (util.py:241-244,295): same on every rank
        random.seed(seed)
        np.random.seed(seed)
    kw = {} if device is None else {"device": device, "_lib": lib, "use_graph": False}
    model = cast_b200.build_model(args.model, usernum, itemnum, ratingnum, args, **kw)
    if device is None:
        cdist.attach(model.engine)
    # every rank draws its own batches from its own stream (seed, rank): nothing is generated to be thrown away
    sargs = args
    if world > 1:
        from types import SimpleNamespace
        sargs = SimpleNamespace(**{**vars(args), "seed": seed + 7919 * rank})
    raw_ts = bool(getattr(args, "device_time_features", False)) and len(model.engine.plan.tables) > 1
    if raw_ts:
        from cast_b200.data import get_delta_range
        lo_td, hi_td = get_delta_range(train)
        model.use_device_time_features(args.bin_in_hours, args.max_bins, args.log_scale, lo_td, hi_td)
    sampler = WarpSampler(sargs, train, usernum, itemnum, batch_size=args.batch_size, maxlen=args.maxlen, n_workers=1,
                          raw_timestamps=raw_ts)

    def train_on(batch, sync=True):
        u, seq, pos, neg, timeseq, _, hours_seq, days_seq, last = batch
        if raw_ts:      # ninth slot = raw int64 event times
            return model.train_step(u, seq, pos, neg, timestamps=last, sync=sync)
        return model.train_step(u, seq, pos, neg, timeseq, hours_seq, days_seq, sync=sync)
    now = datetime.now()
    files_path = os.path.join(args.model_path, os.path.basename(args.dataset),
                              "{}_{}".format(args.train_dir, now.strftime("%m-%d-%Y-%H-%M-%S")))
    save_path = os.path.join(files_path, "model.ckpt")

    next_batch = sampler.next_batch

    if args.test_model:
        try:
            if os.path.exists(args.test_model):
                print("loaded saved model {}".format(args.test_model))
                load_checkpoint(model, args, args.test_model)
                auc, loss = train_on(next_batch())  # as main.py:167-175
                print(auc)
                print(loss)
                # as util.py:329-336: the attention map averaged over the evaluated users goes next to the checkpoint
                # (the reference renders attention_weights.svg; the array is stored instead)
                t_test, avg_attn = evaluate(model, dataset, args, None, batch_users=args.eval_batch,
                                            avg_attention=True)
                logger.info("test (NDCG@10: %.4f, HR@10: %.4f)" % (t_test[0], t_test[1]))
                if rank == 0:
                    np.save(os.path.join(args.test_model, "avg_attention_weights.npy"), avg_attn)
                    with open(os.path.join(args.test_model, "test_seq_len.txt"), "a") as f:
                        f.write("{},{},{}\n".format(args.test_seq_len, t_test[0], t_test[1]))
                if getattr(args, "recommend", 0) > 0:
                    write_recommendations(model, dataset, args, rank, world)
                if getattr(args, "similar_items", 0) > 0:
                    write_similar_items(model, args, rank, world)
            else:
                print("{} not found".format(args.test_model))
        finally:
            sampler.close()
        return 0

    if rank == 0:
        os.makedirs(files_path, exist_ok=True)
        with open(os.path.join(files_path, "params.txt"), "w") as f:
            json.dump(args.__dict__, f, indent=2)
    log = open(os.path.join(files_path, "log.txt"), "w") if rank == 0 else None
    args.train_files_path = files_path
    T = 0.0
    t0 = time.time()
    rc = 0
    try:
        for epoch in range(1, args.num_epochs + 1):
            auc = loss = None
            for _ in range(num_batch):   # the epoch's last (auc, loss) is what gets logged: nothing waits in between
                train_on(next_batch(), sync=False)
            if num_batch > 0:
                auc, loss = model.last_metrics()
            if auc is not None:
                line = "epoch:%d TRAIN/loss %.6f TRAIN/auc %.6f" % (epoch, loss, auc)
                if getattr(args, "clip_grad", False):
                    line += " TRAIN/grad_norm %.6f" % model.last_grad_norm()
                logger.info(line)
            if epoch % args.eval_every == 0:
                if rank == 0:
                    logger.info("Model saved in path: %s" % save_checkpoint(model, args, save_path))
                logger.info("Evaluating")
                T += time.time() - t0
                t_test = evaluate(model, dataset, args, None, batch_users=args.eval_batch, mode=args.eval_mode)
                t_valid = evaluate_valid(model, dataset, args, None, batch_users=args.eval_batch, mode=args.eval_mode)
                logger.info("")
                logger.info("epoch:%d, time: %f(s), valid (NDCG@10: %.4f, HR@10: %.4f), test (NDCG@10: %.4f, "
                            "HR@10: %.4f)" % (epoch, T, t_valid[0], t_valid[1], t_test[0], t_test[1]))
                if log:
                    # the reference's line format (main.py:238): plain Python floats, not numpy reprs
                    log.write(str(tuple(float(x) for x in t_valid)) + " " + str(tuple(float(x) for x in t_test)) + "\n")
                    log.flush()
                t0 = time.time()
    except Exception as e:  # as the reference: close the sampler and the log, report, exit code 1
        logger.error(e)
        rc = 1
        if world > 1:       # the other ranks are blocked in this step's exchange: fail the whole job fast
            sampler.close()
            if log:
                log.close()
            os._exit(1)
    finally:
        sampler.close()
        if log:
            log.close()
    if world > 1:
        import torch.distributed as tdist
        if tdist.is_initialized():
            cdist.quiesce(model.engine)      # no rank leaves while a peer's last optimizer pass reads its gradients
            tdist.destroy_process_group()
    if rc == 0:
        print("Done")
    return rc


if __name__ == "__main__":
    logging.basicConfig(level=logging.DEBUG,
                        format="%(asctime)s [%(threadName)-12.12s] [%(levelname)-5.5s]  %(message)s",
                        handlers=[logging.FileHandler("./output.log"), logging.StreamHandler()])
    sys.exit(run(build_parser().parse_args()))
