#!/usr/bin/env python
"""Drop-in for the reference's inference.py (same positional arguments and options, inference.py:116-135):

    python inference.py <config.yaml> <sub_index> <checkpoint.pth.tar> [-epoch N] [-t TOPK] [-p PRINT_FREQ] [-b BATCH]

loads the yaml with the reference's DEFAULTS merge, builds the inference dataset (`.npy` feature streams + the
`deepfake_test_sub{sub_index}.txt` list), the meta-arch by name, loads `checkpoint['state_dict_ema']` (DataParallel
`module.` keys accepted) and writes `<ckpt dir>/<sub_index>/data_left*.json` exactly like inference_one_epoch does.
New: `-b` videos per model call (default 32; the reference is fixed to 1) and `--merge` to also write the challenge's
prediction.txt / prediction.json (generate_results.ipynb) for this shard. Every result file is formatted on the GPU from
the device records (libs/utils/result_writer.py), byte for byte what json.dump writes.
`--window SEC [--hop SEC]` (hop defaults to window / 2): recordings longer than SEC seconds run as overlapping windows at
the model's trained time scale, merged into one result per recording on the GPU (libs/modeling/windows.py); such runs
always go through inference_sharded, single-process and torchrun alike. The window is a user choice: no setting of it
has been validated for detection quality.

Multi-GPU: launched under torchrun, one process per GPU,

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 inference.py <cfg> <sub> <ckpt>

every rank takes a strided shard of the sub-list (libs/utils/sharding.py; the reference instead splits the list into 7
files for 7 separate processes, inference.py:116-124), streams it through the model on its own GPU, and the fixed-size
result records are all-gathered once over NCCL; rank 0 writes the same data_left.json a single process writes.
"""
import argparse
import glob
import os
import time

import torch

from audio_visual_deepfake_detection_b200.libs.core import load_config
from audio_visual_deepfake_detection_b200.libs.datasets import make_data_loader, make_inference_dataset
from audio_visual_deepfake_detection_b200.libs.modeling import make_meta_arch
from audio_visual_deepfake_detection_b200.libs.utils import fix_random_seed, merge_results
from audio_visual_deepfake_detection_b200.libs.utils.infer_utils import one_epoch_records, sharded_records
from audio_visual_deepfake_detection_b200.libs.utils.result_writer import write_predictions


def main(args):
    if not os.path.isfile(args.config):
        raise ValueError("Config file does not exist.")
    cfg = load_config(args.config)
    assert len(cfg["test_split"]) > 0, "Test set must be specified!"
    if not os.path.isfile(args.ckpt):
        raise ValueError("CKPT file does not exist!")
    if args.topk > 0:
        cfg["model"]["test_cfg"]["max_seg_num"] = args.topk
    fix_random_seed(0, include_cuda=True)
    dataset = make_inference_dataset(cfg["dataset_name"], False, cfg["test_split"], args.sub_index, **cfg["dataset"])
    loader = make_data_loader(dataset, False, None, args.batch, cfg["loader"]["num_workers"])
    model = make_meta_arch(cfg["model_name"], **cfg["model"], max_batch=args.batch)
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        device = torch.device("cuda", local)             # one process per GPU: the yaml's `devices` names one GPU only
        torch.cuda.set_device(device)
        dist.init_process_group("nccl", device_id=device)
    else:
        device = torch.device(cfg["devices"][0] if torch.cuda.is_available() else "cpu")
    checkpoint = torch.load(args.ckpt, map_location="cpu")
    model.load_state_dict(checkpoint["state_dict_ema"])
    del checkpoint
    model.to(device).eval()
    out_dir = os.path.join(os.path.dirname(args.ckpt), str(args.sub_index))
    start = time.time()
    if world > 1 or args.window is not None:
        res = sharded_records(dataset, model, out_dir, batch_size=args.batch, rank=rank, world=world, print_freq=args.print_freq,
                              window=args.window, hop=args.hop)
        files = [] if res is None else [("data_left.json",) + res]
    else:
        written, _ = one_epoch_records(loader, model, out_dir)
        files = [(name, ids, rec, None, K) for name, ids, rec, K in written]
    if rank == 0:
        print("All done! Total time: {:0.2f} sec".format(time.time() - start))
        if args.merge:
            write_merged(out_dir, files)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def write_merged(out_dir, files):
    """prediction.txt / prediction.json of this shard. When the folder's result files (those merge_results reads) are
    exactly the files this run wrote, they are written on the GPU from the records in hand, in merge_results' file order;
    otherwise (files of an earlier run in the folder) merge_results reads the folder as before."""
    names = sorted(os.path.basename(p) for p in glob.glob(os.path.join(out_dir, "*.json"))
                   if not os.path.basename(p).startswith("prediction"))
    if not files or names != sorted(f[0] for f in files):
        merge_results([out_dir], out_dir)
        return
    files = sorted(files, key=lambda f: f[0])
    K = max(f[4] for f in files)
    ids, recs, orders, base = [], [], [], 0
    for name, f_ids, rec, order, k in files:
        if k != K:                       # widen to the common K: segments move to their K-strided place
            wide = torch.zeros((rec.shape[0], 3 + 3 * K), dtype=rec.dtype, device=rec.device)
            wide[:, :3 + k] = rec[:, :3 + k]
            wide[:, 3 + K:3 + K + 2 * k] = rec[:, 3 + k:]
            rec = wide
        ids += f_ids
        orders.append((torch.arange(len(f_ids), device=rec.device, dtype=torch.int32) if order is None else order) + base)
        recs.append(rec)
        base += rec.shape[0]
    write_predictions(out_dir, ids, torch.cat(recs), K, order=torch.cat(orders))


if __name__ == "__main__":
    parser = argparse.ArgumentParser(description="Localization inference on the B200 path")
    parser.add_argument("config", type=str, metavar="DIR", help="path to a config file")
    parser.add_argument("sub_index", type=int, help="sub test index (deepfake_test_sub{N}.txt)")
    parser.add_argument("ckpt", type=str, metavar="DIR", help="path to a checkpoint")
    parser.add_argument("-epoch", type=int, default=-1, help="checkpoint epoch (kept for CLI compatibility)")
    parser.add_argument("-t", "--topk", default=-1, type=int, help="max number of output segments (default: -1)")
    parser.add_argument("-p", "--print-freq", default=10, type=int, help="print frequency")
    parser.add_argument("-b", "--batch", default=32, type=int, help="videos per model call")
    parser.add_argument("--merge", action="store_true", help="also write prediction.txt / prediction.json for this shard")
    parser.add_argument("--window", type=float, default=None, help="sliding window (seconds) for recordings longer than it")
    parser.add_argument("--hop", type=float, default=None, help="hop between windows (seconds, default: window / 2)")
    main(parser.parse_args())
