"""Golden batches of the reference's training loader (build container only; writes loader_ml100k.npz).

Runs the UNMODIFIED reference pipeline -- Config / create_dataset / data_preparation on the bundled
ml-100k KG, KnowledgeBasedDataLoader in RSKG mode (what KGTrainer._train_epoch selects,
trainer.py:647-666) -- for two epochs with seed 2024 and freezes:
  * the arrays the loader draws from (train interactions, KG triples) and the table sizes,
  * numpy's MT19937 state right before the first batch (the samplers' stream),
  * a CRC32 of every id vector of every step, and the full id vectors of a few steps.
tests/test_loader_cpu.py and tests/test_gpu_loader.py rebuild the batches from these without hopwise.

    cd /tmp && python /root/repo/tests/golden/make_golden_loader.py
"""
import os
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from _ref_harness import import_reference  # noqa: E402

KEYS = ("user_id", "item_id", "neg_item_id", "head_id", "relation_id", "tail_id", "neg_tail_id")
FULL_STEPS = ((0, 0), (0, 1), (0, 38), (1, 0), (1, 38))


def main():
    import_reference()
    from hopwise.config import Config
    from hopwise.data import create_dataset, data_preparation
    from hopwise.utils import init_seed
    from hopwise.utils.enum_type import KGDataLoaderState

    config = Config(model="TransE", dataset="ml-100k",
                    config_dict={"embedding_size": 64, "train_batch_size": 2048, "use_gpu": False, "epochs": 1,
                                 "show_progress": False, "seed": 2024})
    init_seed(config["seed"], config["reproducibility"])
    dataset = create_dataset(config)
    train_data, _, _ = data_preparation(config, dataset)
    gl, kl = train_data.general_dataloader, train_data.kg_dataloader
    inter, kg = gl._dataset.inter_feat, kl._dataset.kg_feat
    out = {
        "seed": np.int64(2024), "batch": np.int64(gl.step),
        "n_users": np.int64(dataset.user_num), "n_items": np.int64(dataset.item_num),
        "n_entities": np.int64(dataset.entity_num), "n_relations": np.int64(dataset.relation_num),
        "inter_user": inter["user_id"].numpy().astype(np.int32), "inter_item": inter["item_id"].numpy().astype(np.int32),
        "kg_head": kg["head_id"].numpy().astype(np.int32), "kg_rel": kg["relation_id"].numpy().astype(np.int32),
        "kg_tail": kg["tail_id"].numpy().astype(np.int32),
    }
    # what the reference KGSampler filters with, the dataset's full head / tail arrays (sampler.py:321-336), are the
    # KG triples' own columns: the tests filter with kg_head / kg_tail, so they are not stored twice
    assert np.array_equal(np.asarray(dataset.head_entities), out["kg_head"])
    assert np.array_equal(np.asarray(dataset.tail_entities), out["kg_tail"])
    # the rec sampler's train-phase used ids (sampler.py:229-252) as COO
    used = gl._sampler.used_ids
    uu, ii = [], []
    for u, s in enumerate(used):
        for i in sorted(s):
            uu.append(u)
            ii.append(i)
    out["used_user"], out["used_item"] = np.array(uu, dtype=np.int32), np.array(ii, dtype=np.int32)
    st = np.random.get_state()
    out["mt_key"], out["mt_pos"] = st[1].astype(np.uint32), np.int64(st[2])
    train_data.set_mode(KGDataLoaderState.RSKG)
    crcs, lens = [], []
    for ep in range(2):
        for i, b in enumerate(train_data):
            row, ln = [], []
            for k in KEYS:
                v = b[k].numpy().astype(np.int64)
                row.append(zlib.crc32(v.tobytes()))
                ln.append(v.shape[0])
                if (ep, i) in FULL_STEPS:
                    out[f"full_{ep}_{i}_{k}"] = v.astype(np.int32)
            crcs.append(row)
            lens.append(ln)
    out["crc"] = np.array(crcs, dtype=np.int64).reshape(2, -1, len(KEYS))
    out["lens"] = np.array(lens, dtype=np.int64).reshape(2, -1, len(KEYS))
    st2 = np.random.get_state()
    out["mt_key_end"], out["mt_pos_end"] = st2[1].astype(np.uint32), np.int64(st2[2])
    path = os.path.join(HERE, "loader_ml100k.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes; steps/epoch", out["crc"].shape[1])


if __name__ == "__main__":
    main()
