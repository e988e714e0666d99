"""Knowledge-database builder (SURVEY.md §8 f1): the offline steps of KEDs that produce
`cc_image_databases.pt`, `cc_text_databases.pt` and `database_names.txt`.

  reference                                                    here
  -----------------------------------------------------------  --------------------------------------
  database.py:14-17   random.sample(os.listdir(text_dir), 500000)   sample_pairs()
  src/data.py:636-671 LoadDataBase: torch.load one .pt per pair      load_pair_folders()
  src/main.py:445-469 cat, bases / bases.norm(dim=1, keepdim=True)   build_knowledge_base(normalize=True):
                      (CPU, 1.5 GB per base)                          rows are normalised on the GPU while
                                                                     they are added (one pass emits the fp32
                                                                     master, the bf16 operand and the norms)
  README.md:17        the three artefacts                            save_artefacts() / KnowledgeBase.load()

File formats are the reference's: each per-pair file holds one 768-d feature tensor; the artefacts
are float32 [N, 768] CPU tensors saved with torch.save plus one basename per line.
"""
from __future__ import annotations

import os
import random
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from .index import METRIC_L2
from .retrieval import KnowledgeBase


def sample_pairs(all_files: Sequence[str], n: int = 500000, seed: Optional[int] = None) -> List[str]:
    """database.py:17 -- `random.sample(all_files, 500000)`; a seed makes the draw reproducible."""
    rng = random.Random(seed) if seed is not None else random
    return rng.sample(list(all_files), min(int(n), len(all_files)))


def load_pair_folders(folder: str, names: Optional[Sequence[str]] = None) -> Tuple[torch.Tensor, torch.Tensor, List[str]]:
    """LoadDataBase (src/data.py:636-671) without the DataLoader: read image_feature_database/<name>
    and text_feature_database/<name> for every name (default: every file of the image folder) and
    stack them to float32 [N, d] tensors. A pair is kept only if both files exist (database.py:28)."""
    image_folder = os.path.join(folder, "image_feature_database")
    text_folder = os.path.join(folder, "text_feature_database")
    if names is None:
        names = sorted(os.listdir(image_folder))
    img, txt, kept = [], [], []
    for name in names:
        ip, tp = os.path.join(image_folder, name), os.path.join(text_folder, name)
        if not (os.path.isfile(ip) and os.path.isfile(tp)):
            continue
        img.append(torch.load(ip, map_location="cpu").detach().reshape(-1).to(torch.float32))
        txt.append(torch.load(tp, map_location="cpu").detach().reshape(-1).to(torch.float32))
        kept.append(name)
    if not kept:
        raise FileNotFoundError(f"no feature pairs under {folder}")
    return torch.stack(img), torch.stack(txt), kept


def build_knowledge_base(image_rows: torch.Tensor, text_rows: torch.Tensor, names: Sequence[str],
                         device: int = 0, metric: int = METRIC_L2, normalize: bool = True) -> KnowledgeBase:
    """Rows -> searchable database on `device`. With normalize=True the rows are L2-normalised on
    the GPU during add (src/main.py:465-466); the CPU tensors kept in the KnowledgeBase (the .pt
    layout) are read back from the device so both sides hold identical bits."""
    kb = KnowledgeBase.__new__(KnowledgeBase)
    KnowledgeBase._init_indices(kb, image_rows, text_rows, names, device, metric, normalize)
    return kb


def drop_near_duplicates(image_rows: torch.Tensor, text_rows: torch.Tensor, names: Sequence[str], radius: float,
                         device: int = 0, batch: int = 65536):
    """Leave out the later copies of near-duplicate images (CC3M holds one photo under several names,
    and a copy of a query's own pair would come back as its first neighbour). Row j is dropped when
    some row i < j has a normalised-image inner product > radius with it: a range self-join of the
    base on the GPU, exact in fp32, in query batches of `batch` rows. The rule depends neither on the
    batch size nor on the order of the batches. Returns (image_rows, text_rows, names, dropped_rows)
    with the kept rows in their order and dropped_rows an int64 tensor of the dropped row numbers."""
    from .index import METRIC_INNER_PRODUCT, GpuIndexFlat

    n = int(image_rows.shape[0])
    if int(text_rows.shape[0]) != n or len(names) != n:
        raise ValueError(f"drop_near_duplicates: {n} image rows, {int(text_rows.shape[0])} text rows, {len(names)} names")
    if int(batch) <= 0:
        raise ValueError("drop_near_duplicates: batch must be positive")
    dev = torch.device("cuda", device)
    index = GpuIndexFlat(int(image_rows.shape[1]), METRIC_INNER_PRODUCT, device)
    index.add(image_rows.to(dev, torch.float32).contiguous(), normalize=True)
    drop = torch.zeros(n, dtype=torch.bool, device=dev)
    for b0 in range(0, n, int(batch)):
        b1 = min(n, b0 + int(batch))
        q = torch.from_numpy(index.get_rows(b0, b1 - b0)).to(dev)
        lims, _, I = index.range_search(q, radius)
        row = torch.repeat_interleave(torch.arange(b0, b1, device=dev), lims[1:] - lims[:-1])
        drop[row[I < row]] = True
    del index
    keep = (~drop).cpu()
    kept_names = [nm for nm, k in zip(names, keep.tolist()) if k]
    return image_rows[keep], text_rows[keep], kept_names, drop.nonzero().flatten().cpu()


def save_artefacts(kb: KnowledgeBase, out_dir: str) -> Tuple[str, str, str]:
    """Write cc_image_databases.pt / cc_text_databases.pt / database_names.txt (README.md:17)."""
    os.makedirs(out_dir, exist_ok=True)
    paths = (os.path.join(out_dir, "cc_image_databases.pt"), os.path.join(out_dir, "cc_text_databases.pt"),
             os.path.join(out_dir, "database_names.txt"))
    torch.save(kb.image_bases, paths[0])
    torch.save(kb.text_bases, paths[1])
    with open(paths[2], "w") as f:
        f.write("\n".join(kb.basenames) + ("\n" if kb.basenames else ""))
    return paths
