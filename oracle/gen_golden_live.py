"""Generate tests/golden/reference_live_*.npz: the reference's answers for the randomised cases of tests/test_reference_live.py.

    python oracle/gen_golden_live.py <reference checkout>

The reference is imported and executed from where it lies, as in oracle/gen_golden.py.  Every case builds its inputs from the
same seeded stream as the test, so only the reference's outputs are stored.  Outputs too large to keep whole are sampled at
positions drawn from a seeded generator the test draws again, with sums or norms beside them so that the unsampled part is
still checked in aggregate.
"""
from __future__ import annotations

import importlib
import os
import sys
import types

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import gen_golden as gg           # noqa: E402
from oracle import hd_oracle as hdo            # noqa: E402
from oracle import tokenpacker_oracle as tpo  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")

MODULE_CASES = [(2, 64, 901), (3, 96, 902), (4, 160, 903), (6, 32, 904), (12, 64, 905)]
GRADIENT_CASES = [(2, 64, 911), (3, 32, 912), (4, 96, 913), (8, 32, 914)]
# positions kept per output (drawn with np.random.default_rng(seed).integers(0, size, n)); tests/test_reference_live.py
# draws the same positions
MODULE_SAMPLES, GRAD_SAMPLES, TILE_SAMPLES = 1024, 128, 512


def gen_projector(builder):
    out = {}
    for s, hidden, seed in MODULE_CASES:
        params = tpo.make_params(hidden, seed=seed)
        x0, xm = tpo.make_inputs(2, seed=seed + 1000)
        m = builder.TokenPacker(hidden_size=hidden, scale_factor=s)
        m.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
        with torch.no_grad():
            ref = m.eval()((torch.from_numpy(x0), torch.from_numpy(xm))).numpy()
        key = f"module_s{s}_h{hidden}_seed{seed}"
        out[key + "_sample"] = ref.reshape(-1)[np.random.default_rng(seed).integers(0, ref.size, MODULE_SAMPLES)]
        out[key + "_row_sum"] = ref.astype(np.float64).sum(axis=-1)
    for s, hidden, seed in GRADIENT_CASES:
        params = tpo.make_params(hidden, seed=seed)
        x0, xm = tpo.make_inputs(2, seed=seed + 1000)
        gw = torch.from_numpy(np.random.default_rng(seed).standard_normal((2, (24 // s) ** 2, hidden)).astype(np.float32))
        m = builder.TokenPacker(hidden_size=hidden, scale_factor=s)
        m.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
        (m((torch.from_numpy(x0), torch.from_numpy(xm))) * gw).sum().backward()
        # one row per parameter, in named_parameters() order
        names, samples, argmax, peak, norm = [], [], [], [], []
        rng = np.random.default_rng(seed)
        for name, p in m.named_parameters():
            g = p.grad.numpy().reshape(-1)
            names.append(name)
            samples.append(g[rng.integers(0, g.size, GRAD_SAMPLES)])
            argmax.append(int(np.argmax(np.abs(g))))
            peak.append(g[argmax[-1]])
            norm.append(np.linalg.norm(g.astype(np.float64)))
        key = f"grad_s{s}_h{hidden}_seed{seed}"
        out[key + "_names"] = np.asarray(names)
        out[key + "_sample"] = np.stack(samples)
        out[key + "_argmax"] = np.asarray(argmax, dtype=np.int64)
        out[key + "_max"] = np.asarray(peak, dtype=np.float32)
        out[key + "_norm"] = np.asarray(norm, dtype=np.float64)
    np.savez_compressed(os.path.join(OUT, "reference_live_projector.npz"), **out)


def gen_hd(pd):
    out = {}
    # grid selector: 200 sizes per patch_num, extreme aspect ratios included
    rng = np.random.default_rng(4242)
    rows = []
    for patch_num in (9, 16, 25):
        ip = pd.Image_Patch(image_size=336, patch_num=patch_num)
        sizes = [tuple(int(v) for v in rng.integers(16, 3200, size=2)) for _ in range(170)]
        sizes += [(int(rng.integers(16, 200)), int(rng.integers(2000, 6000))) for _ in range(15)]
        sizes += [(int(rng.integers(2000, 6000)), int(rng.integers(16, 200))) for _ in range(15)]
        rows += [(h, w, patch_num) + tuple(int(v) for v in ip.calculate(h, w)) for h, w in sizes]
    out["grid_table"] = np.asarray(rows, dtype=np.int32)

    # tiling block (eval/model_vqa.py:88-123, no function boundary upstream), exec'd where it lies
    src = gg.source_range("llava/eval/model_vqa.py", 88, 123)
    assert src.lstrip().startswith("image = preprocess(image)")
    rng = np.random.default_rng(515)
    meta = []
    for trial in range(18):
        patch_num = (9, 16, 25)[trial % 3]
        h, w = (int(v) for v in rng.integers(40, 1500, size=2))
        img = rng.standard_normal((3, h, w)).astype(np.float32)
        ns = {"image": torch.from_numpy(img), "preprocess": (lambda t: t),
              "image_patch": pd.Image_Patch(image_size=336, patch_num=patch_num), "F": F, "torch": torch}
        exec(src, ns)
        want = ns["image_tensor"].numpy()
        meta.append((h, w, patch_num, int(ns["h_block"]), int(ns["w_block"]), want.shape[0]))
        out[f"tile{trial}_sample"] = want.reshape(-1)[np.random.default_rng(trial).integers(0, want.size, TILE_SAMPLES)]
        out[f"tile{trial}_crop_sum"] = want.astype(np.float64).sum(axis=(1, 2, 3))
        out[f"tile{trial}_crop_abs"] = np.abs(want.astype(np.float64)).sum(axis=(1, 2, 3))
    out["tile_meta"] = np.asarray(meta, dtype=np.int64)

    # slice assembly (llava_arch.py:141-155), exec'd where it lies
    src = gg.source_range("llava/model/llava_arch.py", 141, 155)
    assert src.lstrip().startswith("image_feature_list = []")
    rng = np.random.default_rng(606)
    for trial in range(20):
        m, hdim = int(rng.integers(1, 6)), 4
        grids = [(int(rng.integers(1, 6)), int(rng.integers(1, 6))) for _ in range(int(rng.integers(1, 6)))]
        sep_row = rng.standard_normal(hdim).astype(np.float32)
        ret_row = rng.standard_normal(hdim).astype(np.float32)
        total = sum(hdo.n_crops(a, b) for a, b in grids)
        feats = rng.standard_normal((total, m, hdim)).astype(np.float32)

        class _Model:
            def embed_tokens(self, tok):
                return torch.from_numpy(sep_row if int(tok[0]) == 0 else ret_row)[None]

        class _Self:
            def get_model(self):
                return _Model()

        ns = {"image_features": torch.from_numpy(feats), "h_block": [g[0] for g in grids], "w_block": [g[1] for g in grids],
              "self": _Self(), "sep": torch.tensor([0]), "ret": torch.tensor([1]), "torch": torch, "cur_image_idx": 0}
        want = []
        for b in range(len(grids)):
            ns["batch_idx"] = b
            exec(src, ns)
            want.append(ns["cur_image_features"].numpy())
        out[f"assemble{trial}_packed"] = np.concatenate(want, axis=0)
        out[f"assemble{trial}_cu"] = np.concatenate([[0], np.cumsum([q.shape[0] for q in want])]).astype(np.int64)
    np.savez_compressed(os.path.join(OUT, "reference_live_hd.npz"), **out)


def gen_splice():
    """prepare_inputs_labels_for_multimodal (llava_arch.py:100-233) on random batches: both mm_use_im_start_end branches,
    'pad' and 'slice' modes, ragged and image-free samples.  Per branch the 40 trials' outputs are stored flattened and
    concatenated, with each trial's (B, Lmax)."""
    for name, sub in (("llava", "llava"), ("llava.model", "llava/model")):      # bypass the two __init__.py (transformers-4.31 imports)
        if name not in sys.modules:
            mod = types.ModuleType(name)
            mod.__path__ = [os.path.join(gg.REF, sub)]
            sys.modules[name] = mod
    arch = importlib.import_module("llava.model.llava_arch")

    class _Model:
        def __init__(self, table):
            self.table = table

        def embed_tokens(self, ids):
            return self.table[ids]

    class _Tok:
        def convert_tokens_to_ids(self, toks):
            return [{",": 5, "\n": 6}[t] for t in toks]

    class _Fake(arch.LlavaMetaForCausalLM):
        def __init__(self, table, feats, start_end):
            self._m, self._f, self.tokenizer = _Model(table), feats, _Tok()
            self.config = types.SimpleNamespace(tune_mm_mlp_adapter=start_end, mm_use_im_start_end=start_end)
            self.device = torch.device("cpu")

        def get_model(self):
            return self._m

        def get_vision_tower(self):
            return object()

        def encode_images(self, images):
            return self._f

    out = {}
    for start_end in (False, True):
        rng = np.random.default_rng(77 if start_end else 78)
        hdim, vocab, m = 8, 40, 3
        table = rng.standard_normal((vocab, hdim)).astype(np.float32)
        shapes, embeds, labels_out, masks = [], [], [], []
        for trial in range(40):
            B, L = int(rng.integers(1, 4)), int(rng.integers(6, 12))
            slice_mode = (not start_end) and trial % 2 == 1
            ids = rng.integers(7, vocab, size=(B, L))
            n_img = []
            for b in range(B):
                k = 1 if slice_mode else int(rng.integers(0, 3))
                if start_end:
                    pos = sorted(rng.choice(np.arange(2, L - 1, 3), size=min(k, (L - 3) // 3), replace=False).tolist())
                    for p in pos:
                        ids[b, p - 1], ids[b, p], ids[b, p + 1] = 30, -200, 31
                    n_img.append(len(pos))
                else:
                    pos = sorted(rng.choice(L, size=k, replace=False).tolist())
                    ids[b, pos] = -200
                    n_img.append(k)
            labels = ids.copy()
            mask = np.ones_like(ids, dtype=bool)
            if slice_mode:
                grids = [(int(rng.integers(1, 4)), int(rng.integers(1, 4))) for _ in range(B)]
                crops = sum(hdo.n_crops(a, b) for a, b in grids)
                feats = rng.standard_normal((crops, m, hdim)).astype(np.float32)
                hb, wb = [g[0] for g in grids], [g[1] for g in grids]
                mode = "slice"
            else:
                n_seq = sum(max(k, 1) for k in n_img)
                feats = rng.standard_normal((n_seq, m, hdim)).astype(np.float32)
                hb = wb = None
                mode = "pad"
            fake = _Fake(torch.from_numpy(table), torch.from_numpy(feats), start_end)
            _, ref_mask, _, ref_embeds, ref_labels = fake.prepare_inputs_labels_for_multimodal(
                torch.from_numpy(ids), torch.from_numpy(mask), None, torch.from_numpy(labels), object(), mode, hb, wb)
            shapes.append(tuple(ref_labels.shape))
            embeds.append(ref_embeds.numpy().reshape(-1))
            labels_out.append(ref_labels.numpy().reshape(-1))
            masks.append(ref_mask.numpy().reshape(-1))
        pre = f"start_end{int(start_end)}"
        out[pre + "_shape"] = np.asarray(shapes, dtype=np.int64)
        out[pre + "_embeds"] = np.concatenate(embeds)
        out[pre + "_labels"] = np.concatenate(labels_out).astype(np.int32)
        out[pre + "_mask"] = np.concatenate(masks)
    np.savez_compressed(os.path.join(OUT, "reference_live_splice.npz"), **out)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    gg.REF = sys.argv[1]
    torch.set_num_threads(os.cpu_count())
    gen_projector(gg.load_by_path("ref_builder_live", "llava/model/multimodal_projector/builder.py"))
    gen_hd(gg.load_by_path("ref_patch_divide_live", "llava/patch_divide.py"))
    gen_splice()
