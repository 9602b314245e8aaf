"""Randomised comparison against the REFERENCE ITSELF: the reference's answers on these cases were produced by running it
(oracle/gen_golden_live.py) and are stored in tests/golden/reference_live_*.npz.  Widens the pin of the oracle and of the
product's host logic beyond the fixed fixture cases: fresh seeds every run of this file would defeat reproducibility, so the
seeds are fixed but different from the fixture seeds.  Each case builds its inputs from the same seeded stream as the
generator; outputs too large to store whole are compared at the generator's seeded positions and through sums or norms."""
import os

import numpy as np
import pytest


@pytest.fixture(scope="module")
def live_projector(golden_dir):
    return np.load(os.path.join(golden_dir, "reference_live_projector.npz"))


@pytest.fixture(scope="module")
def live_hd(golden_dir):
    return np.load(os.path.join(golden_dir, "reference_live_hd.npz"))


@pytest.fixture(scope="module")
def live_splice(golden_dir):
    return np.load(os.path.join(golden_dir, "reference_live_splice.npz"))


@pytest.mark.parametrize("s,hidden,seed", [(2, 64, 901), (3, 96, 902), (4, 160, 903), (6, 32, 904), (12, 64, 905)])
def test_oracle_vs_reference_module(live_projector, s, hidden, seed):
    """Fresh weights (every 1-D parameter perturbed so LayerNorm / bias paths matter), odd hidden sizes, N=2."""
    import torch
    from oracle import tokenpacker_oracle as tpo
    from oracle import torch_port
    params = tpo.make_params(hidden, seed=seed)
    x0, xm = tpo.make_inputs(2, seed=seed + 1000)
    key = f"module_s{s}_h{hidden}_seed{seed}"
    ref_sample, ref_row_sum = live_projector[key + "_sample"], live_projector[key + "_row_sum"]
    with torch.no_grad():
        port = torch_port.forward({k: torch.from_numpy(v) for k, v in params.items()}, torch.from_numpy(x0), torch.from_numpy(xm), s).numpy()
    out = tpo.tokenpacker_forward(params, x0, xm, s)
    assert out.shape == port.shape == ref_row_sum.shape + (hidden,)
    idx = np.random.default_rng(seed).integers(0, out.size, ref_sample.size)
    assert np.abs(out.reshape(-1)[idx] - ref_sample).max() < 5e-6
    assert np.abs(port.reshape(-1)[idx] - ref_sample).max() < 1e-6
    # every element within the bound above keeps each row sum within hidden times it
    assert np.abs(out.sum(axis=-1) - ref_row_sum).max() < 5e-6 * hidden
    assert np.abs(port.astype(np.float64).sum(axis=-1) - ref_row_sum).max() < 1e-6 * hidden


def test_grid_selector_vs_reference_random(live_hd):
    """Product (C ABI, host arithmetic) and oracle vs Image_Patch.calculate on 600 fresh sizes incl. extreme aspect ratios."""
    from oracle import hd_oracle as hdo
    from tokenpacker_b200 import hd_grid
    table = live_hd["grid_table"].tolist()
    assert len(table) == 600 and {p for _, _, p, _, _ in table} == {9, 16, 25}
    for h, w, patch_num, hb, wb in table:
        assert hd_grid(h, w, patch_num) == (hb, wb), (h, w, patch_num)
        assert tuple(hdo.hd_grid(h, w, patch_num)) == (hb, wb), (h, w, patch_num)


@pytest.mark.parametrize("start_end", [False, True])
def test_splice_vs_reference_method_random(live_splice, start_end):
    """Random batches through the reference's prepare_inputs_labels_for_multimodal vs the oracle AND the product's host planner
    (llava_arch.py:100-233, both mm_use_im_start_end branches, 'pad' and 'slice' modes, ragged and image-free samples)."""
    from oracle import hd_oracle as hdo
    from oracle import splice_oracle as spo
    from tokenpacker_b200 import splice_plan
    pre = f"start_end{int(start_end)}"
    shapes = live_splice[pre + "_shape"]
    all_embeds, all_labels, all_mask = live_splice[pre + "_embeds"], live_splice[pre + "_labels"], live_splice[pre + "_mask"]
    assert shapes.shape == (40, 2)
    rng = np.random.default_rng(77 if start_end else 78)
    hdim, vocab, m = 8, 40, 3
    table = rng.standard_normal((vocab, hdim)).astype(np.float32)
    tok_off = emb_off = 0
    for trial in range(40):
        B, L = int(rng.integers(1, 4)), int(rng.integers(6, 12))
        slice_mode = (not start_end) and trial % 2 == 1
        ids = rng.integers(7, vocab, size=(B, L))
        n_img = []
        for b in range(B):
            k = 1 if slice_mode else int(rng.integers(0, 3))
            if start_end:
                # <im_start> IMAGE <im_end> triples (30 / 31 stand-ins), never at position 0 (upstream always has a BOS first)
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
            packed, cu = hdo.hd_assemble(feats, hb, wb, table[5], table[6])
            seqs = [packed[cu[i]:cu[i + 1]] for i in range(B)]
        else:
            n_seq = sum(max(k, 1) for k in n_img)          # an image-free sample still consumes one (llava_arch.py:121-134)
            feats = rng.standard_normal((n_seq, m, hdim)).astype(np.float32)
            seqs = [feats[i] for i in range(n_seq)]
        rb, lmax = (int(v) for v in shapes[trial])
        assert rb == B
        n_tok = B * lmax
        ref_embeds = all_embeds[emb_off:emb_off + n_tok * hdim].reshape(B, lmax, hdim)
        ref_labels = all_labels[tok_off:tok_off + n_tok].reshape(B, lmax)
        ref_mask = all_mask[tok_off:tok_off + n_tok].reshape(B, lmax)
        tok_off, emb_off = tok_off + n_tok, emb_off + n_tok * hdim
        o_mask, o_embeds, o_labels = spo.splice(ids, mask, labels, seqs, table, im_start_end=start_end)
        np.testing.assert_array_equal(o_embeds, ref_embeds)
        np.testing.assert_array_equal(o_labels, ref_labels)
        np.testing.assert_array_equal(o_mask, ref_mask)
        visual = np.concatenate(seqs, axis=0)
        cu_seq = np.concatenate([[0], np.cumsum([q.shape[0] for q in seqs])])
        plan = splice_plan(ids, cu_seq, labels, mask, im_start_end=start_end)
        rows = np.zeros((plan.src_index.shape[0], hdim), dtype=np.float32)
        src = plan.src_index
        rows[src >= 0] = table[src[src >= 0]]
        rows[src <= -2] = visual[-src[src <= -2] - 2]
        np.testing.assert_array_equal(rows.reshape(B, plan.lmax, hdim), ref_embeds)
        np.testing.assert_array_equal(plan.labels, ref_labels)
        np.testing.assert_array_equal(plan.attention_mask, ref_mask)
    assert tok_off == all_labels.size and emb_off == all_embeds.size


def test_tiling_block_vs_reference_source_random(live_hd):
    """The resize -> pad -> split -> thumbnail block has no function boundary upstream (pasted inline 9 times); the source range
    eval/model_vqa.py:88-123, run on fresh image sizes, vs the oracle restatement."""
    from oracle import hd_oracle as hdo
    meta = live_hd["tile_meta"].tolist()
    assert len(meta) == 18
    rng = np.random.default_rng(515)
    for trial in range(18):
        patch_num = (9, 16, 25)[trial % 3]
        h, w = (int(v) for v in rng.integers(40, 1500, size=2))
        img = rng.standard_normal((3, h, w)).astype(np.float32)
        assert tuple(meta[trial][:3]) == (h, w, patch_num)
        crops, hb, wb = hdo.hd_tile(img[None], patch_num)
        assert (hb, wb) == tuple(meta[trial][3:5])
        assert crops.shape == (meta[trial][5], 3, 336, 336), crops.shape
        want = live_hd[f"tile{trial}_sample"]
        got = crops.reshape(-1)[np.random.default_rng(trial).integers(0, crops.size, want.size)]
        assert np.abs(got - want).max() <= 2e-6, (h, w, patch_num, float(np.abs(got - want).max()))
        # every pixel within the bound above keeps each crop's sums within 336 * 336 * 3 times it
        bound = 2e-6 * crops[0].size
        c64 = crops.astype(np.float64)
        assert np.abs(c64.sum(axis=(1, 2, 3)) - live_hd[f"tile{trial}_crop_sum"]).max() <= bound
        assert np.abs(np.abs(c64).sum(axis=(1, 2, 3)) - live_hd[f"tile{trial}_crop_abs"]).max() <= bound


@pytest.mark.parametrize("s,hidden,seed", [(2, 64, 911), (3, 32, 912), (4, 96, 913), (8, 32, 914)])
def test_gradient_oracle_vs_reference_autograd(live_projector, s, hidden, seed):
    """tests/test_backward_gpu.py uses autograd over oracle/torch_port.py as the gradient oracle: pin THAT to autograd through the
    reference module itself (fp32, CPU), every parameter."""
    import torch
    from oracle import tokenpacker_oracle as tpo
    from oracle import torch_port
    params = tpo.make_params(hidden, seed=seed)
    x0, xm = tpo.make_inputs(2, seed=seed + 1000)
    x0, xm = torch.from_numpy(x0), torch.from_numpy(xm)
    gw = torch.from_numpy(np.random.default_rng(seed).standard_normal((2, (24 // s) ** 2, hidden)).astype(np.float32))
    p = {k: torch.from_numpy(v).clone().requires_grad_(True) for k, v in params.items()}
    (torch_port.forward(p, x0, xm, s) * gw).sum().backward()
    key = f"grad_s{s}_h{hidden}_seed{seed}"
    names = live_projector[key + "_names"].tolist()
    assert sorted(names) == sorted(params)
    rng = np.random.default_rng(seed)
    for i, name in enumerate(names):
        g = p[name].grad.numpy().reshape(-1)
        want = live_projector[key + "_sample"][i]
        at, peak, norm = int(live_projector[key + "_argmax"][i]), float(live_projector[key + "_max"][i]), float(live_projector[key + "_norm"][i])
        scale = abs(peak) + 1e-12
        tol = 2e-5 * scale + 1e-7
        got = g[rng.integers(0, g.size, want.size)]
        assert float(np.abs(got - want).max()) <= tol, (name, float(np.abs(got - want).max()), scale)
        assert abs(float(g[at]) - peak) <= tol, (name, float(g[at]), peak)
        assert float(np.abs(g).max()) <= scale + tol, (name, float(np.abs(g).max()), scale)
        # every element within tol keeps the gradient's norm within tol * sqrt(size)
        assert abs(float(np.linalg.norm(g.astype(np.float64))) - norm) <= tol * np.sqrt(g.size), name


def test_slice_assembly_vs_reference_source_random(live_hd):
    """llava_arch.py:141-155, run on random grids, vs the oracle and the product's host plan (tp_hd_plan)."""
    from oracle import hd_oracle as hdo
    from tokenpacker_b200 import hd_plan
    rng = np.random.default_rng(606)
    for trial in range(20):
        m, hdim = int(rng.integers(1, 6)), 4
        grids = [(int(rng.integers(1, 6)), int(rng.integers(1, 6))) for _ in range(int(rng.integers(1, 6)))]
        sep_row = rng.standard_normal(hdim).astype(np.float32)
        ret_row = rng.standard_normal(hdim).astype(np.float32)
        total = sum(hdo.n_crops(a, b) for a, b in grids)
        feats = rng.standard_normal((total, m, hdim)).astype(np.float32)
        want, want_cu = live_hd[f"assemble{trial}_packed"], live_hd[f"assemble{trial}_cu"]
        hb, wb = [g[0] for g in grids], [g[1] for g in grids]
        packed, cu = hdo.hd_assemble(feats, hb, wb, sep_row, ret_row)
        np.testing.assert_array_equal(packed, want)
        np.testing.assert_array_equal(cu, want_cu)
        plan = hd_plan(hb, wb, m)
        np.testing.assert_array_equal(plan.cu_seqlens.numpy(), want_cu)
        rebuilt = np.full_like(want, np.nan)
        for c, r0 in enumerate(plan.seg_row_offset.tolist()):
            rebuilt[r0:r0 + m] = feats[c]
        rebuilt[plan.sep_rows.numpy()] = sep_row
        rebuilt[plan.ret_rows.numpy()] = ret_row
        np.testing.assert_array_equal(rebuilt, want)
