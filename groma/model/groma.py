"""`groma.model.groma` surface: GromaConfig / GromaModel with the reference's forward / generate contract
(reference groma/model/groma.py:31-431), executed by the B200-native engine.

Kept from the reference (SURVEY.md section 8b): constructor + from_pretrained, init_special_token_id and the token-id
attributes, mutable config.{nms_thres, box_score_thres, max_region_num}, forward(...) -> CausalLMOutputWithPast with
hidden_states=(llm_hidden_states, vis_outputs), tuple-of-tuples past_key_values [B,32,ctx,128], in-place edit of the
caller's input_ids for <refer_box>/<ground_box> placeholders (T8), torch.randperm on the global CPU RNG (T6), the
all-ones decode mask (T7), generate(...).sequences / .hidden_states[0][-1].  There is no CPU path: construction fails
without a CUDA device."""
from __future__ import annotations

import copy
import glob
import json
import os
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch
from transformers import AutoConfig, AutoModel, LlamaConfig, PretrainedConfig
from transformers.modeling_outputs import CausalLMOutputWithPast

from groma.constants import IGNORE_INDEX
from groma.model.ddetr import CustomDDETRConfig, CustomDDETRModel, perceiver_fields
from groma_b200 import ops as G
from groma_b200.config import PathConfig
from groma_b200.engine import GromaEngine


class GromaConfig(PretrainedConfig):
    model_type = "groma"

    def __init__(self, llm_cfg=None, perceiver_cfg=None, num_new_token=0, nms_thres=0.6, box_score_thres=0.15,
                 max_region_num=100, **kwargs):
        super().__init__(**kwargs)
        if perceiver_cfg is None:
            self.perceiver_cfg = CustomDDETRConfig()
        elif isinstance(perceiver_cfg, dict):
            self.perceiver_cfg = CustomDDETRConfig(**perceiver_cfg)
        elif isinstance(perceiver_cfg, CustomDDETRConfig):
            self.perceiver_cfg = perceiver_cfg
        else:
            raise NotImplementedError("currently only supports CustomDDETR as perceiver.")
        if llm_cfg is None:
            self.llm_cfg = LlamaConfig()
        elif isinstance(llm_cfg, dict):
            self.llm_cfg = LlamaConfig(**llm_cfg)
        elif isinstance(llm_cfg, LlamaConfig):
            self.llm_cfg = llm_cfg
        else:
            raise NotImplementedError("currently only supports LlamaModel as LLM.")
        self.nms_thres = nms_thres
        self.box_score_thres = box_score_thres
        self.max_region_num = max_region_num
        self.num_new_token = num_new_token
        self.vocab_size = self.llm_cfg.vocab_size + num_new_token

    def to_json_string(self, use_diff: bool = True) -> str:
        d = copy.deepcopy(self)
        if use_diff:
            d.perceiver_cfg = json.loads(d.perceiver_cfg.to_json_string(True))
            d.llm_cfg = d.llm_cfg.to_diff_dict()
            d = d.to_diff_dict()
        else:
            d.perceiver_cfg = json.loads(d.perceiver_cfg.to_json_string(False))
            d.llm_cfg = d.llm_cfg.to_dict()
            d = d.to_dict()
        return json.dumps(d, indent=2, sort_keys=True, default=str) + "\n"

    def to_path_config(self, image_size: int = 448, **overrides) -> PathConfig:
        l = self.llm_cfg
        f = perceiver_fields(self.perceiver_cfg)
        f.update(image_size=image_size, llm_hidden=l.hidden_size, llm_layers=l.num_hidden_layers, llm_heads=l.num_attention_heads,
                 llm_inter=l.intermediate_size, vocab=l.vocab_size, num_new_token=self.num_new_token, rms_eps=l.rms_norm_eps,
                 rope_theta=_rope_theta(l),
                 max_pos=l.max_position_embeddings, nms_thres=self.nms_thres, box_score_thres=self.box_score_thres,
                 max_region_num=self.max_region_num)
        if l.num_key_value_heads not in (None, l.num_attention_heads):
            raise NotImplementedError("Vicuna-7B is MHA; GQA is not on the path")
        f.update(overrides)
        return PathConfig(**f)

    @classmethod
    def from_path_config(cls, p: PathConfig) -> "GromaConfig":
        from transformers import Dinov2Config
        vis = Dinov2Config(hidden_size=p.vit_hidden, num_hidden_layers=p.vit_layers, num_attention_heads=p.vit_heads,
                           mlp_ratio=p.vit_mlp // p.vit_hidden, image_size=p.vit_pos_grid * p.patch, patch_size=p.patch,
                           layer_norm_eps=p.vit_ln_eps)
        det = _ddetr_cfg(p)
        llm = LlamaConfig(hidden_size=p.llm_hidden, num_hidden_layers=p.llm_layers, num_attention_heads=p.llm_heads,
                          num_key_value_heads=p.llm_heads, intermediate_size=p.llm_inter, vocab_size=p.vocab,
                          rms_norm_eps=p.rms_eps, max_position_embeddings=p.max_pos)
        return cls(llm_cfg=llm, perceiver_cfg=CustomDDETRConfig(vis_encoder_cfg=vis, ddetr_cfg=det), num_new_token=p.num_new_token,
                   nms_thres=p.nms_thres, box_score_thres=p.box_score_thres, max_region_num=p.max_region_num)


def _rope_theta(l) -> float:
    rt = getattr(l, "rope_theta", None)
    if rt is None:
        rt = (getattr(l, "rope_parameters", None) or {}).get("rope_theta", 10000.0)
    return float(rt)


def _ddetr_cfg(p: PathConfig):
    from transformers import DeformableDetrConfig
    kw = dict(d_model=p.d_model, encoder_layers=p.enc_layers, decoder_layers=p.dec_layers,
              encoder_attention_heads=p.ddetr_heads, decoder_attention_heads=p.ddetr_heads, encoder_n_points=p.n_points,
              decoder_n_points=p.n_points, encoder_ffn_dim=p.ddetr_ffn, decoder_ffn_dim=p.ddetr_ffn, num_queries=p.num_queries,
              two_stage_num_proposals=p.num_queries, num_feature_levels=1, two_stage=True, with_box_refine=True)
    try:
        return DeformableDetrConfig(use_timm_backbone=False, use_pretrained_backbone=False, **kw)
    except Exception:
        return DeformableDetrConfig(**kw)


@dataclass
class GenerateOutput:
    sequences: torch.Tensor
    hidden_states: Tuple
    past_key_values: Optional[Tuple] = None


def _load_generation_config(path: Optional[str], config: "GromaConfig"):
    """`model.generation_config` as the reference's checkpoints carry it: train.py:108-112 stores the tokenizer's
    eos / pad / bos ids in `generation_config.json`, and every eval script passes it back to generate()
    (eval/run_groma.py:92).  Falls back to the ids in config.json (top level, then llm_cfg) when the file is absent."""
    from transformers import GenerationConfig
    if path is not None and os.path.isfile(os.path.join(path, "generation_config.json")):
        return GenerationConfig.from_pretrained(path)
    l = config.llm_cfg

    def pick(name):
        v = config.__dict__.get(name)
        return v if v is not None else getattr(l, name, None)
    return GenerationConfig(eos_token_id=pick("eos_token_id"), pad_token_id=pick("pad_token_id"), bos_token_id=pick("bos_token_id"))


def _eos_list(eos) -> List[int]:
    if eos is None:
        return []
    if isinstance(eos, torch.Tensor):
        return [int(v) for v in eos.reshape(-1).tolist()]
    if isinstance(eos, (list, tuple)):
        return [int(v) for v in eos]
    return [int(eos)]


def _c2c(b: torch.Tensor) -> torch.Tensor:
    return torch.cat([b[:, :2] - 0.5 * b[:, 2:], b[:, :2] + 0.5 * b[:, 2:]], -1)


def _box_iou(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    area_a = (a[:, 2] - a[:, 0]) * (a[:, 3] - a[:, 1])
    area_b = (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])
    lt = torch.max(a[:, None, :2], b[None, :, :2])
    rb = torch.min(a[:, None, 2:], b[None, :, 2:])
    wh = (rb - lt).clamp(min=0)
    inter = wh[..., 0] * wh[..., 1]
    return inter / (area_a[:, None] + area_b[None, :] - inter)


class GromaModel(torch.nn.Module):
    config_class = GromaConfig
    supports_gradient_checkpointing = False

    def __init__(self, config: GromaConfig, state_dict: Optional[Dict[str, torch.Tensor]] = None, image_size: int = 448,
                 path_config: Optional[PathConfig] = None):
        super().__init__()
        if state_dict is None:
            raise ValueError("GromaModel needs weights: use GromaModel.from_pretrained(path) or pass state_dict=")
        self.config = config
        self._path_cfg = path_config if path_config is not None else config.to_path_config(image_size)
        self.engine = GromaEngine(self._path_cfg, state_dict)
        self.perceiver = CustomDDETRModel(config.perceiver_cfg, engine=self.engine)
        self.generation_config = _load_generation_config(None, config)
        self.pad_token_id = None
        self.img_token_id = None
        self.reg_token_id = None
        self.refer_box_token_id = None
        self.refer_feat_token_id = None
        self.ground_box_token_id = None
        self.box_idx_token_ids = None
        self.use_cuda_graph = True
        self.kv_headroom = 64      # decode positions reserved by forward(use_cache=True) beyond the prompt (grows on demand)
        self._graph = None
        self.profile = None   # set to a list to collect (stage name, cuda event) marks during generate()

    def _mark(self, name: str):
        if self.profile is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.profile.append((name, ev))

    # ------------------------------------------------------------------ loading (SURVEY N4: HF checkpoint layout)
    @classmethod
    def from_pretrained(cls, path: str, *model_args, torch_dtype=None, config=None, **kwargs) -> "GromaModel":
        """`GromaModel.from_pretrained(dir)` (eval/run_groma.py:43-61) and `AutoModel.from_pretrained(dir)` (which resolves
        GromaConfig -> GromaModel through the registration at the bottom of this file and passes `config=`).  torch_dtype is
        accepted and ignored: the arithmetic type of the path is bf16 with fp32 accumulation (== the autocast region the
        reference's callers wrap generate() in)."""
        if kwargs.get("load_in_8bit") or kwargs.get("load_in_4bit") or kwargs.get("quantization_config") is not None:
            raise NotImplementedError("8/4-bit loading would change results; the B200 path is bf16")
        from groma_b200.checkpoint import ShardedStateDict, load_config_dict
        path = os.path.expanduser(str(path))
        cd = load_config_dict(path)
        cd.pop("model_type", None)
        if not isinstance(config, GromaConfig):
            config = GromaConfig(**cd)
        # lazy view over the (sharded) checkpoint: the engine packs tensor by tensor into its bf16 device arena
        view = ShardedStateDict(path)
        # region-encoder widths are code constants in the reference (roi_align.py:97-116,233-271), not config fields:
        # read them off the parameter shapes so any checkpoint of that architecture loads
        re_ = "region_encoder."
        geom = dict(region_mid=view.shape(re_ + "roi_align.flatten_linear.weight")[0],
                    pos_hidden=view.shape(re_ + "roi_align.pos_embedd.0.weight")[0],
                    fuse_rounds=sum(1 for k in view if k.startswith(re_ + "mlvl_fuse.fuse_convs.") and k.endswith(".conv.weight")))
        geom.update(cd.get("path_overrides") or {})     # e.g. {"gn_groups": 8} for miniature test checkpoints (reference: 64)
        model = cls(config, state_dict=view, path_config=config.to_path_config(**geom))
        model.generation_config = _load_generation_config(path, config)
        return model

    def cuda(self, device=None):
        return self

    def eval(self):
        return self

    def to(self, *a, **k):
        return self

    def init_special_token_id(self, tokenizer):
        from groma.constants import DEFAULT_TOKENS, REGION_IDX_TOKENS
        self.pad_token_id = tokenizer.pad_token_id
        self.img_token_id = tokenizer.convert_tokens_to_ids([DEFAULT_TOKENS["image"]])[0]
        self.reg_token_id = tokenizer.convert_tokens_to_ids([DEFAULT_TOKENS["region"]])[0]
        self.refer_box_token_id = tokenizer.convert_tokens_to_ids([DEFAULT_TOKENS["rbox"]])[0]
        self.refer_feat_token_id = tokenizer.convert_tokens_to_ids([DEFAULT_TOKENS["rfeat"]])[0]
        self.ground_box_token_id = tokenizer.convert_tokens_to_ids([DEFAULT_TOKENS["gbox"]])[0]
        self.box_idx_token_ids = tokenizer.convert_tokens_to_ids(REGION_IDX_TOKENS)

    def get_perceiver(self):
        return self.perceiver

    def get_llm(self):
        return None

    def prepare_inputs_for_generation(self, input_ids, past_key_values=None, attention_mask=None, inputs_embeds=None, **kwargs):
        if past_key_values:
            input_ids = input_ids[:, -1:]
        model_inputs = {"inputs_embeds": inputs_embeds} if (inputs_embeds is not None and past_key_values is None) else {"input_ids": input_ids}
        model_inputs.update({"past_key_values": past_key_values, "attention_mask": attention_mask, "use_cache": kwargs.get("use_cache"),
                             "images": kwargs.get("images"), "refer_boxes": kwargs.get("refer_boxes"), "ground_boxes": kwargs.get("ground_boxes")})
        return model_inputs

    # ------------------------------------------------------------------ host-side integer bookkeeping
    def _match(self, ids_h: torch.Tensor, labels_h, selected, refer_boxes, ground_boxes):
        """groma.py:283-309, on host copies; returns refer_box_inds."""
        refer_inds = []
        bidx = torch.tensor(self.box_idx_token_ids)
        for i in range(ids_h.shape[0]):
            if (ids_h[i] == self.refer_box_token_id).any():
                m = torch.max(_box_iou(_c2c(refer_boxes[i].float().cpu()), _c2c(selected[i])), dim=-1).indices
                refer_inds.append(m)
                ids_h[i].masked_scatter_(ids_h[i] == self.refer_box_token_id, bidx[m])
            else:
                refer_inds.append(torch.zeros(0, dtype=torch.long))
            if (ids_h[i] == self.ground_box_token_id).any():
                m = torch.max(_box_iou(_c2c(ground_boxes[i].float().cpu()), _c2c(selected[i])), dim=-1).indices
                mask = ids_h[i] == self.ground_box_token_id
                ids_h[i].masked_scatter_(mask, bidx[m])
                if labels_h is not None:
                    labels_h[i].masked_scatter_(mask, bidx[m])
        return refer_inds

    def _assemble(self, ids_h: torch.Tensor, labels_h, num_regions: List[int], n_img: int):
        """groma.py:317-357."""
        new_ids, new_labels = [], []
        for i in range(ids_h.shape[0]):
            ids = ids_h[i]
            ipos = (ids == self.img_token_id).nonzero(as_tuple=True)[0]
            rpos = (ids == self.reg_token_id).nonzero(as_tuple=True)[0]
            assert len(ipos) > 0 and len(rpos) > 0, "prompt needs one <image> and one <region> placeholder"
            ip, rp = int(ipos[0]), int(rpos[0])
            ppos = (ids == self.pad_token_id).nonzero(as_tuple=True)[0]
            pe = int(ppos[0]) if len(ppos) > 0 else len(ids)
            assert ip < rp
            regs = torch.tensor([v for j in range(num_regions[i]) for v in (self.box_idx_token_ids[j], self.reg_token_id)], dtype=torch.long)
            new_ids.append(torch.cat((ids[:ip], torch.full((n_img,), self.img_token_id, dtype=torch.long), ids[ip + 1:rp], regs, ids[rp + 1:pe])))
            if labels_h is not None:
                lb = labels_h[i]
                new_labels.append(torch.cat((lb[:ip], torch.full((n_img,), IGNORE_INDEX, dtype=torch.long), lb[ip + 1:rp],
                                             torch.full((2 * num_regions[i],), IGNORE_INDEX, dtype=torch.long), lb[rp + 1:pe])))
        ids_out = torch.nn.utils.rnn.pad_sequence(new_ids, batch_first=True, padding_value=self.pad_token_id)
        labels_out = torch.nn.utils.rnn.pad_sequence(new_labels, batch_first=True, padding_value=IGNORE_INDEX) if labels_h is not None else None
        return ids_out, labels_out

    # ------------------------------------------------------------------ vision + splice (groma.py:219-375)
    @torch.no_grad()
    def _prefill_inputs(self, input_ids, images, refer_boxes, ground_boxes, labels=None, selected_override=None):
        eng, cfg = self.engine, self.config
        dev = eng.dev
        self._mark("start")
        # host copies of the ids / labels first (the GPU is idle here): reading them back later would wait for the whole vision stage
        ids_h0 = input_ids.detach().cpu()
        ids_h = ids_h0.clone()
        labels_h = labels.detach().cpu().clone() if labels is not None else None
        hs = eng.vit(images)
        self._mark("vit")
        img_tok = eng.image_tokens(hs[-1])
        n_extra = 0
        B = images.shape[0]
        if refer_boxes is not None or ground_boxes is not None:
            n_extra = max((len(refer_boxes[i]) if refer_boxes is not None else 0) + (len(ground_boxes[i]) if ground_boxes is not None else 0) for i in range(B))
        pc, px, sc, det_logits = eng.proposer(hs, n_extra)
        self._mark("proposer")
        # The fused maps of the region encoder do not depend on the selection: they are queued right behind the NMS read-back
        # copies, so the GPU works through them (~38 ms at B = 16) while the host waits for the keep lists, draws the
        # permutations, matches refer / ground boxes and builds the RoI list -- no idle gap at the one host sync of the vision stage.
        maps = {}

        def _queue_maps():
            maps["xs"] = eng.region_maps(hs)
        if selected_override is not None:
            selected = [b.float().cpu() for b in selected_override]
            _queue_maps()
        else:
            selected = eng.select_regions(pc, px, sc, refer_boxes, ground_boxes, cfg.nms_thres, cfg.box_score_thres, cfg.max_region_num,
                                          overlap=_queue_maps)
        refer_inds = self._match(ids_h, labels_h, selected, refer_boxes, ground_boxes)
        if not torch.equal(ids_h, ids_h0):
            input_ids.copy_(ids_h.to(input_ids.device))           # the reference edits the caller's tensor in place (T8)
            if labels is not None:
                labels.copy_(labels_h.to(labels.device))
        self._mark("select+maps")
        region = eng.region_tokens(maps["xs"], selected)
        self._mark("region_tokens")
        counts = [len(b) for b in selected]
        ids_new, labels_new = self._assemble(ids_h, labels_h, counts, img_tok.shape[1])
        Bn, T = ids_new.shape
        x = eng.embed(ids_new)
        flat = ids_new.reshape(-1)
        img_pos = (flat == self.img_token_id).nonzero(as_tuple=True)[0]
        reg_pos = (flat == self.reg_token_id).nonzero(as_tuple=True)[0]
        G.scatter_rows(img_pos.to(dev), img_tok.reshape(-1, x.shape[-1]), x)
        if len(reg_pos) > 0:
            G.scatter_rows(reg_pos.to(dev), region, x)
        ref_pos = (flat == self.refer_feat_token_id).nonzero(as_tuple=True)[0]
        if len(ref_pos) > 0:
            offs, o = [], 0
            for c, ind in zip(counts, refer_inds):
                offs.append(ind + o)
                o += c
            src = G.gather_rows(torch.cat(offs).to(dev).contiguous(), region)
            G.scatter_rows(ref_pos.to(dev), src, x)
        attn_mask = ids_new.ne(self.pad_token_id)
        vis_outputs = {"pred_boxes": [b.to(dev) for b in selected], "image_features": img_tok, "region_features": region}
        aux = dict(pred_all=pc[:, :eng.cfg.num_queries], scores=sc[:, :eng.cfg.num_queries], det_logits=det_logits)
        return x, ids_new, labels_new, attn_mask, vis_outputs, aux

    def _kv_tuple(self, ctx: int):
        kv = self.engine.kv
        return tuple((kv[i, 0][:, :, :ctx], kv[i, 1][:, :, :ctx]) for i in range(kv.shape[0]))

    # ------------------------------------------------------------------ forward (groma.py:202-427)
    @torch.no_grad()
    def forward(self, input_ids=None, inputs_embeds=None, labels=None, attention_mask=None, images=None, refer_boxes=None,
                ground_boxes=None, past_key_values=None, use_cache=False, output_attentions=False, output_hidden_states=False,
                return_dict=False, _selected_override=None, _reserve=0):
        eng = self.engine
        vis_outputs = None
        if past_key_values is None:
            x, ids_new, labels_new, mask, vis_outputs, aux = self._prefill_inputs(input_ids, images, refer_boxes, ground_boxes, labels,
                                                                                  _selected_override)
            B, T = ids_new.shape
            eng.ensure_rope(T + 1)
            # room for a step-wise decode loop over forward(past_key_values=...) (serve/model_worker.py:288-304, serve/cli.py
            # and HF generate all drive the model that way); the cache grows geometrically beyond it
            eng.alloc_kv(B, T + max(int(_reserve), self.kv_headroom))
            kv_len = mask.sum(1).to(torch.int32).to(eng.dev)
            logits = eng.llm_prefill(x, B, T, kv_len).reshape(B, T, -1)
            self._last = dict(ids=ids_new, mask=mask, aux=aux)
        else:
            B = past_key_values[0][0].shape[0]
            past = past_key_values[0][0].shape[-2]
            if eng.kv is None or past != eng.past or B != eng.kv.shape[2]:
                raise RuntimeError("past_key_values must be the cache returned by the previous forward() of this model")
            if past + 1 > eng.kv_cap:
                eng.grow_kv(max(past + 1, 2 * eng.kv_cap))      # new storage: the captured decode graph is keyed on it
            eng.ensure_rope(past + 1)
            d = eng._decode_buffers(B)
            d["ids"].copy_(input_ids.reshape(-1).to(eng.dev))
            d["pos"].fill_(past)
            d["kv_len"].fill_(past + 1)               # all-ones mask over past+1 (groma.py:376-379)
            # step-wise callers (serve/model_worker.py:288-304, serve/cli.py) get the same CUDA-graph step as generate() from
            # their second decode step on; the first one runs eagerly (it also warms every kernel up outside the capture)
            self._fwd_decode_steps = getattr(self, "_fwd_decode_steps", 0) + 1
            if self.use_cuda_graph and self._fwd_decode_steps >= 2:
                self._capture(B).replay()
                logits = d["logits"].clone().reshape(B, 1, -1)
            else:
                logits = eng.decode_step(B).clone().reshape(B, 1, -1)
            eng.past = past + 1
            labels_new = None
        loss = None
        if labels is not None and past_key_values is None:
            lab = labels_new.to(logits.device)
            loss = torch.nn.functional.cross_entropy(logits[:, :-1].reshape(-1, logits.shape[-1]).float(), lab[:, 1:].reshape(-1),
                                                     ignore_index=IGNORE_INDEX)
        pkv = self._kv_tuple(eng.past) if use_cache else None
        if not return_dict:
            out = (logits, pkv)
            return (loss,) + out if loss is not None else out
        return CausalLMOutputWithPast(loss=loss, logits=logits, past_key_values=pkv, hidden_states=(None, vis_outputs), attentions=None)

    __call__ = forward

    # ------------------------------------------------------------------ greedy generate (HF greedy_search contract)
    @torch.no_grad()
    def generate(self, input_ids, images=None, refer_boxes=None, ground_boxes=None, use_cache=True, do_sample=False,
                 max_new_tokens=None, return_dict_in_generate=False, output_hidden_states=False, generation_config=None,
                 eos_token_id=None, _selected_override=None, **kwargs):
        if do_sample:
            raise NotImplementedError("the path is greedy decoding (eval scripts use do_sample=False)")
        gc = generation_config or self.generation_config
        if max_new_tokens is None:
            max_new_tokens = getattr(gc, "max_new_tokens", None) or 20
        eos_ids = _eos_list(eos_token_id if eos_token_id is not None else getattr(gc, "eos_token_id", None))
        pad_id = getattr(gc, "pad_token_id", None)
        eng = self.engine
        dev = eng.dev
        x, ids_new, _, mask, vis_outputs, aux = self._prefill_inputs(input_ids, images, refer_boxes, ground_boxes, None, _selected_override)
        B, T = ids_new.shape
        eng.ensure_rope(T + max_new_tokens)        # HF's rotary cache extends on demand; ours is rebuilt before the kernels index it
        eng.alloc_kv(B, T + max_new_tokens)
        kv_len = mask.sum(1).to(torch.int32).to(dev)
        self._last = dict(ids=ids_new, mask=mask, aux=aux)
        self._mark("assemble+embed")
        logits = eng.llm_prefill(x, B, T, kv_len, last_only=True)          # [B, V] at the last (padded) position
        self._mark("llm_prefill")
        d = eng._decode_buffers(B)
        G.argmax(logits, out=d["ids"])
        d["pos"].fill_(T)
        d["kv_len"].fill_(T + 1)
        out_tokens = torch.empty((max_new_tokens, B), dtype=torch.int64, device=dev)
        out_tokens[0].copy_(d["ids"])
        self._step_logits = [logits.clone()] if kwargs.get("_keep_logits") else None
        eos_t = torch.tensor(eos_ids, dtype=torch.int64, device=dev) if eos_ids else None
        graph = None
        steps_done = 1
        check_every = 16
        for s in range(1, max_new_tokens):
            if eos_t is not None and (s == 1 or s % check_every == 0):
                # one host sync every `check_every` steps: stop once every row has produced an EOS
                if bool(torch.isin(out_tokens[:steps_done], eos_t).any(0).all()):
                    break
            if self.use_cuda_graph and graph is None and s >= 2:
                graph = self._capture(B)
            if graph is not None:
                graph.replay()
            else:
                eng.decode_step(B)
            out_tokens[s].copy_(d["ids"])
            if self._step_logits is not None:
                self._step_logits.append(d["logits"].clone())
            steps_done = s + 1
        self._mark("decode")
        eng.past = T + steps_done - 1
        new = out_tokens[:steps_done].t().contiguous()
        if eos_t is not None:
            # HF greedy_search semantics: a row that has emitted EOS is fed / reported as pad_token_id from then on, and
            # generation ends with the step at which the last unfinished row emits its EOS
            if pad_id is None:
                pad_id = self.pad_token_id if self.pad_token_id is not None else eos_ids[0]
            is_eos = torch.isin(new, eos_t)
            after = (is_eos.cumsum(1) - is_eos.long()) > 0
            new = torch.where(after, torch.full_like(new, pad_id), new)
            finished_at = torch.where(is_eos.any(1), is_eos.float().argmax(1) + 1, torch.full((B,), new.shape[1], device=dev))
            new = new[:, :int(finished_at.max())]
        sequences = torch.cat([input_ids.to(dev), new], 1)
        if not return_dict_in_generate:
            return sequences
        return GenerateOutput(sequences=sequences, hidden_states=((None, vis_outputs),) if output_hidden_states else (),
                              past_key_values=self._kv_tuple(eng.past) if use_cache else None)

    def _capture(self, B: int):
        """Capture one decode step (all 32 layers + heads + argmax + position advance) into a CUDA graph."""
        eng = self.engine
        key = (B, eng.kv.data_ptr(), eng.kv_cap, eng.rope_cos.data_ptr())
        if self._graph is not None and self._graph[0] == key:
            return self._graph[1]
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        d = eng._decode_buffers(B)
        saved = {k: d[k].clone() for k in ("ids", "pos", "kv_len")}
        l0 = G.LAUNCHES
        with torch.cuda.stream(s):
            # thread_local: NCCL's watchdog thread may touch the CUDA API while this thread captures
            with torch.cuda.graph(g, stream=s, capture_error_mode="thread_local"):
                eng.decode_step(B)
        self._graph_kernels = G.LAUNCHES - l0
        torch.cuda.current_stream().wait_stream(s)
        for k, v in saved.items():      # capture does not execute; restore just in case of warm-up side effects
            d[k].copy_(v)
        self._graph = (key, g)
        return g


try:
    AutoConfig.register("groma", GromaConfig)
    AutoModel.register(GromaConfig, GromaModel)
except ValueError:
    pass
