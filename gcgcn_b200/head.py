"""Everything GCGCN computes between ``context_output`` and the logits (/root/reference/models/GCGCN_glove.py:293-358)
for a ragged batch of documents, on the GPU, from the wire format: mention->entity pooling, two hops of
(edge-feature producer -> graph block), the classifier-side pair features and the relation classifier.

``GraphHead`` uses the reference model's own attribute names, so the corresponding slice of a ``GCGCN_glove``
``state_dict`` loads unchanged (everything except the encoder: word_emb, entity_embed, rnn, linear_re).
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np
import torch
from torch import nn

from . import _lib
from .batch import PairTables, PoolTable, RaggedBatch, node_relative_pos
from .classifier import pair_bce_loss, relation_logits
from .edgefeat import EdgeFeatures, EdgeTables
from .functional import EdgeMeanFn, LinearFn
from .modules import HIDDEN, GraphBlocks, pair_dense, pool_nodes


class HeadBatch:
    """Host-built tables of one ragged batch (built once per batch; every array is tiny next to the tensors):
    the batch descriptor, the pooling CSR, the active-slot tables of the edge-feature producer, the pair index
    tables and the entity types.  ``docs`` are ``featurize.WireDoc`` objects."""

    def __init__(self, docs: Sequence, device):
        self.device = torch.device(device)
        self.docs = list(docs)
        self.batch = RaggedBatch([d.n for d in docs], self.device)
        self.pool = PoolTable.from_spans([d.spans for d in docs], [d.length for d in docs], device=self.device)
        self.edge = EdgeTables(docs, self.batch, self.device)
        self.pairs = PairTables(self.batch, [node_relative_pos(d.first_pos) for d in docs], device=self.device)
        self.node_type = torch.from_numpy(np.concatenate([np.asarray(d.node_type, dtype=np.int64) for d in docs])
                                          if docs else np.zeros(0, np.int64)).to(self.device)
        self.total_tokens = self.pool.total_tokens
        # entities pooled and the producer's active context rows fetched in ONE pass over context_output
        self.pool_and_active = PoolTable.concat(self.pool, self.edge.gather, self.device)

    @property
    def wire_nbytes(self) -> int:
        return sum(d.nbytes for d in self.docs)


class GraphHead(nn.Module):
    """``GraphHead()`` = GCGCN_glove's head (G:250-279); ``GraphHead(4, 4, cls_dim=768)`` = the BERT variant's
    (models/GraphCNN_multihead_bert_gate_cls.py:247-267), which adds ``linear_cls`` on BERT's first-token feature."""

    def __init__(self, layer_num=2, head_num=8, relation_num=97, dis_size=20, dis_num=21, entity_type_size=20,
                 hidden_size=HIDDEN, graph_hop=2, cls_dim: int = 0):
        super().__init__()
        blocks = GraphBlocks(layer_num, head_num, hidden_size=hidden_size, graph_hop=graph_hop, overlap=False)
        # the graph modules under the reference model's attribute names (G:254-262)
        self.get_weighted_adj_matrix = blocks.get_weighted_adj_matrix
        self.get_adj_matrix = blocks.get_adj_matrix
        self.graphcnn = blocks.graphcnn
        object.__setattr__(self, "_blocks", blocks)            # shares the modules above; not registered twice
        edge = EdgeFeatures(hidden_size, dis_size, graph_hop)
        self.word_attention = edge.word_attention              # G:266-269
        self.sentence_attention = edge.sentence_attention
        self.linear_word_att = edge.linear_word_att
        self.linear_sentence_att = edge.linear_sentence_att
        object.__setattr__(self, "_edge", edge)
        self.dense_layer = nn.Linear(hidden_size * (graph_hop + 1) + dis_size + entity_type_size, hidden_size)   # G:272
        self.bili_layer_01 = nn.Bilinear(hidden_size, hidden_size, relation_num)                                 # G:275
        self.classification_layer_01 = nn.Linear(hidden_size * 2, relation_num)                                  # G:276
        if cls_dim:
            self.linear_cls = nn.Linear(cls_dim, relation_num)                                                   # B:265
        self.dis_embed = nn.Embedding(dis_num, dis_size)                                                         # G:279
        self.ner_emb = nn.Embedding(7, entity_type_size, padding_idx=0)                                          # G:242

    def train(self, mode: bool = True):
        super().train(mode)
        self._blocks.train(mode)
        return self

    def forward(self, context: torch.Tensor, hb: HeadBatch, edge_dtype=torch.float32, labels: Optional[torch.Tensor] = None,
                cls_feat: Optional[torch.Tensor] = None, classifier_dtype=torch.float32):
        """context [total_tokens, 128] = ``context_output`` of every document back to back; cls_feat [num_docs, cls_dim]
        = BERT's first-token feature of every document (BERT variant only, B:277).  ``classifier_dtype`` is the operand
        type of the relation classifier's bilinear form (torch.float32 or torch.bfloat16, ``classifier.relation_logits``);
        parameters and their gradients stay fp32.  Returns a dict with x0, e0, y1, e1, y2, entity_feature_h / _t,
        logits [total_pairs, R] and, given labels, the per-document loss."""
        if classifier_dtype not in (torch.float32, torch.bfloat16):
            raise _lib.GcgcnError(f"GraphHead: classifier_dtype must be torch.float32 or torch.bfloat16, got {classifier_dtype}")
        if not context.is_cuda:
            raise _lib.GcgcnError("GraphHead: gcgcn_b200 runs on CUDA only (no CPU fallback)")
        bt, blocks, edge = hb.batch, self._blocks, self._edge
        dis = self.dis_embed.weight
        rows = pool_nodes(context, hb.pool_and_active)                                 # G:297-298 + the rows G:300 reads
        x0, ctx_act = rows[:bt.total_nodes], rows[bt.total_nodes:]
        e0 = edge(0, None, x0, dis, hb.edge, edge_dtype, ctx_act)                      # G:313-326, i = 0
        y1, a0 = blocks.hop0(x0, e0, bt)                                               # G:330-341
        e1 = edge(1, None, y1, dis, hb.edge, edge_dtype, ctx_act)                      # G:313-326, i = 1
        y2, a1 = blocks.hop1(y1, e1, bt)                                               # G:336-341 (dead for the logits, G:338)
        type_feats = nn.functional.embedding(hb.node_type, self.ner_emb.weight, padding_idx=0)
        feats = torch.cat([x0, x0, y1, type_feats], 1)                                 # G:343-347: cat[x0, x0, y1, type]
        fh, ft = pair_dense(feats, self.dense_layer, dis, hb.pairs, bt)                # G:351-355
        cls_feature = None
        if hasattr(self, "linear_cls"):
            if cls_feat is None:
                raise _lib.GcgcnError("GraphHead(cls_dim=...) needs cls_feat [num_docs, cls_dim] (B:277)")
            cls_feature = LinearFn.apply(cls_feat, self.linear_cls.weight, self.linear_cls.bias)              # B:346
        logits = relation_logits(fh, ft, self.bili_layer_01, self.classification_layer_01, cls_feature, bt,
                                 dtype=classifier_dtype)                                               # G:356-358
        out = {"x0": x0, "e0": e0, "y1": y1, "e1": e1, "y2": y2, "a0": a0, "a1": a1, "entity_feature_h": fh,
               "entity_feature_t": ft, "logits": logits}
        if labels is not None:
            out["loss"] = pair_bce_loss(logits, labels, bt)                            # C:355-364
        return out
