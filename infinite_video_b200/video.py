"""Model-level chunk loop of the LTM path (SURVEY.md section 8f N2).

In the reference the loop over the chunks of a video lives in the eval scripts: they call the video Q-former once per
chunk with `new_video=(chunk == 0)` (infty-Video-LLaMA/InfVideoLLaMA/models/infinityqa.py:280-344 `encode_video`,
infty-VideoChat2/models/videochat2_it_mistral.py:181-253 `encode_img`) and keep a running mean of the chunk embeddings
(eval_code/eval/run_inference_inf_video_llama_nextqa.py:194).  Inside the Q-former every LTM layer (2 in
Video-LLaMA, 6 in VideoChat2) is handed the SAME `encoder_hidden_states` and pools its frames again
(long_term_attention_gibbs.py:304).

`consolidate_video` is that loop for a batch of independent videos and all LTM layers at once:
  * the frames of a chunk are pooled ONCE (25 MB per video at the NExT-QA shape) and shared by every layer;
  * the pooling of chunk c+1 runs on a side stream while the layers consolidate chunk c;
  * chunks of a video stay strictly sequential, videos and layers are independent.

`split_videos` cuts whole videos of different lengths into those chunks as views, so that every chunk is pooled where
it lives, with no padded batch built first.
"""
import torch

from .batched import BatchedRectLTM, _Entries


def split_videos(videos, frames_per_chunk, tokens_per_frame):
    """videos: Bv tensors [F_v*T, e], whole videos of F_v frames of T = tokens_per_frame tokens.  Returns the chunks
    `chunks[c][v]` for `consolidate_video` / `BatchedRectLTM.step` (with chunk_frames=frames_per_chunk): chunk c of
    video v is the view `videos[v][c*L*T : (c+1)*L*T]` (L = frames_per_chunk; nothing is copied), None once the video
    has ended.  A video whose last chunk would hold a single frame is refused (chunks of one frame are not supported)."""
    L, T = int(frames_per_chunk), int(tokens_per_frame)
    if L < 2 or T < 1:
        raise ValueError("frames_per_chunk must be >= 2 and tokens_per_frame >= 1")
    frames = []
    for v, x in enumerate(videos):
        if x.dim() != 2 or x.shape[0] % T or x.shape[0] == 0:
            raise ValueError(f"video {v} must be [F*{T}, e] with F >= 1, not {list(x.shape)}")
        F = x.shape[0] // T
        if F % L == 1:
            raise ValueError(f"video {v} has {F} frames: its last chunk of {L} would hold one frame (not supported)")
        frames.append(F)
    C = max(-(-F // L) for F in frames) if frames else 0
    return [[x[c * L * T:(c + 1) * L * T] if c * L < F else None for x, F in zip(videos, frames)] for c in range(C)]


@torch.no_grad()
def consolidate_video(engines, chunks, queries, uniforms=None, new_doc=True, reduce=None, lengths=None,
                      chunk_frames=None):
    """engines:  one `BatchedRectLTM` per LTM layer (same device, same chunk geometry).
    chunks:   C tensors [Bv, L*T, e] -- the `encoder_hidden_states` of each chunk, in order -- or per-video lists (see
              `BatchedRectLTM.step`, `split_videos`) with `chunk_frames` = L: each video's frames are read where they
              live, and the lengths follow from the entries (None = the video has ended).
    queries:  `queries[layer][c]` tensors [Bv, Q, D], or a callable `queries(layer, c, prev)` returning that tensor
              (`prev` = context of the previous layer for this chunk, None for the first layer): in the Q-former the
              queries of a layer depend on the output of the layer before it.
    uniforms: `uniforms[layer][c]` float64 [Bv, 512] for c >= 1 (sticky engines); None entries allowed at c == 0.
    new_doc:  whether chunk 0 starts a new document for every video.
    reduce:   None -> `ctx[layer][c]`;  "mean" -> running mean over the chunks, `ctx[layer]` [Bv, Q, D].
    lengths:  videos of different lengths: `lengths[c]` holds Bv host ints, the frames video v has in chunk c (its
              chunk padded to L frames; 0 once the video has ended -- its memory is kept and its ctx rows are zero).
              "mean" then divides each video by the number of chunks it actually had.
    """
    if not engines or any(not isinstance(e, BatchedRectLTM) for e in engines):
        raise ValueError("consolidate_video takes a list of BatchedRectLTM engines (one per LTM layer)")
    dev = engines[0].device
    if any(e.device != dev or e.T != engines[0].T or e.e != engines[0].e for e in engines):
        raise ValueError("all layers must live on one device and share the chunk geometry")
    if reduce not in (None, "mean"):
        raise ValueError("reduce must be None or 'mean'")
    C = len(chunks)
    if lengths is not None and len(lengths) != C:
        raise ValueError("lengths must hold one entry per chunk")
    lens = [None] * C if lengths is None else lengths
    pool_eng = engines[0]
    # a chunk given per video is checked once and handed on in checked form to the pooling and every layer's step
    chunks = [pool_eng._entries(ch, chunk_frames, lens[c]) if isinstance(ch, (list, tuple)) else ch
              for c, ch in enumerate(chunks)]
    # which videos each chunk holds (None: all of them)
    present = [[x > 0 for x in ch.lens] if isinstance(ch, _Entries) else None if lens[c] is None
               else [int(x) > 0 for x in lens[c]] for c, ch in enumerate(chunks)]
    with torch.cuda.device(dev):
        main = torch.cuda.current_stream(dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(main)                                    # the chunks were produced on the caller's stream
        pooled, ready = [None] * C, [None] * C

        def pool_ahead(c):
            with torch.cuda.stream(side):
                pooled[c] = pool_eng.pool(chunks[c], lengths=lens[c])
                ready[c] = torch.cuda.Event()
                ready[c].record(side)

        pool_ahead(0)
        out = [[] for _ in engines]
        acc = [None] * len(engines)
        for c in range(C):
            main.wait_event(ready[c])
            pooled[c].record_stream(main)
            if c + 1 < C:
                pool_ahead(c + 1)
            prev = None
            for li, eng in enumerate(engines):
                q = queries(li, c, prev) if callable(queries) else queries[li][c]
                u = None if uniforms is None else uniforms[li][c]
                ctx = eng.step(chunks[c], q, u if c > 0 or not new_doc else None, new_doc=(new_doc and c == 0),
                               pooled=pooled[c], beside_pooling=(c + 1 < C), lengths=lens[c])
                prev = ctx
                if reduce == "mean":
                    acc[li] = ctx.clone() if acc[li] is None else acc[li].add_(ctx)
                else:
                    out[li].append(ctx)
            pooled[c] = None
        if reduce == "mean":
            if all(p is None for p in present):
                return [a / C for a in acc]
            Bv = acc[0].shape[0]
            had = torch.as_tensor([[True] * Bv if p is None else p for p in present]).sum(0).clamp_min(1)
            return [a / had.to(dev, a.dtype).view(-1, 1, 1) for a in acc]
        return out
