"""Reference for the stage-1 step whose teacher sees the clip at another resolution (run_stage1.py:360-377: the teacher's copy of
the clip is resized, bicubic, align_corners=False; the student keeps the clip as it is), composed from the oracle's own pieces."""
import torch
import torch.nn.functional as F

from oracle import unite_oracle as O


def resize_for_teacher(videos, R):
    """[B,C,T,H,W] -> [B,C,T,R,R] as the reference's engine resizes the teacher's copy; the clip itself when R == H == W."""
    B, C, T, H, W = videos.shape
    if R == H and R == W:
        return videos
    return F.interpolate(videos.view(B, C * T, H, W), size=(R, R), mode="bicubic", align_corners=False).view(B, C, T, R, R)


def stage1_step_at(student_sd, teacher_sd, videos, q, scfg, tcfg, R, mask_ratio=0.8, with_grads=True):
    """oracle.stage1_step for the shipped loss ('l2', clip_loss_data 'mixed'), with the teacher fed resize_for_teacher(videos, R).
    Same keys as oracle.stage1_step."""
    B = videos.shape[0]
    with torch.no_grad():
        feat, attn = O.teacher_forward(teacher_sd, resize_for_teacher(videos, R), tcfg)
        mask = O.multinomial_mask(attn, q, mask_ratio, B)
        K, C = feat.shape[0], feat.shape[-1]
        targets = feat[~mask.unsqueeze(0).repeat(K, 1, 1)].reshape(K, B, -1, C)
    params = {k: v.detach().clone().requires_grad_(with_grads) for k, v in student_sd.items()}
    out = O.student_forward(params, videos, mask, scfg, clip_only=True)
    loss = O.alignment_loss(out, targets, "l2")
    res = dict(attn=attn, mask=mask, vis_idx=O.visible_indices(mask), targets=targets, outputs=out.detach(), loss=loss.detach())
    if with_grads:
        loss.backward()
        grads = {k: v.grad for k, v in params.items() if v.grad is not None}
        res["grads"] = grads
        res["grad_norm"] = torch.norm(torch.stack([g.norm(2) for g in grads.values()]), 2)
    return res
