"""The cases behind tests/golden/filters_golden.json: (reference object, CUDA object, settings, input clip) per case.
Inputs come from handbrake_b200.synth only, so the same clips can be rebuilt on a machine without the reference."""
import numpy as np

from handbrake_b200 import synth

FMT = {8: synth.PIX_FMT_YUV420P, 10: synth.PIX_FMT_YUV420P10}


def _mixed_interlaced(fmt, w, h, n, seed):
    frames = list(synth.interlaced_clip(fmt, w, h, n, seed=seed)) + list(synth.progressive_clip(fmt, w, h, 3, seed=seed + 1, noise=3))
    return np.stack(frames)


def _decomb_inputs(depth, w, h, n, seed):
    clip = _mixed_interlaced(FMT[depth], w, h, n, seed)
    k = clip.shape[0]
    flags = np.array([synth.PIC_FLAG_TOP_FIELD_FIRST if i % 4 != 3 else 0 for i in range(k)], np.uint16)
    flags[k - 1] = synth.PIC_FLAG_PROGRESSIVE_FRAME
    combed = np.array([(2, 1, 0, 2, 1)[i % 5] for i in range(k)], np.uint8)
    return clip, flags, combed


def cases():
    """name -> dict(ref=[objects], cuda=[objects], settings=[...], depth, w, h, clip, flags, combed)"""
    out = {}

    def add(name, ref, cuda, settings, depth, w, h, clip, flags=None, combed=None):
        as_list = lambda v: v if isinstance(v, list) else [v]
        out[name] = dict(ref=as_list(ref), cuda=as_list(cuda), settings=as_list(settings), depth=depth, w=w, h=h, clip=clip, flags=flags, combed=combed)

    for depth in (8, 10):
        w, h = 176, 112
        clip = _mixed_interlaced(FMT[depth], w, h, 9, 12345)
        tff = np.full(clip.shape[0], synth.PIC_FLAG_TOP_FIELD_FIRST, np.uint16)
        add(f"comb_detect_default_{depth}", "hb_filter_comb_detect", "hb_filter_comb_detect_cuda",
            "mode=3:spatial-metric=2:motion-thresh=1:spatial-thresh=1:filter-mode=2:block-thresh=40:block-width=16:block-height=16", depth, w, h, clip, tff)
        add(f"comb_detect_fast_{depth}", "hb_filter_comb_detect", "hb_filter_comb_detect_cuda",
            "mode=0:spatial-metric=2:motion-thresh=2:spatial-thresh=3:filter-mode=1:block-thresh=80", depth, w, h, clip, tff)

        w, h = 200, 106
        clip, flags, combed = _decomb_inputs(depth, w, h, 7, 5)
        add(f"decomb_yadif_blend_cubic_{depth}", "hb_filter_decomb", "hb_filter_decomb_cuda", "mode=7", depth, w, h, clip, flags, combed)
        add(f"decomb_bob_{depth}", "hb_filter_decomb", "hb_filter_decomb_cuda", "mode=23", depth, w, h, clip, flags)
        add(f"decomb_selective_{depth}", "hb_filter_decomb", "hb_filter_decomb_cuda", "mode=39", depth, w, h, clip, flags, combed)
        w, h = 208, 120
        clip, flags, combed = _decomb_inputs(depth, w, h, 6, 11)
        add(f"decomb_eedi2bob_{depth}", "hb_filter_decomb", "hb_filter_decomb_cuda", "mode=31", depth, w, h, clip, flags)
        add(f"decomb_eedi2_selective_{depth}", "hb_filter_decomb", "hb_filter_decomb_cuda", "mode=63", depth, w, h, clip, flags, combed)
        # the chain libhb builds: comb_detect tags, decomb acts on the tags
        w, h = 320, 180
        clip, flags, _ = _decomb_inputs(depth, w, h, 8, 9)
        add(f"chain_comb_detect_decomb_{depth}", ["hb_filter_comb_detect", "hb_filter_decomb"], ["hb_filter_comb_detect_cuda", "hb_filter_decomb_cuda"],
            [None, "mode=39"], depth, w, h, clip, flags)

        w, h = 200, 90
        clip = synth.progressive_clip(FMT[depth], w, h, 4, seed=31, noise=20)
        add(f"lapsharp_medium_{depth}", "hb_filter_lapsharp_mt", "hb_filter_lapsharp_cuda", "y-strength=0.2:y-kernel=isolap", depth, w, h, clip)
        add(f"lapsharp_mixed_{depth}", "hb_filter_lapsharp_mt", "hb_filter_lapsharp_cuda", "y-strength=1.1:y-kernel=lap:cb-strength=0.5:cb-kernel=isolog", depth, w, h, clip)
        w, h = 150, 98
        clip = synth.progressive_clip(FMT[depth], w, h, 3, seed=51)
        add(f"unsharp_default_{depth}", "hb_filter_unsharp_mt", "hb_filter_unsharp_cuda", None, depth, w, h, clip)
        add(f"unsharp_size15_{depth}", "hb_filter_unsharp_mt", "hb_filter_unsharp_cuda", "y-strength=1.5:y-size=15:cb-strength=0.3:cb-size=3", depth, w, h, clip)
        add(f"chroma_smooth_{depth}", "hb_filter_chroma_smooth_mt", "hb_filter_chroma_smooth_cuda", "cb-strength=1.2:cb-size=5", depth, w, h, clip)
        w, h = 160, 96
        clip = synth.progressive_clip(FMT[depth], w, h, 6, seed=61, noise=10)
        add(f"hqdn3d_default_{depth}", "hb_filter_denoise", "hb_filter_denoise_cuda", None, depth, w, h, clip)
        add(f"hqdn3d_strong_{depth}", "hb_filter_denoise", "hb_filter_denoise_cuda", "y-spatial=7:cb-spatial=7:cr-spatial=7:y-temporal=7:cb-temporal=5:cr-temporal=5", depth, w, h, clip)
        w, h = 128, 80
        clip = synth.progressive_clip(FMT[depth], w, h, 4, seed=21)
        add(f"nlmeans_prefilter_median_reduce_{depth}", "hb_filter_nlmeans", "hb_filter_nlmeans_cuda", "y-strength=6:y-prefilter=514:threads=1", depth, w, h, clip)
        # range 1 (no spatial displacement, only the temporal ones): chroma inherits it, so all three planes run it
        add(f"nlmeans_range1_{depth}", "hb_filter_nlmeans", "hb_filter_nlmeans_cuda", "y-strength=6:y-range=1:y-frame-count=3", depth, w, h, clip)
        if depth == 8:
            add("nlmeans_range1_luma_8", "hb_filter_nlmeans", "hb_filter_nlmeans_cuda", "y-strength=6:y-range=1:y-frame-count=3:cb-strength=0", depth, w, h, clip)

        w, h = 160, 96
        clip, flags = synth.telecined_clip(FMT[depth], w, h, 16, seed=71)
        add(f"detelecine_hard_{depth}", "hb_filter_detelecine", "hb_filter_detelecine_cuda", None, depth, w, h, clip, flags)
        clip, flags = synth.telecined_clip(FMT[depth], w, h, 12, seed=72, soft=True, tff=False, video_tail=5)
        add(f"detelecine_soft_video_tail_{depth}", "hb_filter_detelecine", "hb_filter_detelecine_cuda", "strict-breaks=1", depth, w, h, clip, flags)
    # BASELINE config 5's chain order (libhb orders by filter id): decomb -> NLMeans medium -> lapsharp
    w, h = 192, 108
    clip, flags, _ = _decomb_inputs(10, w, h, 5, 17)
    add("chain_config5_small_10", ["hb_filter_decomb", "hb_filter_nlmeans", "hb_filter_lapsharp_mt"], ["hb_filter_decomb_cuda", "hb_filter_nlmeans_cuda", "hb_filter_lapsharp_cuda"],
        ["mode=7", "y-strength=6", "y-strength=0.2:y-kernel=isolap"], 10, w, h, clip, flags)
    return out


def digest(result):
    """what is pinned per case: picture digests, timestamps, combed tags"""
    import hashlib
    return dict(sha256=[hashlib.sha256(f.tobytes()).hexdigest() for f in result.frames],
                start=[int(v) for v in result.start], combed=[int(v) for v in result.combed])
