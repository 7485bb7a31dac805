import os, sys, torch, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from devis_b200 import synthetic, clip_geometry
torch.manual_seed(0)
def analyse(sigma, label, frames=(2,), heads=(0,3)):
    clip = synthetic.make_clip(dist="local", device="cpu", seed=100, sigma_px=sigma)
    shapes = clip["shapes"]; L=len(shapes)
    geom = clip_geometry.ClipGeometry(shapes, 6, clip["frame_table"])
    order = geom.tile_order("cpu", 8, 8).numpy()
    S = geom.spatial_size
    tot_live = np.zeros(L); tot_rows_tile64 = np.zeros(L); tot_rows_cta16 = np.zeros(L); tot_pair = np.zeros(L); tot_warp=np.zeros(L)
    for t in frames:
        for m in heads:
            for seg, loc in (("c", clip["loc_curr"]), ("t", clip["loc_temporal"])):
                nslots = loc.shape[3]
                for s in range(nslots):
                    l = s % L
                    H, W = shapes[l]
                    xy = loc[t,:,m,s].numpy().astype(np.float32)   # (S, P, 2)
                    x = xy[...,0]*np.float32(W) - np.float32(0.5); y = xy[...,1]*np.float32(H) - np.float32(0.5)
                    inr = (x>-1)&(y>-1)&(x<W)&(y<H)
                    x0=np.floor(x).astype(int); y0=np.floor(y).astype(int)
                    rows=[]; live=[]
                    for dy in (0,1):
                        for dx in (0,1):
                            xx=x0+dx; yy=y0+dy
                            ok = inr & (xx>=0)&(xx<W)&(yy>=0)&(yy<H)
                            rows.append(np.where(ok, yy*W+xx, -1)); live.append(ok)
                    rows=np.stack(rows,-1)   # (S,P,4)
                    rows_o = rows[order]      # tile order
                    tot_live[l] += (rows>=0).sum()
                    # distinct rows per 64-query tile and per 16-query CTA, in tile order
                    for chunk, acc in ((64, tot_rows_tile64), (16, tot_rows_cta16), (4, tot_warp)):
                        n = (S + chunk-1)//chunk
                        for c in range(n):
                            r = rows_o[c*chunk:(c+1)*chunk].reshape(-1)
                            r = r[r>=0]
                            acc[l] += len(np.unique(r))
                    # QPG=2 x-adjacent pair: queries (2i, 2i+1) in tile order rows of 8 -> x-adjacent; same point index: TR(q)==TL(q+1), BR(q)==BL(q+1)
                    a = rows_o[0:(S//2)*2:2]; b = rows_o[1:(S//2)*2:2]
                    tot_pair[l] += ((a[...,1]==b[...,0])&(a[...,1]>=0)).sum() + ((a[...,3]==b[...,2])&(a[...,3]>=0)).sum()
    print(label)
    for l in range(L):
        print(f"  target level {l} {shapes[l]}: live corners {tot_live[l]:.0f}  share {tot_live[l]/tot_live.sum():.3f}  distinct rows per 64-q tile: {tot_rows_tile64[l]:.0f} (x{tot_live[l]/max(tot_rows_tile64[l],1):.2f} fewer)  per 16-q CTA: x{tot_live[l]/max(tot_rows_cta16[l],1):.2f}  per warp (4 q): x{tot_live[l]/max(tot_warp[l],1):.2f}  in-register pair merge removes {tot_pair[l]/tot_live[l]*100:.2f} %")
    print(f"  all levels: tile64 x{tot_live.sum()/tot_rows_tile64.sum():.2f}, cta16 x{tot_live.sum()/tot_rows_cta16.sum():.2f}, warp x{tot_live.sum()/tot_warp.sum():.2f}, pair merge {tot_pair.sum()/tot_live.sum()*100:.2f} %")
analyse(2.0, "D-local (bench workload): ray (i+1) px + N(0, 2 px)")
analyse(0.0, "at-init pattern: ray (i+1) px, no jitter")
analyse(0.5, "ray + N(0, 0.5 px)")
