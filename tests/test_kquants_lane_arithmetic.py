"""The lane arithmetic of llm_b200/csrc/kquants.cu restated word for word in Python (uint32 shifts / masks, dp4a with signed bytes, the xor-shuffle
reductions, lane = 8 * part + L) and checked against oracle/kquants_np.py, which tests/test_oracle_kquants.py pins to the reference's compiled k_quants.c.
CPU only: it guards the index / mask expressions of the CUDA kernel (all five K-quant types) independently of a GPU run."""
import os

import numpy as np
import pytest

from oracle import bindings as B
from oracle import kquants_np as KN

from conftest import GOLDEN

f32 = np.float32
M = 0xffffffff
def s8(b): return b-256 if b>=128 else b
def dp4a(a,b,c):
    a&=M; b&=M
    return c+sum(s8((a>>(8*i))&255)*s8((b>>(8*i))&255) for i in range(4))
def u32(buf,off): return int(buf[off])|int(buf[off+1])<<8|int(buf[off+2])<<16|int(buf[off+3])<<24
def k4_scale(q,j): return (q[j]&63) if j<4 else ((q[j+4]&0xF)|((q[j-4]>>6)<<4))
def k4_min(q,j): return (q[j+4]&63) if j<4 else ((q[j+4]>>4)|((q[j]>>6)<<4))
BYTES={10:84,11:110,12:144,13:176,14:210}; QS={10:16,11:32,12:16,13:48,14:0}; QH={13:16}
def kernel_row(t,wrow,xblocks):
    nsb=len(xblocks); acc=[f32(0)]*32; accm=[f32(0)]*32
    for i in range(nsb):
        wb=[int(v) for v in wrow[i*BYTES[t]:(i+1)*BYTES[t]]]; raw=wrow[i*BYTES[t]:(i+1)*BYTES[t]]
        yd,q8,bs=xblocks[i]; qsb=[int(v)&255 for v in q8.astype(np.int8).view(np.uint8)]
        h2f=lambda o: f32(np.frombuffer(bytes(raw[o:o+2]),np.float16)[0])
        pl=[0]*32
        for lane in range(32):
            L=lane&7; part=lane>>3
            if t in (10,11):
                j=part>>1
                if t==10:
                    d=f32(yd*h2f(80)); dmin=f32(f32(-yd)*h2f(82))
                    prod=(wb[2*L]>>4)*int(bs[2*L])+(wb[2*L+1]>>4)*int(bs[2*L+1])
                    acc[lane]=KN._fma(dmin,f32(prod),acc[lane])
                    w=u32(wb,16+32*j+4*L); hm=0
                else:
                    d=f32(yd*h2f(108)); hm=u32(wb,4*L); w=u32(wb,32+32*j+4*L)
                p=0
                for kk in range(2):
                    k=2*(part&1)+kk; si=8*j+2*k+(1 if L>=4 else 0)
                    lo=(w>>(2*k))&0x03030303
                    xw=u32(qsb,128*j+32*k+4*L)
                    if t==10: p+=(wb[si]&0xF)*dp4a(lo,xw,0)
                    else:
                        q3h=(((~(hm>>(4*j+k)))&M)&0x01010101)<<2
                        s=wb[96:108]; wd=si>>2; c=si&3
                        sc=(((s[(wd&1)*4+c]>>(4*(wd>>1)))&0xF)|(((s[8+c]>>(2*wd))&3)<<4))-32
                        p+=sc*(dp4a(lo,xw,0)-dp4a(q3h,xw,0))
                pl[lane]=p
            elif t==14:
                d=f32(yd*h2f(208)); j=part>>1; hs=part&1
                wl=u32(wb,64*j+32*hs+4*L); wh=u32(wb,128+32*j+4*L); p=0
                for kk in range(2):
                    k=hs+2*kk
                    nib=((wl>>4) if kk else wl)&0x0F0F0F0F
                    q=nib|(((wh>>(2*k))&0x03030303)<<4)
                    xw=u32(qsb,128*j+32*k+4*L)
                    dot=dp4a(q,xw,0)-32*dp4a(0x01010101,xw,0)
                    p+=s8(wb[192+2*(4*j+k)+(1 if L>=4 else 0)])*dot
                pl[lane]=p
            else:
                d=f32(yd*h2f(0)); dmin=f32(f32(-yd)*h2f(2)); scq=wb[4:16]
                w=u32(wb,QS[t]+32*part+4*L); lo=w&0x0F0F0F0F; hi=(w>>4)&0x0F0F0F0F
                if t==13:
                    hb=u32(wb,QH[t]+4*L); lo|=((hb>>(2*part))&0x01010101)<<4; hi|=((hb>>(2*part+1))&0x01010101)<<4
                x0=u32(qsb,64*part+4*L); x1=u32(qsb,64*part+32+4*L)
                pl[lane]=k4_scale(scq,2*part)*dp4a(lo,x0,0)+k4_scale(scq,2*part+1)*dp4a(hi,x1,0)
                tt=lane&3
                q8a=int(np.int16(int(bs[4*tt])+int(bs[4*tt+1]))); q8b=int(np.int16(int(bs[4*tt+2])+int(bs[4*tt+3])))
                accm[lane]=k4_min(scq,2*tt)*q8a+k4_min(scq,2*tt+1)*q8b      # prod (int) for now
        # shuffles: p += xor 8, xor 16
        ps=[pl[l]+pl[l^8] for l in range(32)]; ps=[ps[l]+ps[l^16] for l in range(32)]
        for lane in range(32): acc[lane]=KN._fma(d,f32(ps[lane]),acc[lane])
        if t in (12,13):
            prod=[accm[l] for l in range(32)]
            if t==13:
                prod=[prod[l]+prod[l^1] for l in range(32)]; prod=[prod[l]+prod[l^2] for l in range(32)]
            if i==0: am=[f32(0)]*32
            am=[KN._fma(dmin,f32(prod[l]),am[l]) for l in range(32)]
    v=list(acc)
    for o in (4,2,1): v=[f32(v[l]+v[l^o]) for l in range(32)]
    if t==12:
        for o in (2,1): am=[f32(am[l]+am[l^o]) for l in range(32)]
    if t in (12,13): v=[f32(v[l]+am[l]) for l in range(32)]
    return v[0]


def lane_inputs():
    rng = np.random.default_rng(5)
    K = 512
    x = (rng.standard_normal((2, K)) * rng.uniform(0.1, 5, (2, 1))).astype(f32)
    x[1] = np.round(x[1] * 4) / 4
    w = (rng.standard_normal((3, K)) / 22).astype(f32)
    w[:, :16] *= 8
    return x, w


@pytest.mark.parametrize("name,t", list(B.KQUANT_TYPES.items()))
def test_kernel_lane_arithmetic_matches_the_pinned_restatement(name, t):
    x, _ = lane_inputs()
    wq = np.load(os.path.join(GOLDEN, "kquants_ref.npz"))[f"lane_{name}_wq"]      # the reference's quantize_row_{name} of lane_inputs()'s w
    for b in range(2):
        xq = KN.quantize_row_q8_K(x[b])
        for n in range(3):
            got, want = f32(kernel_row(t, wq[n], xq)), KN.vec_dot(t, wq[n], xq)
            assert got.view(np.uint32) == want.view(np.uint32), (name, b, n, got, want)
