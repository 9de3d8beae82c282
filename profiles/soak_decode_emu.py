"""CPU soak of the decoder logic shared with the kernels (tests/emu build): random sizes, qualities, contents, chroma layouts
(4:4:4 / 4:2:2 / 4:2:0), restart intervals and optimised Huffman tables against Pillow and OpenCV. Development aid."""
import io, sys, ctypes, numpy as np, cv2
import os; ROOT=os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0,ROOT); sys.path.insert(0,os.path.join(ROOT,'tests'))
from PIL import Image
import test_jpeg_emu as T
libs=[T.Emu(T._build("full",[]),0), T.Emu(T._build("tiny",T.TINY),0)]
rng=np.random.default_rng(123)
bad=0; n=0
for it in range(700):
    h=int(rng.integers(1,140)); w=int(rng.integers(1,180)); q=int(rng.integers(1,101))
    kind=it%4
    if kind==0: img=rng.integers(0,256,(h,w,3),dtype=np.uint8)
    elif kind==1: img=cv2.GaussianBlur(rng.integers(0,256,(h,w,3),dtype=np.uint8),(0,0),2.0)
    elif kind==2: img=np.full((h,w,3),int(rng.integers(256)),np.uint8)
    else: img=np.where(rng.integers(0,2,(h,w,3))>0,255,0).astype(np.uint8)
    ss=int(rng.integers(0,3)); kw={}
    r=int(rng.integers(0,4))
    if r==1: kw={"restart_marker_blocks":int(rng.integers(1,40))}
    elif r==2: kw={"restart_marker_rows":int(rng.integers(1,4))}
    if it%7==0: kw["optimize"]=True
    buf=io.BytesIO(); Image.fromarray(img).save(buf,"JPEG",quality=q,subsampling=ss,**kw); data=buf.getvalue()
    ref=np.asarray(Image.open(io.BytesIO(data)).convert("RGB")); g=cv2.imdecode(np.frombuffer(data,np.uint8),cv2.IMREAD_GRAYSCALE)
    for lib in libs:
        n+=1
        try:
            out=T.emu_decode(lib,data)
            if not (np.array_equal(out["rgb"],ref) and np.array_equal(out["gray"],g)): bad+=1; print("MISMATCH",h,w,q,ss,kw)
        except Exception as e:
            bad+=1; print("ERR",h,w,q,ss,kw,e)
print("cases",n,"bad",bad)
