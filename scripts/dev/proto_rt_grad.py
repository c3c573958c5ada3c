import numpy as np, torch, sys, os
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', '..'))
torch.manual_seed(0)
dt=torch.float64
def embed(c):  # even extension per dim
    for d in range(c.dim()):
        idx=[slice(None)]*c.dim(); idx[d]=slice(1,-1)
        c=torch.cat([c, torch.flip(c[tuple(idx)],[d])],dim=d)
    return c
def RT(c, v, dims):
    C=embed(c.view(dims)); D=torch.fft.fftn(C).real.clamp(min=1e-6); s=torch.sqrt(D)
    N=C.shape
    pad=torch.zeros((v.shape[0],)+tuple(N),dtype=dt); pad[(slice(None),)+tuple(slice(0,m) for m in dims)]=v.view((-1,)+dims)
    y=torch.fft.ifftn(s*torch.fft.fftn(pad,dim=tuple(range(1,1+len(dims)))),dim=tuple(range(1,1+len(dims)))).real
    return y.reshape(v.shape[0],-1), D
for dims in [(5,7),(4,3,6),(6,)]:
    M=int(np.prod(dims)); Dn=len(dims)
    # a PSD-ish column: matern-like decay, plus some entries that will clamp
    grids=np.meshgrid(*[np.arange(m) for m in dims],indexing='ij')
    r=np.sqrt(sum((g*0.7)**2 for g in grids))
    c0=torch.tensor(np.exp(-r**2/3.0).reshape(-1),dtype=dt); c0[0]+=1e-3    # sqexp: tiny eigenvalues -> clamps
    c=c0.clone().requires_grad_(True)
    B=3
    v=torch.randn(B,M,dtype=dt); 
    y,D=RT(c,v,dims)
    G=torch.randn_like(y)
    (y*G).sum().backward()
    gref=c.grad.clone()
    nclamp=int((D<=1e-6).sum())
    # ---- my formula
    N=[2*m-2 for m in dims]; Ntot=int(np.prod(N))
    Dm=D[tuple(slice(0,m) for m in dims)]   # unique values on the m-grid
    s=torch.sqrt(Dm)
    mask=(Dm>1e-6).to(dt)
    # symmetrised circular correlation on the N grid, folded to the m grid: qs
    pad=torch.zeros((B,)+tuple(N),dtype=dt); pad[(slice(None),)+tuple(slice(0,m) for m in dims)]=v.view((-1,)+dims)
    Gn=G.view((B,)+tuple(N))
    ax=tuple(range(1,1+Dn))
    q=torch.fft.ifftn(torch.conj(torch.fft.fftn(pad,dim=ax))*torch.fft.fftn(Gn,dim=ax),dim=ax).real.sum(0)   # q[tau]=sum_t v[t] G[t+tau]
    # per-dim reflection average
    qs=q.clone()
    for d in range(Dn):
        idx=(-torch.arange(N[d]))%N[d]
        qs=0.5*(qs+qs.index_select(d,idx))
    qs=qs[tuple(slice(0,m) for m in dims)]
    def dct1(x):   # out[k]=sum_j w_j x[j] cos(pi j k/(m-1)), separable
        for d in range(x.dim()):
            m=x.shape[d]
            j=torch.arange(m,dtype=dt); w=torch.full((m,),2.0,dtype=dt); w[0]=1; w[-1]=1
            Cm=torch.cos(np.pi*j[:,None]*j[None,:]/(m-1))*w[None,:]     # [k][j]
            x=torch.movedim(torch.tensordot(Cm,torch.movedim(x,d,0),dims=([1],[0])),0,d)
        return x
    wgt=torch.ones(dims,dtype=dt)
    for d in range(Dn):
        w=torch.full((dims[d],),2.0,dtype=dt); w[0]=1; w[-1]=1
        shape=[1]*Dn; shape[d]=dims[d]; wgt=wgt*w.view(shape)
    A=dct1(qs)
    X=mask*A/(2*Ntot*s)
    H=dct1(X)
    g=(wgt*H).reshape(-1)
    print(dims,'clamped',nclamp,'rel err',float((g-gref).norm()/gref.norm()))
