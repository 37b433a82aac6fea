"""Lane-utilisation diagnostics of the render kernel (COUNT_TRAVERSAL variant)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import shirley_raytracing_rs_b200 as rt
spp = int(sys.argv[1]) if len(sys.argv) > 1 else 100
scene = rt.Scene.named("random", seed=0xDEADBEEF)
cam = rt.default_camera(1200)
rt.render(scene, cam, samples=8, seed=1)
_, st0 = rt.render(scene, cam, samples=spp, seed=1)
acc, st = rt.render(scene, cam, samples=spp, seed=1, count_traversal=True)
d = list(st.diag)
envs = {k: v for k, v in os.environ.items() if k.startswith("B200RT_")}
print(f"{envs}  kernel {st0.kernel_ms:.1f} ms -> {st0.rays / st0.kernel_ms / 1e3:.0f} Mrays/s  rays {st.rays} paths {st.paths}")
print(f"   outer iterations {d[0]}  alive lanes/iter {d[1]/max(d[0],1):.2f}  out-of-work lanes/iter {d[2]/max(d[0],1):.2f}  regenerated/iter {d[6]/max(d[0],1):.2f}  shaded/iter {d[5]/max(d[0],1):.2f}")
print(f"   traversal rounds {d[3]}  traversing lanes/round {d[4]/max(d[3],1):.2f}  inner warp-steps {d[7]}  lanes per inner warp-step {st.node_visits/max(d[7],1):.2f}")
