import numpy as np, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ.setdefault("FL_PK_DEBUG", "0")
from fastllm_b200 import models, presets
cls, cf = presets.PRESETS["mistral7b"]
model,_ = cls.initialize_model(cf, None, "bf16", 0, random_seed=0)
cache = models.DeviceCache(model.dev, 1, 2200)
cache.fill_synthetic(1, 2048)
for i in range(3):
    cache.forward(np.array([[5]],dtype=np.uint32), 2048+i)
