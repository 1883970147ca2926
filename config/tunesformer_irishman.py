# TunesFormer-shaped model at full size on IrishMAN ABC tunes (the shape of the reference's tunesformer/config.py): patch level
# 9 layers, character level 3 layers, 768 wide, 12 heads, biases, HF's tanh GELU, 128 patches of 32 characters per tune
train_data = "data/irishman/train.json"
eval_data = "data/irishman/validation.json"
out_dir = "out-tunesformer-irishman"
patch_num_layers = 9
char_num_layers = 3
n_embd = 768
n_head = 12
bias = True
activation = "gelu_tanh"
patch_block_size = 128
learning_rate = 5e-5
